"""The attention oracle (tests/attention_oracle.py) on the CPU: its results against torch autograd in fp64 for every head
pair the kernels support, and its bounds against planted faults — each fault a kernel could make (a dropped key, a padded
key with weight, a row, head or window mixed up, a wrong scale, D of another row) must be flagged, while the exact result
rounded to bf16 passes.  This is what makes the element-wise bounds of tests/test_gpu_attention_matrix.py worth anything."""
import math

import pytest
import torch

import attention_oracle as ao

PAIRS = [(64, 64), (48, 48), (32, 32), (64, 8), (80, 8), (96, 8), (112, 8), (128, 8)]


def _inputs(hq, hv, n_win=3, T=7, H=2, seed=0, pad=8):
    """q, k, v, dO: bf16 2-D views with a leading dimension larger than H*hd (the padding is NaN)."""
    g = torch.Generator().manual_seed(seed * 131 + hq + hv)
    rows = n_win * T

    def mat(hd):
        buf = torch.full((rows + 2, H * hd + pad), float("nan"), dtype=torch.bfloat16)
        buf[:rows, :H * hd] = torch.randn(rows, H * hd, generator=g).to(torch.bfloat16)
        return buf
    return mat(hq), mat(hq), mat(hv), mat(hv)


def _torch_attention(q, k, v, n_win, T, H, hq, hv, scale):
    Q, K, V = (ao.heads(x, n_win, T, H, d).clone().requires_grad_(True) for x, d in ((q, hq), (k, hq), (v, hv)))
    o = torch.softmax((Q @ K.transpose(-1, -2)) * scale, dim=-1) @ V
    return Q, K, V, o


@pytest.mark.parametrize("hq,hv", PAIRS)
def test_forward_matches_autograd(hq, hv):
    n_win, T, H = 3, 7, 2
    q, k, v, _ = _inputs(hq, hv)
    scale = ao.f32(1 / math.sqrt(hq))
    o, bound, p = ao.attention_fwd_ref(q, k, v, n_win, T, H, hq, hv, scale)
    _, _, _, want = _torch_attention(q, k, v, n_win, T, H, hq, hv, scale)
    torch.testing.assert_close(o, ao.flat(want.detach()), rtol=1e-12, atol=1e-12)
    torch.testing.assert_close(p.sum(-1), torch.ones(n_win, H, T, dtype=torch.float64))
    assert bool((bound > 0).all()) and not ao.max_violation(o.to(torch.bfloat16), o, bound)


@pytest.mark.parametrize("hq,hv", PAIRS)
@pytest.mark.parametrize("d_from", ["exact", "stored_o"])
def test_backward_matches_autograd(hq, hv, d_from):
    """dq, dk (and dv for the pairs that produce it) against autograd.  D from the stored output: passing the exact
    output as that output must give the exact gradients."""
    n_win, T, H = 3, 7, 2
    q, k, v, d_o = _inputs(hq, hv, seed=1)
    scale = ao.f32(1 / math.sqrt(hq))
    Q, K, V, o = _torch_attention(q, k, v, n_win, T, H, hq, hv, scale)
    o.backward(ao.heads(d_o, n_win, T, H, hv))
    got = ao.attention_bwd_ref(q, k, v, d_o, n_win, T, H, hq, hv, scale,
                               o=None if d_from == "exact" else ao.flat(o.detach()))
    names = ("dq", "dk", "dv") if hv >= 16 else ("dq", "dk")
    for name, t in zip(names, (Q, K, V)):
        torch.testing.assert_close(got[name], ao.flat(t.grad), rtol=1e-10, atol=1e-12)
        assert not ao.max_violation(got[name].to(torch.bfloat16), got[name], got["b_" + name]), name


def test_bias_sums_and_zero_key_bias():
    """The fused bias sums: init + column sums; the key-bias gradient is zero in exact arithmetic and its bound covers
    the bf16-rounded summands."""
    n_win, T, H, hd = 4, 9, 3, 32
    q, k, v, d_o = _inputs(hd, hd, n_win, T, H, seed=2)
    r = ao.attention_bwd_ref(q, k, v, d_o, n_win, T, H, hd, hd, ao.f32(1 / math.sqrt(hd)))
    init = torch.full((H * hd,), 0.5)
    ref, bound = ao.bias_ref(r["dk"], r["b_dk"], init)
    assert float((ref - 0.5).abs().max()) < 1e-12
    got = init.double() + r["dk"].to(torch.bfloat16).double().sum(0)
    assert not ao.max_violation(got.view(1, -1), ref.view(1, -1), bound.view(1, -1))


# ---- planted faults ------------------------------------------------------------------------------------------------
def _attend(Q, K, V, scale, extra_zero_key=False, drop_last=False):
    s = (Q @ K.transpose(-1, -2)) * scale
    if drop_last:
        s[..., -1] = -math.inf
    if extra_zero_key:                  # one padded key (zero row) whose raw score 0 was not masked
        s = torch.cat([s, torch.zeros_like(s[..., :1])], -1)
        V = torch.cat([V, torch.zeros_like(V[..., :1, :])], -2)
    return torch.softmax(s, -1) @ V


FWD_FAULTS = ["drop_last_key", "padded_key_scored_0", "query_row_shift", "heads_swapped", "window_shift", "scale_1pct"]


@pytest.mark.parametrize("hq,hv", PAIRS)
@pytest.mark.parametrize("fault", FWD_FAULTS)
def test_forward_bound_flags_planted_fault(hq, hv, fault):
    n_win, T, H = 3, 7, 2
    q, k, v, _ = _inputs(hq, hv, seed=3)
    scale = ao.f32(1 / math.sqrt(hq))
    o, bound, _ = ao.attention_fwd_ref(q, k, v, n_win, T, H, hq, hv, scale)
    Q, K, V = ao.heads(q, n_win, T, H, hq), ao.heads(k, n_win, T, H, hq), ao.heads(v, n_win, T, H, hv)
    O = ao.heads(o, n_win, T, H, hv)
    if fault == "drop_last_key":
        bad = _attend(Q, K, V, scale, drop_last=True)
    elif fault == "padded_key_scored_0":
        bad = _attend(Q, K, V, scale, extra_zero_key=True)
    elif fault == "query_row_shift":
        bad = O.clone()
        bad[:, :, 3] = O[:, :, 4]
    elif fault == "heads_swapped":
        bad = O.flip(1)
    elif fault == "window_shift":
        bad = O.roll(1, 0)
    else:
        bad = _attend(Q, K, V, scale * 1.01)
    assert not ao.max_violation(o.to(torch.bfloat16), o, bound)
    assert ao.max_violation(ao.flat(bad).to(torch.bfloat16), o, bound), f"{fault} not flagged"


BWD_FAULTS = ["D_from_next_row", "drop_last_key", "scale_1pct", "dS_not_scaled"]


@pytest.mark.parametrize("hq,hv", PAIRS)
@pytest.mark.parametrize("fault", BWD_FAULTS)
def test_backward_bound_flags_planted_fault(hq, hv, fault):
    """dq and dk of a backward with a planted fault: at least one of them leaves its bound."""
    n_win, T, H = 3, 7, 2
    q, k, v, d_o = _inputs(hq, hv, seed=4)
    scale = ao.f32(1 / math.sqrt(hq))
    r = ao.attention_bwd_ref(q, k, v, d_o, n_win, T, H, hq, hv, scale)
    Q, K, V, G = (ao.heads(x, n_win, T, H, d) for x, d in ((q, hq), (k, hq), (v, hv), (d_o, hv)))
    sc = scale * (1.01 if fault == "scale_1pct" else 1.0)
    s = (Q @ K.transpose(-1, -2)) * sc
    if fault == "drop_last_key":
        s[..., -1] = -math.inf
    p = torch.softmax(s, -1)
    dP = G @ V.transpose(-1, -2)
    D = (p * dP).sum(-1, keepdim=True)
    if fault == "D_from_next_row":
        D = D.roll(-1, -2)
    dS = p * (dP - D) * (1.0 if fault == "dS_not_scaled" else sc)
    dq, dk = ao.flat(dS @ K), ao.flat(dS.transpose(-1, -2) @ Q)
    assert not ao.max_violation(r["dq"].to(torch.bfloat16), r["dq"], r["b_dq"])
    assert not ao.max_violation(r["dk"].to(torch.bfloat16), r["dk"], r["b_dk"])
    flagged = [n for n, x in (("dq", dq), ("dk", dk)) if ao.max_violation(x.to(torch.bfloat16), r[n], r["b_" + n])]
    assert flagged, f"{fault} not flagged"


def test_case_table_names_every_instantiation_twice():
    """The GPU matrix's rows (tests/attention_cases.py), with the worker rows, name each of the 64 instantiations at least
    twice, and their ids are unique."""
    import collections

    import attention_cases as ac
    rows = ac.CASES + ac.ENV_CASES
    assert len({c.id for c in rows}) == len(rows)
    named = collections.Counter(k for c in rows for k in c.kerns)
    assert len(ac.ALL_KERNELS) == 64 and set(named) == set(ac.ALL_KERNELS)
    assert min(named.values()) >= 2, [k for k, n in named.items() if n < 2]
    assert ac.parse_kernel_name("void ibm::attn::attn_bwd_long_kernel<(int)64, (int)8, (bool)0, true, 416>(const __nv_bfloat16 *)") \
        == "attn_bwd_long_kernel<64,8,0,1,416>"
    assert ac.parse_kernel_name("ibm::attn_tc::attn_bwd_tc_kernel(CUtensorMap_st, int)") == "attn_bwd_tc_kernel"
