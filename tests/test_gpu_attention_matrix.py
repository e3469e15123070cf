"""Every instantiation of the attention kernels, each row checked element by element against the fp64 oracle of the
header contract (tests/attention_oracle.py), with the profiler confirming which instantiations the row actually ran.

The rows (tests/attention_cases.py) cover ragged T around the 16-row and 64-key tiles, 1 to 8 heads, window counts that
do not divide the persistent grids (one window up to a few thousand), separate q / k / v with their own leading
dimensions, the fused qkv layout with kv_off > H * hd, outputs at a 4-byte but not 16-byte aligned column, scales 1,
1/sqrt(hd) and one that puts about 80 log2 units of spread into a row, and bias sums present and absent.  Input cells
outside the heads and rows past the last window are NaN, output cells outside the heads sentinels.  The needle and
uniform probes have closed-form answers; the process-wide switches run in worker processes
(tests/workers/attention_env_worker.py).
"""
import dataclasses
import functools
import os
import subprocess
import sys
import tempfile

import pytest
import torch

import attention_cases as ac
import attention_oracle as ao

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
WORKER = os.path.join(ROOT, "tests", "workers", "attention_env_worker.py")
BIAS_KEYS = ("dbias", "dbq", "dbk", "dbv")


def _bias_blocks(c, name):
    """[(output name, first entry)] of the bias vector `name`: which output's column sums land where."""
    if name == "dbias":
        kv = c.H * c.hq + 16
        return [("dq", 0), ("dk", kv), ("dv", 2 * kv)]
    return [(name[1:].replace("b", "d"), 0)]


def check(c, inp, res):
    """The outputs of one launch of row c against the oracle, and the cells around them.  Returns {output: max err/bound}."""
    H, rows = c.H, c.n_win * c.T
    views = ac.out_views(c, res)
    if c.kind == "fwd":
        o, b, _ = ao.attention_fwd_ref(inp["q"], inp["k"], inp["v"], c.n_win, c.T, H, c.hq, c.hv, c.scale_value)
        refs = {"o": (o, b)}
    else:
        r = ao.attention_bwd_ref(inp["q"], inp["k"], inp["v"], inp["do"], c.n_win, c.T, H, c.hq, c.hv, c.scale_value,
                                 o=inp["o"][:rows, :H * c.hv] if c.kind == "bwdl" else None)
        refs = {n: (r[n], r["b_" + n]) for n in views}
    ratios = {}
    for n, (ref, bound) in refs.items():
        msg = ao.max_violation(views[n], ref, bound)
        assert not msg, f"{c.id} {n}: {msg}"
        ratios[n] = ao.err_ratio(views[n], ref, bound)
    for name, m in ac.written_mask(c, res).items():
        assert bool((res[name][~m] == ac.SENTINEL).all()), f"{c.id}: {name} written outside the heads / past the last window"
    for key in BIAS_KEYS:
        if key not in res:
            continue
        bias = res[key]
        n = bias.numel() - 8
        assert bool((bias[n:] == ac.BIAS_SENTINEL).all()), f"{c.id}: {key} written past its end"
        touched = torch.zeros(n, dtype=torch.bool, device=bias.device)
        for out, c0 in _bias_blocks(c, key):
            ref, bound = refs[out]
            w = ref.shape[1]
            bref, bb = ao.bias_ref(ref, bound, torch.full((w,), ac.BIAS_INIT, device=bias.device))
            msg = ao.max_violation(bias[c0:c0 + w].view(1, w), bref.view(1, w), bb.view(1, w))
            assert not msg, f"{c.id} {key} ({out}): {msg}"
            ratios[key + "." + out] = ao.err_ratio(bias[c0:c0 + w].view(1, w), bref.view(1, w), bb.view(1, w))
            touched[c0:c0 + w] = True
        assert bool((bias[:n][~touched] == ac.BIAS_INIT).all()), f"{c.id}: {key} entries outside the heads changed"
    return ratios


def _outputs_equal(c, a, b):
    return all(torch.equal(a[name], b[name]) for name in ac.written_mask(c, a))


def _walk_default():
    v = os.environ.get("IBM_WALK_ORDER", "0")[:1]
    return int(v) if v in ("1", "2") else 0


@pytest.mark.parametrize("c", ac.CASES, ids=lambda c: c.id)
def test_attention_case(c):
    """One row against the oracle; without the bias accumulators bit for bit the same outputs; then again with the
    windows taken in descending order (attn_fwd_pipe_kernel and attn_bwd_tc_kernel reverse, nothing else may change):
    bit for bit the same outputs, bias sums within their bound (fp32 atomics reorder them)."""
    from inferbiomechanics_b200 import ops
    inp = ac.make_inputs(c)
    res = ac.launch_all(c, inp)
    torch.cuda.synchronize()
    ratios = check(c, inp, res)
    if "nobias" in res:
        assert _outputs_equal(c, res, res["nobias"]), f"{c.id}: the bias accumulators changed the outputs"
    ops.set_walk_order(2)            # every launch alternates, starting ascending
    try:
        ac.launch(c, inp)
        rev = ac.launch(c, inp)
        torch.cuda.synchronize()
    finally:
        ops.set_walk_order(_walk_default())
    check(c, inp, rev)
    assert _outputs_equal(c, res, rev), f"{c.id}: descending walk changed the outputs"
    print(f"\nratio {c.id} {' '.join(c.kerns)} " + " ".join(f"{k}={v:.3g}" for k, v in sorted(ratios.items())))


def _per_head(x, c, hd):
    return ao.heads(x, c.n_win, c.T, c.H, hd)


@pytest.mark.parametrize("c", [c for c in ac.CASES if c.kind == "fwd" or c.hv >= 16], ids=lambda c: c.id)
def test_needle_probe(c):
    """Query i of each (window, head) attends to key pi(i) alone: o_i = v_pi(i), and dv_j = dO_pi^-1(j), to within
    2^-20 relative.  Any row, key, head or window indexing error shows up at full size."""
    inp = ac.make_inputs(c, seed=1, needle=True)
    res = ac.launch(c, inp)
    views = ac.out_views(c, res)
    pi = inp["pi"]
    if c.kind == "fwd":
        V = _per_head(inp["v"], c, c.hv)
        want = torch.gather(V, 2, pi.unsqueeze(-1).expand(-1, -1, -1, c.hv))
        got = _per_head(views["o"], c, c.hv)
    else:
        G = _per_head(inp["do"], c, c.hv)
        inv = pi.argsort(-1)
        want = torch.gather(G, 2, inv.unsqueeze(-1).expand(-1, -1, -1, c.hv))
        got = _per_head(views["dv"], c, c.hv)
    err = (got - want).abs()
    assert bool((err <= 2.0 ** -20 * want.abs()).all()), f"{c.id}: {int((err > 2.0 ** -20 * want.abs()).sum())} elements off"


@pytest.mark.parametrize("c", [c for c in ac.CASES if c.kind == "fwd" or c.hv >= 16], ids=lambda c: c.id)
def test_uniform_probe(c):
    """q = 0: every probability is 1/T, so o_i is the mean of exactly the T values of its own window and head (and dv_j
    the mean of the T rows of dO).  The kernels round 1/T or the output once each and sum T terms in fp32:
    |err| <= (2 r + r^2) |mean| + (1 + r) (T + 3) u mean|x|.  A padded or foreign key, or a normaliser error, moves the mean."""
    inp = ac.make_inputs(c, seed=2, q_zero=True)
    res = ac.launch(c, inp)
    views = ac.out_views(c, res)
    src, got = (inp["v"], views["o"]) if c.kind == "fwd" else (inp["do"], views["dv"])
    X = _per_head(src, c, c.hv)
    mean, amean = X.mean(2, keepdim=True), X.abs().mean(2, keepdim=True)
    bound = (2 * ao.R + ao.R ** 2) * mean.abs() + (1 + ao.R) * (c.T + 3) * ao.U * amean
    err = (_per_head(got, c, c.hv) - mean).abs()
    assert bool((err <= bound).all()), f"{c.id}: worst {float((err - bound).max()):.3g} above the bound"


def test_dispatch_reaches_named_kernels():
    """Each row runs exactly the instantiations it names, and the rows (with those of the worker processes) run all 64
    instantiations.  A change of the dispatch rules fails here instead of silently moving what the table covers."""
    seen, wrong = set(), []
    default = _env_run("")
    for c in ac.CASES:
        kerns = set(default[c.id]["kerns"])
        if kerns != set(c.kerns):
            wrong.append(f"{c.id}: ran {sorted(kerns)}, named {sorted(c.kerns)}")
        seen |= kerns
    for env in sorted({c.env for c in ac.ENV_CASES}):
        for r in _env_run(env, kerns_only=True).values():
            seen |= set(r["kerns"])
    assert not wrong, "rows that reached other instantiations:\n" + "\n".join(wrong)
    missing = set(ac.ALL_KERNELS) - seen
    assert not missing, f"instantiations no row reached: {sorted(missing)}"
    assert seen <= set(ac.ALL_KERNELS), f"unlisted instantiations: {sorted(seen - set(ac.ALL_KERNELS))}"
    print(f"\n{len(seen)} attention instantiations reached")


@functools.lru_cache(maxsize=None)
def _env_run(env, kerns_only=False):
    """Run the ENV_CASES rows of one switch in a worker process ("": the CASES rows without a switch)."""
    cases = [c for c in ac.ENV_CASES if c.env == env] if env else ac.CASES
    kerns_only = kerns_only or not env
    extra = dict([env.split("=")]) if env else {}
    with tempfile.TemporaryDirectory() as d:
        out_file = os.path.join(d, "results.pt")
        r = subprocess.run([sys.executable, WORKER] + ["--kerns-only"] * kerns_only + [out_file] + [c.id for c in cases],
                           capture_output=True, text=True, env=dict(os.environ, **extra), cwd=ROOT, timeout=900)
        assert r.returncode == 0, f"{env} worker failed:\n{r.stderr[-3000:]}"
        return torch.load(out_file)


@pytest.mark.parametrize("env", sorted({c.env for c in ac.ENV_CASES}))
def test_env_switch_against_oracle(env):
    """IBM_ATTN_FWD=tc (tcgen05 forward), IBM_ATTN_BWD=mma (mma.sync backward for head_dim 64), IBM_ATTN_LONG=0 (one-shot
    kernel for long windows), IBM_ATTN_LONG_ONE=1 (one CTA per SM for long windows): each row reaches the instantiation
    it names and matches the oracle."""
    res = _env_run(env)
    for c in [c for c in ac.ENV_CASES if c.env == env]:
        r = res[c.id]
        assert set(r["kerns"]) == set(c.kerns), f"{c.id}: ran {r['kerns']}"
        got = {k: v.cuda() for k, v in r.items() if k != "kerns"}
        ratios = check(c, ac.make_inputs(c), got)
        print(f"\nratio {c.id} {' '.join(c.kerns)} " + " ".join(f"{k}={v:.3g}" for k, v in sorted(ratios.items())))


# ---- arguments the kernels do not handle are refused, before anything is launched -------------------------------------
BAD_SCALES = [float("nan"), float("inf"), float("-inf"), 0.0, -1.0]
REFUSAL_ROWS = {"fwd": ac._fwd(3, 50, 2, 64, 64), "bwd": ac._bwd(3, 50, 2, 64), "bwdl": ac._bwdl(3, 100, 2, 48, 48)}


@pytest.mark.parametrize("kind", list(REFUSAL_ROWS))
@pytest.mark.parametrize("scale", BAD_SCALES, ids=str)
def test_bad_scale_refused(kind, scale):
    """The kernels take the row maximum of the raw scores and scale afterwards, which is only right for a finite scale
    > 0 (a negative one overflows ex2 to inf and gives NaN).  Every entry point refuses any other scale with a
    ValueError, and its outputs stay untouched."""
    c = REFUSAL_ROWS[kind]
    inp = ac.make_inputs(c)
    out = ac._outputs(c, "cuda")
    with pytest.raises(ValueError):
        _launch_into(c, inp, out, scale)
    torch.cuda.synchronize()
    for name in out:
        assert bool((out[name] == ac.SENTINEL).all()), f"{name} written by a refused call"


def _launch_into(c, inp, out, scale=None):
    from inferbiomechanics_b200 import ops
    v = ac.out_views(c, out)
    s = c.scale_value if scale is None else scale
    if c.kind == "fwd":
        ops.attention_fwd(inp["q"], inp["k"], inp["v"], v["o"], c.n_win, c.T, c.H, c.hq, c.hv, s)
    elif c.kind == "bwd":
        ops.attention_bwd(inp["qkv"], inp["kv_off"], inp["do"], out["dqkv"], c.n_win, c.T, c.H, c.hq, s)
    else:
        ops.attention_bwd_long(inp["q"], inp["k"], inp["v"], inp["o"], inp["do"], v["dq"], v["dk"], v.get("dv"),
                               c.n_win, c.T, c.H, c.hq, c.hv, s)


@pytest.mark.parametrize("which", ["o", "dq", "dk", "dv"])
def test_odd_output_offset_refused(which):
    """The kernels store o, dq, dk, dv (and read o) as bf16 pairs: a view that starts at an odd bf16 column is a ValueError
    (nothing is launched, so this never makes a misaligned access); a 4-byte aligned view into the same buffer works and
    matches the oracle."""
    from inferbiomechanics_b200 import ops
    if which == "o":
        c = dataclasses.replace(REFUSAL_ROWS["fwd"], out_off=2)
        inp = ac.make_inputs(c)
        out = ac._outputs(c, "cuda")
        rows, cols = c.n_win * c.T, c.H * c.hv
        with pytest.raises(ValueError):
            ops.attention_fwd(inp["q"], inp["k"], inp["v"], out["o_buf"][:rows, 1:1 + cols], c.n_win, c.T, c.H, c.hq,
                              c.hv, c.scale_value)
    else:
        c = dataclasses.replace(REFUSAL_ROWS["bwdl"], out_off=2, dbias=False)
        inp = ac.make_inputs(c)
        out = ac._outputs(c, "cuda")
        rows = c.n_win * c.T
        v = ac.out_views(c, out)
        odd = dict(v)
        odd[which] = out[which + "_buf"][:rows, 1:1 + v[which].shape[1]]
        with pytest.raises(ValueError):
            ops.attention_bwd_long(inp["q"], inp["k"], inp["v"], inp["o"], inp["do"], odd["dq"], odd["dk"], odd["dv"],
                                   c.n_win, c.T, c.H, c.hq, c.hv, c.scale_value)
    torch.cuda.synchronize()
    for name in out:
        assert bool((out[name] == ac.SENTINEL).all()), f"{name} written by a refused call"
    _launch_into(c, inp, out)
    torch.cuda.synchronize()
    check(c, inp, out)


def test_odd_forward_output_offset_refused_for_bwd_long_input():
    """ibm_attention_bwd_long reads the forward output o as bf16 pairs too: an o at an odd column is refused."""
    from inferbiomechanics_b200 import ops
    c = dataclasses.replace(REFUSAL_ROWS["bwdl"], dbias=False)
    inp = ac.make_inputs(c)
    rows, cols = c.n_win * c.T, c.H * c.hv
    shifted = torch.zeros(rows, cols + 8, dtype=torch.bfloat16, device="cuda")
    shifted[:, 1:1 + cols] = inp["o"][:rows, :cols]
    out = ac._outputs(c, "cuda")
    v = ac.out_views(c, out)
    with pytest.raises(ValueError):
        ops.attention_bwd_long(inp["q"], inp["k"], inp["v"], shifted[:, 1:1 + cols], inp["do"], v["dq"], v["dk"], v["dv"],
                               c.n_win, c.T, c.H, c.hq, c.hv, c.scale_value)
    torch.cuda.synchronize()
    for name in out:
        assert bool((out[name] == ac.SENTINEL).all()), f"{name} written by a refused call"
