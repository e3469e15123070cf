"""Groundlink's own kernels one layer at a time, against references in fp64 and numpy indexing:

- the replicate-pad / fold kernels of the padded row layout (frame t of window b at row b*(T + 2 pad) + pad + t), bit for
  bit on small-integer values whose sums are exact;
- the three Conv1d weight re-layouts, bit for bit;
- every conv layer of the real engine on its own stored inputs: forward, weight / bias / input gradients;
- the whole model at the edges the golden tests do not reach (cnn_kernel = 1, one-frame windows, the graphed batch-of-one
  inference path).

Bars: one bf16 rounding of a GEMM output 1/128 * max|ref|, two (dgrad, then fold) 1/64 * max|ref|, fp32 GEMM outputs
2e-4 * max|ref|, as in test_gpu_gemm.py; whole-model cases at the bars of test_gpu_groundlink.py."""
import numpy as np
import pytest
import torch

from oracle import loss as ol
from oracle import models as om
from oracle.gen_golden import seeded_inputs, seeded_out_labels
from oracle.seeded import seeded_state_dict

pytestmark = pytest.mark.gpu
Q = (ol.COP, ol.FORCE, ol.TORQUE, ol.WRENCH)
SENTINEL = 0x7FA5                   # a bf16 NaN bit pattern: any read-modify-write of a pad column changes it
GUARD = 4                           # rows of sentinel before and after the windows


# ---------------------------------------------------------------------------------------------------------------------
# 1. replicate / fold of the pad rows
# ---------------------------------------------------------------------------------------------------------------------
def _padded(n_win, T, pad, cols, ld, seed, small_int=True):
    """bf16 [GUARD + n_win * Tp + GUARD, ld] on the host: window rows hold values in columns < cols; the columns >= cols
    and the guard rows hold SENTINEL."""
    Tp = T + 2 * pad
    g = torch.Generator().manual_seed(seed)
    full = torch.full((n_win * Tp + 2 * GUARD, ld), SENTINEL, dtype=torch.int16).view(torch.bfloat16)
    if small_int:
        vals = torch.randint(-8, 9, (n_win * Tp, cols), generator=g).to(torch.bfloat16)
    else:
        vals = torch.randn(n_win * Tp, cols, generator=g).to(torch.bfloat16)
    full[GUARD:GUARD + n_win * Tp, :cols] = vals
    return full


def _replicate_model(w, T, pad, cols):
    """w: (n_win, Tp, cols) values of the window rows, changed in place."""
    w[:, :pad] = w[:, pad:pad + 1]
    w[:, T + pad:] = w[:, T + pad - 1:T + pad]


def _fold_model(w, T, pad, cols):
    left = w[:, :pad].sum(axis=1)
    right = w[:, T + pad:].sum(axis=1)
    w[:, pad] += left                            # T == 1: the same row gains both sides
    w[:, T + pad - 1] += right
    w[:, :pad] = 0
    w[:, T + pad:] = 0


def _run_pad_op(op, full, n_win, T, pad, cols):
    from inferbiomechanics_b200 import ops
    d = full.cuda()
    view = d[GUARD:GUARD + n_win * (T + 2 * pad)]
    (ops.replicate_pad_rows if op == "replicate" else ops.fold_pad_rows)(view, n_win, T, pad, cols)
    return d.cpu()


def _check_pad_op(op, n_win, T, pad, cols, ld, seed):
    Tp = T + 2 * pad
    full = _padded(n_win, T, pad, cols, ld, seed)
    got = _run_pad_op(op, full, n_win, T, pad, cols)
    what = f"{op} n_win={n_win} T={T} pad={pad} cols={cols} ld={ld}"
    bits, got_bits = full.view(torch.int16), got.view(torch.int16)
    assert torch.equal(got_bits[:, cols:], bits[:, cols:]), f"{what}: columns >= cols changed"
    assert torch.equal(got_bits[:GUARD], bits[:GUARD]) and torch.equal(got_bits[-GUARD:], bits[-GUARD:]), \
        f"{what}: rows outside the windows changed"
    rows = slice(GUARD, GUARD + n_win * Tp)
    # small integers: every sum is exact in fp32 and in bf16, whatever the order
    want = full[rows, :cols].float().numpy().reshape(n_win, Tp, cols)
    (_replicate_model if op == "replicate" else _fold_model)(want, T, pad, cols)
    got_v = got[rows, :cols].float().numpy().reshape(n_win, Tp, cols)
    bad = np.argwhere(got_v != want)
    if bad.size:
        b, r, c = bad[0]
        raise AssertionError(f"{what}: {len(bad)} values differ; first at window {b}, padded row {r}, column {c}: "
                             f"got {got_v[b, r, c]}, want {want[b, r, c]}")


PAD_T = [1, 2, 3, 4, 7, 50]
PAD_PAD = [1, 2, 3, 4]
PAD_COLS = [8, 128, 184, 256]


@pytest.mark.parametrize("op", ["replicate", "fold"])
@pytest.mark.parametrize("n_win", [1, 3, 4096])
@pytest.mark.parametrize("T", PAD_T)
def test_pad_rows_match_numpy_model(op, n_win, T):
    """Frame rows unchanged, pad rows = edge frame (replicate); edge frames += their side's pad rows, both sides at T = 1,
    pad rows zero, interior unchanged (fold).  T <= pad included; ld > cols with a sentinel that must survive."""
    for pad in PAD_PAD:
        for cols in PAD_COLS:
            _check_pad_op(op, n_win, T, pad, cols, cols + 8 * (1 + pad % 2), seed=T * 1000 + pad * 10 + cols)


@pytest.mark.parametrize("op", ["replicate", "fold"])
def test_pad_rows_grid_stride_loop(op):
    """More (window, chunk[, pad row]) items than the launch has threads, so every thread loops."""
    threads = torch.cuda.get_device_properties(0).multi_processor_count * 16 * 256      # ew_grid's cap x 256 threads
    n_win, T, pad, cols = 12000, 2, 3, 256
    items = n_win * 2 * (cols // 8) * (pad if op == "replicate" else 1)
    assert items > threads
    _check_pad_op(op, n_win, T, pad, cols, cols + 8, seed=5)


@pytest.mark.parametrize("T", [1, 2, 7])
def test_pad_rows_adjoint_identity(T):
    """<replicate(X), G> = <X, fold(G)> in fp64 on random bf16 values.  fold stores its fp32 edge sums as bf16, so the two
    sides differ by at most one bf16 rounding (2^-9 relative) of each folded edge value times |X| there."""
    n_win, pad, cols, ld = 37, 3, 184, 192
    Tp = T + 2 * pad
    X = _padded(n_win, T, pad, cols, ld, seed=1, small_int=False)
    G = _padded(n_win, T, pad, cols, ld, seed=2, small_int=False)
    rows = slice(GUARD, GUARD + n_win * Tp)
    frames = torch.zeros(n_win, Tp, dtype=torch.bool)
    frames[:, pad:pad + T] = True
    frames = frames.reshape(-1)
    RX = _run_pad_op("replicate", X, n_win, T, pad, cols)[rows, :cols].double()
    FG = _run_pad_op("fold", G, n_win, T, pad, cols)[rows, :cols].double()
    Xv, Gv = X[rows, :cols].double(), G[rows, :cols].double()
    lhs = (RX * Gv).sum().item()
    rhs = (Xv[frames] * FG[frames]).sum().item()             # X's pad rows are outputs of replicate, not inputs
    edge = torch.zeros(n_win, Tp, dtype=torch.bool)
    edge[:, pad] = True
    edge[:, T + pad - 1] = True
    edge = edge.reshape(-1)
    tol = 2.0 ** -9 * (Xv[edge].abs() * FG[edge].abs()).sum().item() + 1e-9 * (RX.abs() * Gv.abs()).sum().item()
    assert abs(lhs - rhs) <= tol, f"T={T}: {lhs} vs {rhs} (tol {tol})"


def test_pad_rows_arguments():
    from inferbiomechanics_b200 import ops
    X = torch.zeros(2 * 8, 136, dtype=torch.bfloat16, device="cuda")
    Y = torch.zeros(2 * 8, 132, dtype=torch.bfloat16, device="cuda")
    for fn in (ops.replicate_pad_rows, ops.fold_pad_rows):
        with pytest.raises(ValueError):
            fn(X, 2, 2, 3, 12)                                  # cols % 8
        with pytest.raises(ValueError):
            fn(Y, 2, 2, 3, 128)                                 # ld % 8
        with pytest.raises(ValueError):
            fn(X, 2, 2, -1, 128)                                # negative pad
        with pytest.raises(ValueError):
            fn(X, 2, 0, 3, 128)                                 # no frames
    # pad == 0 (kernel size 1) is a no-op
    R = torch.randn(2 * 8, 136, device="cuda").to(torch.bfloat16)
    before = R.clone()
    ops.replicate_pad_rows(R, 2, 8, 0, 136)
    ops.fold_pad_rows(R, 2, 8, 0, 136)
    torch.cuda.synchronize()
    assert torch.equal(R.view(torch.int16), before.view(torch.int16))


# ---------------------------------------------------------------------------------------------------------------------
# 2. Conv1d weight re-layouts
# ---------------------------------------------------------------------------------------------------------------------
def _engine_pads(cout, cin):
    from inferbiomechanics_b200 import ops
    return ops.round_up(ops.round_up(cin, 8), 64), ops.round_up(cout, 64)        # GroundlinkEngine's cin_pad, cout_pad


CONV_SHAPES = [(128, 177), (128, 128), (256, 128), (256, 256)]


@pytest.mark.parametrize("k", [1, 3, 7, 9])
@pytest.mark.parametrize("cout,cin", CONV_SHAPES)
def test_conv_weight_relayouts_bit_for_bit(cout, cin, k):
    from inferbiomechanics_b200 import ops
    cin_pad, cout_pad = _engine_pads(cout, cin)
    g = torch.Generator().manual_seed(cout + cin + k)
    W = torch.randn(cout, cin, k, generator=g)
    Wd = W.cuda()
    Wb = W.to(torch.bfloat16)                                   # torch's fp32 -> bf16 is round-to-nearest-even too
    # forward GEMM layout [cout, k * cin_pad]: B[co, j * cin_pad + ci] = W[co, ci, j], zero for ci >= cin
    want = torch.zeros(cout, k, cin_pad, dtype=torch.bfloat16)
    want[:, :, :cin] = Wb.permute(0, 2, 1)
    got = torch.full((cout, k * cin_pad), 3.0, dtype=torch.bfloat16, device="cuda")
    ops.conv_weight_to_gemm(Wd, got, cin_pad)
    assert torch.equal(got.cpu().view(torch.int16), want.reshape(cout, -1).view(torch.int16)), "conv_weight_to_gemm"
    # dgrad layout [cin, k * cout_pad]: B[ci, j * cout_pad + co] = W[co, ci, k - 1 - j], zero for co >= cout
    want = torch.zeros(cin, k, cout_pad, dtype=torch.bfloat16)
    want[:, :, :cout] = Wb.flip(2).permute(1, 2, 0)
    got = torch.full((cin, k * cout_pad), 3.0, dtype=torch.bfloat16, device="cuda")
    ops.conv_weight_to_dgrad(Wd, got, cout_pad)
    assert torch.equal(got.cpu().view(torch.int16), want.reshape(cin, -1).view(torch.int16)), "conv_weight_to_dgrad"
    # wgrad: GEMM-layout fp32 [cout, k * cin_pad] -> (cout, cin, k); the pad columns ci >= cin must never be read
    gm = torch.full((cout, k, cin_pad), float("nan"))
    gm[:, :, :cin] = torch.randn(cout, k, cin, generator=g)
    init = torch.randn(cout, cin, k, generator=g)
    want = gm[:, :, :cin].permute(0, 2, 1).contiguous()
    for acc in (False, True):
        dw = init.cuda()
        ops.conv_wgrad_from_gemm(gm.reshape(cout, -1).cuda(), dw, cin_pad, accumulate=acc)
        ref = (init + want) if acc else want                    # the same single fp32 addition as the kernel
        assert torch.equal(dw.cpu(), ref), f"conv_wgrad_from_gemm accumulate={acc}"


# ---------------------------------------------------------------------------------------------------------------------
# 3. each conv layer of the engine on its own inputs
# ---------------------------------------------------------------------------------------------------------------------
def _elu(x):
    return torch.where(x > 0, x, torch.expm1(x))


def _conv_fwd(Xp, W, b, T):
    """Xp (B, Tp, cin) padded input, W (cout, cin, k) -> pre-activation frames (B, T, cout)."""
    out = b.view(1, 1, -1).expand(Xp.shape[0], T, -1).clone()
    for j in range(W.shape[2]):
        out += Xp[:, j:j + T] @ W[:, :, j].t()
    return out


def _conv_wgrad(G, Xp, k, T):
    return torch.stack([torch.einsum("bto,bti->oi", G, Xp[:, j:j + T]) for j in range(k)], dim=2)


def _conv_dgrad_padded(G, W, Tp):
    """Gradient w.r.t. the padded input: dXp[:, t + j] += G[:, t] @ W[:, :, j]."""
    B, T, _ = G.shape
    dX = torch.zeros(B, Tp, W.shape[1], dtype=G.dtype, device=G.device)
    for j in range(W.shape[2]):
        dX[:, j:j + T] += G @ W[:, :, j]
    return dX


def _fold_frames(dXp, T, pad):
    out = dXp[:, pad:pad + T].clone()
    out[:, 0] += dXp[:, :pad].sum(1)
    out[:, T - 1] += dXp[:, T + pad:].sum(1)
    return out


def _max_rel(got, ref):
    return ((got - ref).abs().max() / (ref.abs().max() + 1e-30)).item()


def _check_layers(m, B, T, dev):
    """Compares the engine's stored layer buffers with fp64 references computed on ``dev``; returns the worst error of each
    family relative to its bar's scale."""
    eng = m.engine()
    st, Tp, Mp = eng._state(B, T)
    pad = eng.pad
    worst = {}

    def note(k, v):
        worst[k] = max(worst.get(k, 0.0), v)

    def buf(name, i, C):
        return st[f"{name}{i}"].view(B, Tp, eng.ld[i])[:, :, :C]

    for i, pos in enumerate(eng.conv_pos):
        cin, cout = eng.ch[i], eng.ch[i + 1]
        conv = m.cnn[pos]
        W = conv.weight.detach().to(torch.bfloat16).to(dev).double()
        bias = conv.bias.detach().to(dev).double()
        Xp = buf("x", i, cin).to(dev).double()
        Y = buf("x", i + 1, cout)
        G = buf("g", i + 1, cout)[:, pad:pad + T].to(dev).double()
        what = f"k={eng.kt} B={B} T={T} layer {i}"
        # forward: frame rows of x{i+1} = ELU(conv(Xp) + b), pad rows = the edge frames bit for bit
        ref = _elu(_conv_fwd(Xp, W, bias, T))
        e = _max_rel(Y[:, pad:pad + T].to(dev).double(), ref)
        note("forward", e * 128)
        assert e <= 1.0 / 128, f"{what} forward: {e:.3g} x max|ref|"
        Yi = Y.view(torch.int16)
        assert torch.equal(Yi[:, :pad], Yi[:, pad:pad + 1].expand(-1, pad, -1)), f"{what}: left pad rows"
        assert torch.equal(Yi[:, T + pad:], Yi[:, T + pad - 1:T + pad].expand(-1, pad, -1)), f"{what}: right pad rows"
        # weight gradient (fp32 GEMM output)
        ref = _conv_wgrad(G, Xp, eng.kt, T)
        e = _max_rel(conv.weight.grad.to(dev).double(), ref)
        note("wgrad", e / 2e-4)
        assert e <= 2e-4, f"{what} weight gradient: {e:.3g} x max|ref|"
        # bias gradient: the frame-row sum of G
        ref = G.sum((0, 1))
        got = conv.bias.grad.to(dev).double()
        e = ((got - ref).abs() / (1e-4 * ref.abs() + 1e-4 * ref.abs().max())).max().item()
        note("bias grad", e)
        assert e <= 1.0, f"{what} bias gradient: {(got - ref).abs().max().item():.3g}"
        if i == 0:
            continue
        # input gradient: fold(ELU'(x_i) * d conv / d Xp), ELU' from the stored output (pad rows included)
        Xs = buf("x", i, cin).to(dev).double()
        dXp = _conv_dgrad_padded(G, W, Tp) * torch.where(Xs > 0, torch.ones_like(Xs), Xs + 1)
        ref = _fold_frames(dXp, T, pad)
        e = _max_rel(buf("g", i, cin)[:, pad:pad + T].to(dev).double(), ref)
        note("dgrad", e * 64)
        assert e <= 1.0 / 64, f"{what} input gradient: {e:.3g} x max|ref|"
    return worst


def _seeded_groundlink(fmt, k, seed):
    from inferbiomechanics_b200.models.Groundlink import Groundlink
    m = Groundlink(23, 12, 10, fmt, cnn_kernel=k, fc_dropout=0.0)
    m.load_state_dict(seeded_state_dict({n: tuple(v.shape) for n, v in m.state_dict().items()}, seed))
    return m


def _train_step(m, B, T, fmt, seed):
    inputs = seeded_inputs(B, T, 23, 30, seed)
    out = m(inputs)
    y = torch.cat([out[q] for q in Q], dim=-1)
    gy = seeded_out_labels(B, T if fmt == "all_frames" else 1, seed + 50)[0]
    gy = torch.cat([gy[q] for q in Q], dim=-1).to(y.device)
    for p in m.parameters():
        p.grad = None
    (y * gy).sum().backward()
    return inputs, out, gy


@pytest.mark.parametrize("fmt", ["all_frames", "last_frame"])
@pytest.mark.parametrize("T", [1, 2, 3, 20, 50])
@pytest.mark.parametrize("k", [1, 3, 7, 9])
def test_conv_layers_match_fp64(k, T, fmt):
    for B in (1, 5):
        m = _seeded_groundlink(fmt, k, seed=k * 100 + T).cuda().train()
        _train_step(m, B, T, fmt, seed=B + T)
        worst = _check_layers(m, B, T, "cpu")
        print(f"k={k} T={T} {fmt} B={B}: worst error / bar " + ", ".join(f"{n} {v:.3f}" for n, v in worst.items()))


def test_conv_layers_match_fp64_at_bench_shape():
    """B = 4096 windows of 50 frames, k = 7 (the benchmarked Groundlink step); the fp64 reference runs on the device."""
    m = _seeded_groundlink("all_frames", 7, seed=77).cuda().train()
    _train_step(m, 4096, 50, "all_frames", seed=78)
    worst = _check_layers(m, 4096, 50, "cuda")
    print("bench shape: worst error / bar " + ", ".join(f"{n} {v:.3f}" for n, v in worst.items()))


# ---------------------------------------------------------------------------------------------------------------------
# 4. the whole model at the new edges
# ---------------------------------------------------------------------------------------------------------------------
def _oracle_grads(m, inputs, gy, fmt):
    sd = {n: v.detach().double().cpu().requires_grad_(True) for n, v in m.state_dict().items()}
    ref = om.groundlink_forward(sd, {k: v.double() for k, v in inputs.items()}, fmt)
    y = torch.cat([ref[q] for q in Q], dim=-1)
    (y * gy.double().cpu()).sum().backward()
    return ref, {n: v.grad for n, v in sd.items()}


@pytest.mark.parametrize("fmt", ["all_frames", "last_frame"])
@pytest.mark.parametrize("k,T", [(1, 20), (1, 1), (7, 1), (3, 1)])
def test_whole_model_at_new_edges_matches_oracle(k, T, fmt):
    B = 6
    m = _seeded_groundlink(fmt, k, seed=900 + k + T).cuda().train()
    inputs, out, gy = _train_step(m, B, T, fmt, seed=31)
    ref, grads = _oracle_grads(m, inputs, gy, fmt)
    for q in Q:
        assert tuple(out[q].shape) == tuple(ref[q].shape)
        err = (out[q].detach().double().cpu() - ref[q].detach()).abs().max().item()
        assert err <= 3e-2 * ref[q].abs().max().item(), f"{q}: {err}"
    for n, p in m.named_parameters():
        got, want = p.grad.double().reshape(-1).cpu(), grads[n].reshape(-1)
        rel = (got - want).norm().item() / (want.norm().item() + 1e-12)
        cos = torch.dot(got, want).item() / (got.norm().item() * want.norm().item() + 1e-30)
        assert rel <= 0.12 and cos >= 0.985, f"{n}: rel L2 {rel:.4f}, cosine {cos:.4f}"


@pytest.mark.parametrize("k,T", [(1, 20), (7, 1), (1, 1)])
def test_batch_of_one_graphed_inference_at_new_edges(monkeypatch, k, T):
    """B = 1 under no_grad in eval mode replays a captured CUDA graph (which contains the pad refreshes): the same bits as
    the eager launches, and the oracle's outputs at the golden bar."""
    m = _seeded_groundlink("last_frame", k, seed=40 + k + T).cuda().eval()
    xs = [seeded_inputs(1, T, 23, 30, 60 + i) for i in range(5)]
    with torch.no_grad():
        monkeypatch.setenv("IBM_INFER_GRAPHS", "0")
        eager = [{q: v.clone() for q, v in m(x).items()} for x in xs]
        monkeypatch.setenv("IBM_INFER_GRAPHS", "1")
        graphed = [{q: v.clone() for q, v in m(x).items()} for x in xs]       # calls 1-2 eager, 3 captures, 4-5 replay
    assert any(st["graph"] is not None for st in m._lat.values())
    for a, b in zip(eager, graphed):
        for q in Q:
            assert torch.equal(a[q], b[q]), q
    # the golden bar is relative to the largest output of a batch: here the batch is the five one-window calls
    sd = {n: v.detach().double().cpu() for n, v in m.state_dict().items()}
    refs = [om.groundlink_forward(sd, {q: v.double() for q, v in x.items()}, "last_frame") for x in xs]
    for q in Q:
        got = torch.cat([b[q].double().cpu() for b in graphed])
        ref = torch.cat([r[q] for r in refs])
        err = (got - ref).abs().max().item()
        assert err <= 3e-2 * ref.abs().max().item(), f"{q}: {err} vs max|ref| {ref.abs().max().item()}"
