"""Every instantiation of the tcgen05 GEMM, each row checked element by element against the fp64 oracle of the header
contract (tests/gemm_oracle.py), with the profiler confirming which instantiation the row actually ran.

The rows (tests/gemm_cases.py) cover ragged M and N around every tile width, K that is not a multiple of 64 or of 8,
both operand majors, bias present and absent, split-K of 1, 2, 7, more than the k blocks and the library's choice, and
taps 2-7 with a per-tap K that is not a multiple of 64.  Every output buffer carries sentinel rows and columns, and the
mask and colsum buffers sentinel bytes and entries, which the kernel must leave alone.  The process-wide switches run in
worker processes (tests/workers/gemm_env_worker.py).
"""
import dataclasses
import functools
import os
import subprocess
import sys
import tempfile

import pytest
import torch

import gemm_cases as gc
import gemm_oracle as go

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
WORKER = os.path.join(ROOT, "tests", "workers", "gemm_env_worker.py")


def check(c, inp, res):
    """The outputs of one launch of row c against the oracle, and the sentinels around them."""
    M, N = c.M, c.N
    out = res["out"]
    ref, bound = go.gemm_ref(inp["A"], inp["B"], M, N, c.K, a_mn=c.a_mn, b_mn=c.b_mn, bias=inp.get("bias"), act=c.act,
                             aux=inp.get("aux"), aux_mode=c.aux_mode, mask=inp.get("mask"), mask_mode=c.mask_mode,
                             taps=c.taps, accumulate=c.accumulate, d_init=inp.get("d_init"), out_f32=c.out_f32)
    msg = go.max_violation(out[:M, :N], ref, bound)
    assert not msg, f"{c.id}: {msg}"
    # TMA clips stores at row M and at column N rounded up to a 16-byte chunk
    n_touched = gc._ru(N, 4 if c.out_f32 else 8)
    assert bool((out[M:] == gc.SENTINEL).all()), f"{c.id}: rows >= M written"
    assert bool((out[:, n_touched:] == gc.SENTINEL).all()), f"{c.id}: columns beyond N written"
    if "mask" in res:
        m = res["mask"]
        assert torch.equal(m[:M, :N // 8], go.mask_bytes(out, M, N)), f"{c.id}: mask bits != sign of the stored output"
        assert bool((m[M:] == gc.MASK_FILL).all()) and bool((m[:, N // 8:] == gc.MASK_FILL).all()), f"{c.id}: mask bytes beyond M x N/8 written"
    if "colsum" in res:
        cs = res["colsum"]
        r, b = go.colsum_ref(out, M, N, torch.full((N,), gc.COLSUM_INIT, device=cs.device))
        msg = go.max_violation(cs[:N].view(1, N), r.view(1, N), b.view(1, N))
        assert not msg, f"{c.id} colsum: {msg}"
        assert bool((cs[N:] == gc.COLSUM_INIT).all()), f"{c.id}: colsum entries beyond N written"


def _walk_default():
    v = os.environ.get("IBM_WALK_ORDER", "0")[:1]
    return int(v) if v in ("1", "2") else 0


@pytest.mark.parametrize("c", gc.CASES, ids=lambda c: c.id)
def test_gemm_case(c):
    """One row against the oracle, then again with the work items taken in descending order: bit for bit the same output
    and mask (each element is computed by the same tile arithmetic), colsum and split-K sums within the oracle bound
    (fp32 atomics reorder them)."""
    from inferbiomechanics_b200 import ops
    inp = gc.make_inputs(c)
    res = gc.launch(c, inp)
    torch.cuda.synchronize()
    check(c, inp, res)
    ops.set_walk_order(2)            # every launch alternates, starting ascending
    try:
        gc.launch(c, inp)
        rev = gc.launch(c, inp)
        torch.cuda.synchronize()
    finally:
        ops.set_walk_order(_walk_default())
    check(c, inp, rev)
    if not c.atomic:
        assert torch.equal(rev["out"], res["out"]), f"{c.id}: descending walk changed the output"
        if "mask" in res:
            assert torch.equal(rev["mask"], res["mask"])


def test_dispatch_reaches_named_kernels():
    """Each row runs exactly the instantiation it names, and the rows (with the A-stationary ones of the IBM_GEMM_AS=1
    worker) run all 30 instantiations ibm_gemm_bf16 can launch.  A change of the dispatch rules fails here instead of
    silently moving what the table covers."""
    seen, wrong = set(), []
    for c in gc.CASES:
        kerns, _ = gc.profiled_launch(c, gc.make_inputs(c))
        if kerns != {c.kern}:
            wrong.append(f"{c.id}: ran {sorted(kerns)}")
        seen |= kerns
    for c in [c for c in gc.ENV_CASES if c.env == "IBM_GEMM_AS=1"]:
        seen |= set(_env_run(c.env)[c.id]["kerns"])
    assert not wrong, "rows that reached another instantiation:\n" + "\n".join(wrong)
    missing = set(gc.ALL_KERNELS) - seen
    assert not missing, f"instantiations no row reached: {sorted(missing)}"
    assert seen <= set(gc.ALL_KERNELS), f"unlisted instantiations: {sorted(seen - set(gc.ALL_KERNELS))}"


@functools.lru_cache(maxsize=None)
def _env_run(env):
    """Run the rows of one switch (ENV_CASES rows with that env, or its BITEXACT_ENVS rows) in a worker process."""
    name, value = env.split("=")
    cases = [c for c in gc.ENV_CASES if c.env == env] or gc.BITEXACT_ENVS[env]
    with tempfile.TemporaryDirectory() as d:
        out_file = os.path.join(d, "results.pt")
        r = subprocess.run([sys.executable, WORKER, out_file] + [c.id for c in cases], capture_output=True, text=True,
                           env=dict(os.environ, **{name: value}), cwd=ROOT, timeout=900)
        assert r.returncode == 0, f"{env} worker failed:\n{r.stderr[-3000:]}"
        return torch.load(out_file)


@pytest.mark.parametrize("env", sorted({c.env for c in gc.ENV_CASES}))
def test_env_switch_against_oracle(env):
    """IBM_GEMM_AS=1 (A-stationary), IBM_GEMM_NT_MINK=512 (two-tile work items at K = 512), IBM_GEMM_NT=1 (no two-tile
    work items), IBM_GEMM_CG=1 (single CTAs): each row reaches the instantiation it names and matches the oracle.  The
    non-atomic rows also come out bit-identical to the default schedule of the same inputs (every schedule sums an
    element's k blocks in the same order); the split-K rows do not, as the switch changes how the k range is split."""
    res = _env_run(env)
    for c in [c for c in gc.ENV_CASES if c.env == env]:
        r = res[c.id]
        assert set(r["kerns"]) == {c.kern}, f"{c.id}: ran {r['kerns']}"
        inp = gc.make_inputs(c)
        got = {k: r[k].cuda() for k in ("out", "mask", "colsum") if k in r}
        check(c, inp, got)
        if not c.atomic:
            default = gc.launch(dataclasses.replace(c, env=""), inp)
            assert torch.equal(default["out"], got["out"]), f"{c.id}: differs from the default schedule"


@pytest.mark.parametrize("env", list(gc.BITEXACT_ENVS))
def test_env_switch_bit_exact(env):
    """IBM_GEMM_FP2=0 (scalar bias adds), IBM_GEMM_STAGGER=0 (no staggered start of two-tile items), IBM_GEMM_PFAUX=1/2
    (aux tiles prefetched into L2) change no arithmetic: the outputs equal this process's bit for bit."""
    res = _env_run(env)
    for c in gc.BITEXACT_ENVS[env]:
        r = res[c.id]
        assert set(r["kerns"]) == {c.kern}, f"{c.id}: ran {r['kerns']}"
        inp = gc.make_inputs(c)
        got = {k: r[k].cuda() for k in ("out", "mask", "colsum") if k in r}
        check(c, inp, got)
        here = gc.launch(c, inp)
        assert torch.equal(here["out"], got["out"]), f"{c.id}: {env} changed the output"
        if "mask" in here:
            assert torch.equal(here["mask"], got["mask"])


# ---- epilogues the kernel does not compute are refused ---------------------------------------------------------------
REJECTED = [
    dict(act="sigmoid", aux_mode=1), dict(act="tanh", aux_mode=1), dict(act="silu", aux_mode=1),
    dict(act="sigmoid", aux_mode=1, out_f32=True), dict(act="silu", aux_mode=1, out_f32=True),
    dict(act="silu", aux_mode=2), dict(act="silu", aux_mode=2, out_f32=True),
    dict(act="relu", mask_mode=2), dict(act="sigmoid", mask_mode=2),
]


@pytest.mark.parametrize("kw", REJECTED, ids=lambda kw: "-".join(f"{k}={v}" for k, v in kw.items()))
def test_unsupported_epilogue_rejected(kw):
    """aux_mode 1 computes act(acc + bias) + aux for act none/relu/elu only; aux_mode 2 needs act' from the output, which
    SiLU does not have; mask_mode 2 gates acc + bias with no activation.  Anything else is a ValueError, not a result
    computed with another activation."""
    from inferbiomechanics_b200 import ops
    kw = dict(kw)
    out_f32 = kw.pop("out_f32", False)
    with pytest.raises(ValueError):
        go.check_epilogue(out_f32=out_f32, **kw)
    M, N, K = 256, 256, 64
    g = torch.Generator(device="cuda").manual_seed(5)
    A = torch.randn(M, K, generator=g, device="cuda").to(torch.bfloat16)
    B = torch.randn(N, K, generator=g, device="cuda").to(torch.bfloat16)
    out = torch.zeros(M, N, dtype=torch.float32 if out_f32 else torch.bfloat16, device="cuda")
    if kw.get("aux_mode"):
        kw["aux"] = torch.rand(M, N, generator=g, device="cuda").to(torch.bfloat16)
    if kw.get("mask_mode"):
        kw["mask"] = torch.full((M, N // 8), 0x55, dtype=torch.uint8, device="cuda")
    with pytest.raises(ValueError):
        ops.gemm(A, B, out, M, N, K, **kw)


def test_misaligned_bias_rejected():
    """The epilogue reads the bias as float4: a bias that is not 16-byte aligned is a ValueError; a 16-byte aligned view
    into the same buffer is fine."""
    from inferbiomechanics_b200 import ops
    c = gc.C(gc.HOT0, 515, 512, 256, "relu")
    inp = gc.make_inputs(c)
    buf = torch.zeros(c.N + 4, device="cuda")
    out = torch.empty(c.M, c.N, dtype=torch.bfloat16, device="cuda")
    buf[1:c.N + 1] = inp["bias"]
    with pytest.raises(ValueError):
        ops.gemm(inp["A"], inp["B"], out, c.M, c.N, c.K, bias=buf[1:c.N + 1], act="relu")
    buf[4:] = inp["bias"]
    res = gc.launch(c, dict(inp, bias=buf[4:]))
    check(c, inp, res)
