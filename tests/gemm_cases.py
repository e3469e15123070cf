"""The GEMM case table: one or more rows per template instantiation of gemm_kernel (csrc/gemm_sm100.cu), each naming the
instantiation the dispatch in ibm_gemm_bf16 must pick for it on a 148-SM B200.  TEST INFRASTRUCTURE ONLY; used by
tests/test_gpu_gemm_matrix.py and its environment-switch worker (tests/workers/gemm_env_worker.py).

An instantiation is the tuple (BN, kOutF32, kAccum, kAux, CG, NT, kAS, MM) of gemm_kernel's template arguments.  The
dispatch rules the shapes below are chosen from:
  - pick_bn: the widest of 256/128/64/32 whose last column tile is at least 75 % full; MN-major B and bf16 outputs
    force BN >= 64
  - CG = 2 (CTA pair) iff M spans at least two 128-row blocks and BN >= 128
  - NT = 2 (two column tiles per work item) iff CG = 2, BN = 256, K >= 1024, an even number of 256-wide column tiles and
    either accumulate or (row blocks x column-tile pairs) >= 148; never for fp32 outputs with aux
  - A-stationary only under IBM_GEMM_AS=1: CG = 2, BN = 256, NT = 1, plain epilogue, K <= 512, >= 2 column tiles and
    >= 148 row blocks
  - MM (mask mode compiled in) only for the 256-wide CTA-pair plain bf16 kernel
"""
from __future__ import annotations

import dataclasses
import re
import zlib

import torch


def kern(bn, f32=0, acc=0, aux=0, cg=1, nt=1, a_st=0, mm=-1):
    return (bn, int(f32), int(acc), int(aux), cg, nt, int(a_st), mm)


AS_BF16, AS_F32 = kern(256, cg=2, a_st=1), kern(256, f32=1, cg=2, a_st=1)
NT_ACC, NT_F32 = kern(256, 1, 1, cg=2, nt=2), kern(256, 1, cg=2, nt=2)
NT_AUX, NT_BF16 = kern(256, aux=1, cg=2, nt=2), kern(256, cg=2, nt=2)
HOT0, HOT1, HOT2 = kern(256, cg=2, mm=0), kern(256, cg=2, mm=1), kern(256, cg=2, mm=2)
P256_ACC, P256_F32, P256_AUX = kern(256, 1, 1, cg=2), kern(256, 1, cg=2), kern(256, aux=1, cg=2)
P128_ACC, P128_F32, P128_AUX, P128_BF16 = kern(128, 1, 1, cg=2), kern(128, 1, cg=2), kern(128, aux=1, cg=2), kern(128, cg=2)


def _single(bn):
    return kern(bn, 1, 1), kern(bn, 1), kern(bn, aux=1), kern(bn)


S256_ACC, S256_F32, S256_AUX, S256_BF16 = _single(256)
S128_ACC, S128_F32, S128_AUX, S128_BF16 = _single(128)
S64_ACC, S64_F32, S64_AUX, S64_BF16 = _single(64)
S32_ACC, S32_F32 = kern(32, 1, 1), kern(32, 1)

# every instantiation ibm_gemm_bf16 can launch (the 31st, <256,bf16,plain,CG 2,MM -1>, serves ibm_debug_gemm_max_clusters)
ALL_KERNELS = [AS_BF16, AS_F32, NT_ACC, NT_F32, NT_AUX, NT_BF16, HOT0, HOT1, HOT2, P256_ACC, P256_F32, P256_AUX,
               P128_ACC, P128_F32, P128_AUX, P128_BF16, S256_ACC, S256_F32, S256_AUX, S256_BF16, S128_ACC, S128_F32,
               S128_AUX, S128_BF16, S64_ACC, S64_F32, S64_AUX, S64_BF16, S32_ACC, S32_F32]

_KNAME = re.compile(r"gemm_kernel<([^>]*)>")


def parse_kernel_name(name: str):
    """The template arguments of a profiler kernel name such as
    'void ibm::gemm::gemm_kernel<(int)256, (bool)0, ..., (int)-1>(CUtensorMap_st, ...)' (or '<256, false, ...>'), or None."""
    m = _KNAME.search(name)
    if m is None:
        return None
    vals = []
    for a in m.group(1).split(","):
        a = re.sub(r"\((?:int|bool)\)", "", a).strip()
        vals.append(1 if a == "true" else 0 if a == "false" else int(a))
    return tuple(vals)


@dataclasses.dataclass(frozen=True)
class Case:
    kern: tuple          # the instantiation this row must reach
    M: int
    N: int
    K: int
    act: str = "none"
    out_f32: bool = False
    accumulate: bool = False
    split_k: int = 0
    aux_mode: int = 0
    mask_mode: int = 0
    colsum: bool = False
    bias: bool = True
    a_mn: bool = False
    b_mn: bool = False
    taps: int = 1
    env: str = ""        # "NAME=value": the process-wide switch this row runs under (in a worker process)

    @property
    def id(self):
        s = f"{'-'.join(map(str, self.kern))}:{self.M}x{self.N}x{self.K}:{self.act}"
        for f, tag in (("out_f32", "f32"), ("accumulate", "acc"), ("colsum", "colsum"), ("a_mn", "amn"), ("b_mn", "bmn")):
            if getattr(self, f):
                s += ":" + tag
        if self.accumulate:
            s += f":split{self.split_k}"
        if self.aux_mode:
            s += f":aux{self.aux_mode}"
        if self.mask_mode:
            s += f":mask{self.mask_mode}"
        if not self.bias:
            s += ":nobias"
        if self.taps > 1:
            s += f":taps{self.taps}"
        if self.env:
            s += ":" + self.env
        return s

    @property
    def atomic(self):
        """Results summed with fp32 atomics in an order that depends on the schedule."""
        return self.accumulate


def C(k, M, N, K, act="none", **kw):
    if k[2]:                      # accumulate: fp32 output, plain epilogue, no bias
        kw.setdefault("bias", False)
        kw["accumulate"], kw["out_f32"] = True, True
    elif k[1]:
        kw["out_f32"] = True
    return Case(k, M, N, K, act, **kw)


CASES = [
    # ---- CTA pair, 256-wide, bf16, mask mode compiled in (the hot shapes) ----
    C(HOT0, 515, 512, 256, "relu"),
    C(HOT0, 129, 200, 64, bias=False),
    C(HOT0, 255, 1000, 68, "sigmoid"),
    C(HOT0, 257, 1000, 200, "tanh", a_mn=True),
    C(HOT0, 1025, 512, 1000, "silu", b_mn=True),
    C(HOT0, 300, 256, 136, "elu", a_mn=True, b_mn=True),
    C(HOT0, 515, 512, 256, "relu", colsum=True),
    C(HOT0, 129, 200, 144, "elu", taps=2),
    C(HOT0, 300, 256, 216, taps=3),
    C(HOT0, 300, 256, 216, taps=3, b_mn=True),
    C(HOT0, 257, 512, 952, "relu", taps=7),
    C(HOT1, 515, 512, 256, "relu", mask_mode=1),
    C(HOT1, 129, 192, 68, "relu", mask_mode=1),
    C(HOT1, 257, 1024, 300, mask_mode=1, b_mn=True, colsum=True),
    C(HOT1, 300, 256, 216, "relu", mask_mode=1, taps=3),
    C(HOT2, 515, 512, 256, mask_mode=2, b_mn=True),
    C(HOT2, 255, 192, 100, mask_mode=2, colsum=True),
    C(HOT2, 1025, 768, 520, mask_mode=2, a_mn=True),
    # ---- CTA pair, 256-wide, generic epilogues ----
    C(P256_ACC, 515, 200, 700, a_mn=True, b_mn=True),
    C(P256_ACC, 300, 256, 4000, a_mn=True, b_mn=True, split_k=1),
    C(P256_ACC, 300, 256, 4000, a_mn=True, b_mn=True, split_k=2),
    C(P256_ACC, 300, 256, 4000, a_mn=True, b_mn=True, split_k=7),
    C(P256_ACC, 300, 256, 4000, a_mn=True, b_mn=True, split_k=100),
    C(P256_ACC, 129, 768, 1111),
    C(P256_F32, 300, 256, 300, "tanh"),
    C(P256_F32, 515, 1000, 68, bias=False),
    C(P256_F32, 257, 200, 1100, b_mn=True),
    C(P256_F32, 300, 512, 216, taps=3),
    C(P256_F32, 515, 512, 256, "elu", aux_mode=1),
    C(P256_F32, 257, 256, 136, aux_mode=1),
    C(P256_F32, 300, 256, 300, "relu", aux_mode=2),
    C(P256_F32, 300, 256, 300, "sigmoid", aux_mode=2),
    C(P256_F32, 300, 256, 300, "elu", aux_mode=2, a_mn=True),
    C(P256_AUX, 515, 512, 256, aux_mode=1),
    C(P256_AUX, 515, 512, 256, "relu", aux_mode=1),
    C(P256_AUX, 257, 1000, 68, "elu", aux_mode=1, b_mn=True),
    C(P256_AUX, 129, 200, 300, "relu", aux_mode=2),
    C(P256_AUX, 300, 256, 300, "sigmoid", aux_mode=2, a_mn=True),
    C(P256_AUX, 300, 256, 300, "tanh", aux_mode=2),
    C(P256_AUX, 300, 512, 256, aux_mode=2),
    C(P256_AUX, 1025, 512, 408, "elu", aux_mode=2, taps=3, bias=False),
    C(P256_AUX, 515, 512, 256, "relu", aux_mode=2, b_mn=True, colsum=True),
    # ---- CTA pair, 128-wide ----
    C(P128_BF16, 129, 128, 64, "relu"),
    C(P128_BF16, 1025, 330, 68, "tanh", a_mn=True),
    C(P128_BF16, 300, 100, 200, b_mn=True, bias=False),
    C(P128_BF16, 257, 128, 256, "relu", mask_mode=1),
    C(P128_BF16, 257, 128, 256, mask_mode=2, colsum=True),
    C(P128_BF16, 300, 128, 144, taps=2),
    C(P128_F32, 257, 100, 300, "sigmoid"),
    C(P128_F32, 300, 330, 1100),
    C(P128_F32, 300, 128, 200, "relu", aux_mode=2),
    C(P128_AUX, 1000, 128, 256, "relu", aux_mode=1),
    C(P128_AUX, 300, 330, 500, "elu", aux_mode=2, b_mn=True),
    C(P128_AUX, 300, 128, 504, "elu", aux_mode=2, taps=7),
    C(P128_ACC, 300, 330, 500, a_mn=True, b_mn=True),
    C(P128_ACC, 129, 128, 1111, split_k=7),
    C(P128_ACC, 300, 100, 3000, a_mn=True, split_k=2),
    # ---- single CTA, 256-wide (M <= 128) ----
    C(S256_BF16, 1, 256, 64),
    C(S256_BF16, 127, 200, 68, "sigmoid", bias=False),
    C(S256_BF16, 128, 1000, 300, "relu", b_mn=True),
    C(S256_BF16, 127, 512, 100, a_mn=True),
    C(S256_BF16, 100, 256, 256, "relu", mask_mode=1),
    C(S256_BF16, 127, 512, 200, mask_mode=2, colsum=True),
    C(S256_BF16, 64, 256, 408, taps=3),
    C(S256_F32, 1, 256, 64),
    C(S256_F32, 127, 1000, 1100, "tanh"),
    C(S256_F32, 64, 200, 200, "relu", aux_mode=2),
    C(S256_F32, 100, 256, 136, "relu", aux_mode=1),
    C(S256_AUX, 127, 256, 300, aux_mode=1),
    C(S256_AUX, 1, 1000, 200, "tanh", aux_mode=2, b_mn=True),
    C(S256_AUX, 100, 512, 144, "elu", aux_mode=2, taps=2),
    C(S256_ACC, 127, 512, 2048, a_mn=True, b_mn=True),
    C(S256_ACC, 100, 200, 5000, split_k=7),
    C(S256_ACC, 1, 1000, 3000, a_mn=True, split_k=100),
    # ---- single CTA, 128-wide ----
    C(S128_BF16, 1, 128, 64),
    C(S128_BF16, 127, 330, 68, "relu", a_mn=True),
    C(S128_BF16, 100, 128, 256, "relu", mask_mode=1, colsum=True),
    C(S128_BF16, 128, 128, 200, mask_mode=2),
    C(S128_BF16, 64, 100, 216, taps=3),
    C(S128_BF16, 64, 100, 144, taps=2, b_mn=True),
    C(S128_F32, 127, 100, 300, "silu"),
    C(S128_F32, 1, 330, 200, "elu", aux_mode=1),
    C(S128_AUX, 127, 128, 300, "relu", aux_mode=1),
    C(S128_AUX, 64, 330, 136, "sigmoid", aux_mode=2, b_mn=True),
    C(S128_ACC, 100, 330, 700),
    C(S128_ACC, 128, 128, 2000, a_mn=True, b_mn=True, split_k=2),
    # ---- single CTA, 64-wide ----
    C(S64_BF16, 1000, 264, 200, "relu"),
    C(S64_BF16, 257, 8, 64),
    C(S64_BF16, 129, 30, 68, "sigmoid", bias=False),
    C(S64_BF16, 1, 72, 300, "tanh", b_mn=True),
    C(S64_BF16, 300, 72, 136, a_mn=True, b_mn=True),
    C(S64_BF16, 300, 64, 256, "relu", mask_mode=1),
    C(S64_BF16, 255, 64, 100, mask_mode=2, colsum=True),
    C(S64_BF16, 1025, 264, 216, taps=3),
    C(S64_F32, 300, 264, 300),
    C(S64_F32, 257, 30, 200, b_mn=True),
    C(S64_F32, 129, 64, 300, "relu", aux_mode=2),
    C(S64_AUX, 1000, 264, 256, "relu", aux_mode=1),
    C(S64_AUX, 129, 72, 200, "tanh", aux_mode=2),
    C(S64_AUX, 255, 30, 64, aux_mode=1, b_mn=True),
    C(S64_ACC, 264, 72, 2000, a_mn=True, b_mn=True),
    C(S64_ACC, 30, 64, 700, a_mn=True, b_mn=True, split_k=7),
    C(S64_ACC, 8, 264, 4000, split_k=7),
    # ---- single CTA, 32-wide (fp32 outputs only) ----
    C(S32_F32, 300, 30, 512),
    C(S32_F32, 1, 8, 68, a_mn=True),
    C(S32_F32, 257, 72, 200, "elu", aux_mode=2),
    C(S32_F32, 129, 30, 216, taps=3),
    C(S32_ACC, 30, 30, 4000, a_mn=True, split_k=7),
    C(S32_ACC, 8, 72, 700),
    C(S32_ACC, 72, 8, 300, a_mn=True, split_k=2),
    # ---- two column tiles per work item (NT = 2): >= 148 (row block, tile pair) items, or accumulate ----
    C(NT_BF16, 19000, 1024, 1024, "relu"),
    C(NT_BF16, 19000, 1000, 1064, "sigmoid", bias=False),
    C(NT_BF16, 38011, 512, 1100, "tanh", a_mn=True),
    C(NT_BF16, 19000, 1024, 1088, "relu", mask_mode=1, colsum=True),
    C(NT_BF16, 19000, 1024, 1024, mask_mode=2, b_mn=True),
    C(NT_BF16, 19000, 1024, 1120, taps=7),
    C(NT_F32, 19000, 1024, 1024),
    C(NT_F32, 19000, 1000, 1100, "elu", b_mn=True),
    C(NT_AUX, 19000, 1024, 1024, "relu", aux_mode=1),
    C(NT_AUX, 19000, 1000, 1064, "relu", aux_mode=2, b_mn=True, colsum=True),
    C(NT_AUX, 19000, 1024, 1024, "sigmoid", aux_mode=2),
    C(NT_ACC, 512, 512, 2048, a_mn=True, b_mn=True),
    C(NT_ACC, 300, 1000, 1111, a_mn=True, b_mn=True, split_k=1),
    C(NT_ACC, 257, 512, 4096, split_k=2),
    C(NT_ACC, 300, 1024, 8000, a_mn=True, b_mn=True, split_k=100),
    C(NT_ACC, 512, 1000, 1111, split_k=7),
]

# rows that run in a worker process under one switch, with the instantiation they must reach there
ENV_CASES = [
    C(AS_BF16, 40000, 512, 512, "relu", env="IBM_GEMM_AS=1"),
    C(AS_BF16, 38011, 1000, 328, "silu", bias=False, env="IBM_GEMM_AS=1"),
    C(AS_BF16, 40000, 512, 200, b_mn=True, env="IBM_GEMM_AS=1"),
    C(AS_BF16, 37900, 600, 68, a_mn=True, env="IBM_GEMM_AS=1"),
    C(AS_F32, 40000, 512, 512, "tanh", env="IBM_GEMM_AS=1"),
    C(AS_F32, 38011, 1000, 136, b_mn=True, env="IBM_GEMM_AS=1"),
    C(NT_BF16, 19000, 1024, 512, "relu", env="IBM_GEMM_NT_MINK=512"),
    C(NT_AUX, 19000, 1024, 512, aux_mode=1, env="IBM_GEMM_NT_MINK=512"),
    C(NT_F32, 19000, 1024, 576, env="IBM_GEMM_NT_MINK=512"),
    C(HOT0, 19000, 1024, 1024, "relu", env="IBM_GEMM_NT=1"),
    C(P256_AUX, 19000, 1024, 1024, "relu", aux_mode=1, env="IBM_GEMM_NT=1"),
    C(P256_F32, 19000, 1024, 1024, env="IBM_GEMM_NT=1"),
    C(P256_ACC, 512, 512, 2048, a_mn=True, b_mn=True, env="IBM_GEMM_NT=1"),
    C(S256_BF16, 515, 512, 256, "relu", env="IBM_GEMM_CG=1"),
    C(S256_BF16, 515, 512, 256, "relu", mask_mode=1, env="IBM_GEMM_CG=1"),
    C(S256_BF16, 19000, 1024, 1024, env="IBM_GEMM_CG=1"),
    C(S128_AUX, 300, 128, 504, "elu", aux_mode=2, taps=7, env="IBM_GEMM_CG=1"),
    C(S128_F32, 257, 100, 300, "sigmoid", env="IBM_GEMM_CG=1"),
    C(S256_ACC, 300, 256, 4000, a_mn=True, b_mn=True, split_k=7, env="IBM_GEMM_CG=1"),
]

# switches that change no arithmetic: the rows (of CASES) whose code they touch must come out bit for bit as by default
BITEXACT_ENVS = {
    "IBM_GEMM_FP2=0": [c for c in CASES if c.bias and not c.atomic and c.kern in (HOT0, NT_BF16, P128_BF16, S64_BF16,
                                                                                   P256_F32, NT_AUX, S256_AUX)][:10],
    "IBM_GEMM_STAGGER=0": [c for c in CASES if c.kern[5] == 2 and (not c.atomic or c.split_k == 1)],
    "IBM_GEMM_PFAUX=1": [c for c in CASES if c.kern[3] == 1][:8],
    "IBM_GEMM_PFAUX=2": [c for c in CASES if c.kern[3] == 1][:8],
}


def find(case_id: str) -> Case:
    for c in CASES + ENV_CASES:
        if c.id == case_id:
            return c
    raise KeyError(case_id)


# ---- inputs, one launch, outputs ------------------------------------------------------------------------------------
SENTINEL = 12352.0           # exactly representable in bf16
MASK_FILL = 0xA5
COLSUM_INIT = 0.5


def _ru(x, m):
    return (x + m - 1) // m * m


def make_inputs(c: Case, device="cuda"):
    """Seeded operands as the contract stores them: zero pad columns up to the 8-element leading dimension, taps' B in
    blocks of round_up(K / taps, 64), an output with 3 extra rows and 16 extra columns of sentinel."""
    g = torch.Generator(device=device).manual_seed(zlib.crc32(c.id.encode()))
    M, N, K = c.M, c.N, c.K

    def rnd(rows, cols, ld, scale=1.0):
        t = torch.zeros(rows, ld, dtype=torch.bfloat16, device=device)
        t[:, :cols] = (torch.randn(rows, cols, generator=g, device=device) * scale).to(torch.bfloat16)
        return t

    s = 1.0 / K ** 0.5
    if c.taps > 1:
        Ct = K // c.taps
        Cp = _ru(Ct, 64)
        A = rnd(M + c.taps - 1, Ct, _ru(Ct, 8))
        if c.b_mn:
            B = torch.zeros(c.taps * Cp, _ru(N, 8), dtype=torch.bfloat16, device=device)
            for j in range(c.taps):
                B[j * Cp:j * Cp + Ct, :N] = rnd(Ct, N, N, s)
        else:
            B = torch.zeros(N, c.taps * Cp, dtype=torch.bfloat16, device=device)
            for j in range(c.taps):
                B[:, j * Cp:j * Cp + Ct] = rnd(N, Ct, Ct, s)
    else:
        A = rnd(K, M, _ru(M, 8)) if c.a_mn else rnd(M, K, _ru(K, 8))
        B = rnd(K, N, _ru(N, 8), s) if c.b_mn else rnd(N, K, _ru(K, 8), s)
    inp = {"A": A, "B": B}
    if c.bias:
        inp["bias"] = torch.randn(N, generator=g, device=device)
    if c.aux_mode:
        z = rnd(M, N, _ru(N, 8))
        if c.aux_mode == 2:
            import gemm_oracle
            z = gemm_oracle.act_fwd(z.float(), c.act).to(torch.bfloat16)
        inp["aux"] = z
    if c.mask_mode == 2:
        inp["mask"] = torch.randint(0, 256, (M + 2, N // 8 + 8), generator=g, device=device, dtype=torch.uint8)
    if c.accumulate:
        inp["d_init"] = torch.randn(M, N, generator=g, device=device)
    return inp


def launch(c: Case, inp):
    """One ops.gemm call on fresh output buffers; returns {"out", "mask"?, "colsum"?}."""
    from inferbiomechanics_b200 import ops
    M, N = c.M, c.N
    gran = 4 if c.out_f32 else 8
    ldd = _ru(N, gran) + 16
    out = torch.full((M + 3, ldd), SENTINEL, dtype=torch.float32 if c.out_f32 else torch.bfloat16, device="cuda")
    if c.accumulate:
        out[:M, :N] = inp["d_init"]
    res = {"out": out}
    kw = {}
    if c.mask_mode == 1:
        res["mask"] = kw["mask"] = torch.full((M + 2, N // 8 + 8), MASK_FILL, dtype=torch.uint8, device="cuda")
    elif c.mask_mode == 2:
        kw["mask"] = inp["mask"]
    if c.colsum:
        res["colsum"] = kw["colsum"] = torch.full((N + 8,), COLSUM_INIT, device="cuda")
    ops.gemm(inp["A"], inp["B"], out, M, N, c.K, a_mn=c.a_mn, b_mn=c.b_mn, bias=inp.get("bias"), act=c.act,
             aux=inp.get("aux"), aux_mode=c.aux_mode, accumulate=c.accumulate, split_k=c.split_k, taps=c.taps,
             mask_mode=c.mask_mode, **kw)
    return res


def profiled_launch(c: Case, inp):
    """launch() under torch.profiler: (set of gemm_kernel instantiations the launch ran, its outputs)."""
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        res = launch(c, inp)
        torch.cuda.synchronize()
    names = [e.name for e in prof.events()]
    names += [k.name for e in prof.events() for k in getattr(e, "kernels", [])]
    return {k for k in map(parse_kernel_name, names) if k is not None}, res
