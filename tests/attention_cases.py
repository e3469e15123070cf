"""The attention case table: rows for every instantiation of the attention kernels (csrc/attention.cu, attention_tc.cu,
attention_bwd_long.cu), each naming the instantiations its launches must reach.  TEST INFRASTRUCTURE ONLY; used by
tests/test_gpu_attention_matrix.py and its environment-switch worker (tests/workers/attention_env_worker.py).

An instantiation is named as the profiler shows it, template arguments normalised: 'attn_fwd_pipe_kernel<64>',
'attn_bwd_long_kernel<64,64,1,0,416>', 'attn_bwd_tc_kernel'.  The dispatch rules the rows are chosen from:
  ibm_attention_fwd   T <= 64, hd (64, 64): attn_fwd_tc_kernel under IBM_ATTN_FWD=tc
                      T <= 64, hd_qk == hd_v in {32, 48, 64}, o 16-byte aligned, ldo % 8 == 0: attn_fwd_pipe_kernel<hd>
                      T > 64: attn_fwd_long_kernel, two CTAs per SM (<HQ,HV,4,416,2>) iff T <= 208 and
                      2 * smem + 4096 <= 227 KB, else <HQ,HV,8,512,1>; IBM_ATTN_LONG_ONE forces the latter,
                      IBM_ATTN_LONG=0 the one-shot kernel
                      everything else: the one-shot attn_fwd_kernel<HQ,HV>
  ibm_attention_bwd   head_dim 64: attn_bwd_tc_kernel (attn_bwd_kernel<64> under IBM_ATTN_BWD=mma); 32, 48: attn_bwd_kernel
  ibm_attention_bwd_long  attn_bwd_long_kernel<HQ,HV,dv != NULL,any dbias,416 iff T <= 208 else 512>
A backward row with dbias runs twice, with and without the bias accumulators, so it reaches both DB variants.
"""
from __future__ import annotations

import dataclasses
import math
import re

import torch

import attention_oracle as ao

SENTINEL = -1234.0              # bf16-exact; output cells no launch may write
BIAS_INIT, BIAS_SENTINEL = 0.5, -777.0
KPAD = 8
PAIRS = [(64, 64), (48, 48), (32, 32), (64, 8), (80, 8), (96, 8), (112, 8), (128, 8)]


def long_fwd_two(hq, hv, T):
    """The two-CTA long forward variant is taken (launch_fwd_long in attention.cu)."""
    tp = (T + 15) // 16 * 16
    smem = 2 * tp * ((hq + KPAD) + (hv + KPAD)) * 2
    return (T + 15) // 16 <= 13 and 2 * smem + 4096 <= 227 * 1024


def K_PIPE(hd):
    return f"attn_fwd_pipe_kernel<{hd}>"


def K_ONE(hq, hv):
    return f"attn_fwd_kernel<{hq},{hv}>"


def K_LONG(hq, hv, two):
    return f"attn_fwd_long_kernel<{hq},{hv},4,416,2>" if two else f"attn_fwd_long_kernel<{hq},{hv},8,512,1>"


K_FWD_TC, K_BWD_TC = "attn_fwd_tc_kernel", "attn_bwd_tc_kernel"


def K_BWD(hd):
    return f"attn_bwd_kernel<{hd}>"


def K_BWDL(hq, hv, db, maxt):
    return f"attn_bwd_long_kernel<{hq},{hv},{int(hv >= 16)},{int(db)},{maxt}>"


ALL_KERNELS = sorted(
    [K_FWD_TC, K_BWD_TC] + [K_PIPE(h) for h in (64, 48, 32)] + [K_BWD(h) for h in (64, 48, 32)]
    + [K_ONE(hq, hv) for hq, hv in PAIRS] + [K_LONG(hq, hv, t) for hq, hv in PAIRS for t in (True, False)]
    + [K_BWDL(hq, hv, db, m) for hq, hv in PAIRS for db in (0, 1) for m in (416, 512)])

_KNAME = re.compile(r"(attn_\w+_kernel)(?:<([^>]*)>)?")


def parse_kernel_name(name: str):
    """'void ibm::attn::attn_bwd_long_kernel<(int)64, (int)8, (bool)0, true, 416>(...)' -> 'attn_bwd_long_kernel<64,8,0,1,416>'."""
    m = _KNAME.search(name)
    if m is None:
        return None
    if m.group(2) is None:
        return m.group(1)
    vals = []
    for a in m.group(2).split(","):
        a = re.sub(r"\((?:int|bool)\)", "", a).strip()
        vals.append("1" if a == "true" else "0" if a == "false" else str(int(a)))
    return f"{m.group(1)}<{','.join(vals)}>"


@dataclasses.dataclass(frozen=True)
class Case:
    kind: str            # "fwd" | "bwd" (ibm_attention_bwd, fused qkv) | "bwdl" (ibm_attention_bwd_long)
    kerns: tuple         # the instantiations the row's launches must reach
    n_win: int
    T: int
    H: int
    hq: int
    hv: int
    scale: str = "rsqrt"  # "1" | "rsqrt" (1/sqrt(hd_qk)) | "wide" (about 80 log2 units of spread per row)
    out_off: int = 0     # column offset (bf16 elements) of the outputs in their buffers: 2 = 4-byte, not 16-byte aligned
    dbias: bool = True
    env: str = ""

    @property
    def id(self):
        s = f"{self.kind}:{self.n_win}x{self.T}x{self.H}:{self.hq}-{self.hv}:{self.scale}"
        if self.out_off:
            s += f":off{self.out_off}"
        if not self.dbias and self.kind != "fwd":
            s += ":nobias"
        if self.env:
            s += ":" + self.env
        return s

    @property
    def scale_value(self):
        if self.scale == "1":
            return 1.0
        if self.scale == "rsqrt":
            return ao.f32(1 / math.sqrt(self.hq))
        # randn rows: s = q.k has standard deviation sqrt(hq); T keys span about 5 of them
        return ao.f32(80 / (ao.LOG2E * 5 * math.sqrt(self.hq)))


def _fwd(n_win, T, H, hq, hv, **kw):
    off = kw.get("out_off", 0)
    if T <= 64 and hq == hv and off % 8 == 0 and kw.get("env") != "IBM_ATTN_FWD=tc":
        k = K_PIPE(hq)
    elif T <= 64 and kw.get("env") == "IBM_ATTN_FWD=tc":
        k = K_FWD_TC
    elif T > 64 and kw.get("env") != "IBM_ATTN_LONG=0":
        k = K_LONG(hq, hv, long_fwd_two(hq, hv, T) and kw.get("env") != "IBM_ATTN_LONG_ONE=1")
    else:
        k = K_ONE(hq, hv)
    return Case("fwd", (k,), n_win, T, H, hq, hv, **kw)


def _bwd(n_win, T, H, hd, **kw):
    k = K_BWD_TC if hd == 64 and kw.get("env") != "IBM_ATTN_BWD=mma" else K_BWD(hd)
    return Case("bwd", (k,), n_win, T, H, hd, hd, **kw)


def _bwdl(n_win, T, H, hq, hv, **kw):
    m = 416 if T <= 208 else 512
    ks = (K_BWDL(hq, hv, 1, m), K_BWDL(hq, hv, 0, m)) if kw.get("dbias", True) else (K_BWDL(hq, hv, 0, m),)
    return Case("bwdl", ks, n_win, T, H, hq, hv, **kw)


CASES = [
    # pipelined short forward; (2003, 50, 8, 64) is the denoiser's shape
    _fwd(2003, 50, 8, 64, 64), _fwd(1, 1, 1, 64, 64, scale="1"), _fwd(7, 64, 2, 64, 64, scale="wide"),
    _fwd(5, 17, 3, 64, 64),
    _fwd(9, 15, 3, 48, 48), _fwd(1, 2, 1, 48, 48, scale="1"), _fwd(13, 63, 2, 48, 48, scale="wide"),
    _fwd(11, 16, 4, 32, 32, scale="1"), _fwd(3, 64, 5, 32, 32), _fwd(301, 2, 7, 32, 32, scale="wide"),
    # one-shot forward: outputs at a 4-byte aligned column, and the value-width-8 pairs at T <= 64
    _fwd(3, 50, 8, 64, 64, out_off=2), _fwd(1, 1, 3, 64, 64, out_off=2, scale="wide"),
    _fwd(2, 17, 1, 48, 48, out_off=2), _fwd(5, 63, 2, 48, 48, out_off=2, scale="1"),
    _fwd(5, 64, 2, 32, 32, out_off=2), _fwd(4, 16, 6, 32, 32, out_off=2, scale="wide"),
] + [c for hq in (64, 80, 96, 112, 128) for c in (_fwd(3, 50, 1, hq, 8, scale="1"), _fwd(2, 17, 2, hq, 8, scale="wide"),
                                                  _fwd(1, 64, 1, hq, 8, out_off=2))
] + [
    # long forward, both variants of every pair; (1201, 200, 3, 48) is the analysis shape
    _fwd(1201, 200, 3, 48, 48),
] + [c for hq, hv in PAIRS for c in (
    _fwd(3, 65, 2, hq, hv, scale="wide"), _fwd(2, 129, 1, hq, hv, out_off=2),
    _fwd(5, 127 if not long_fwd_two(hq, hv, 208) else 208, 3, hq, hv, scale="1"), _fwd(1, 128, 8, hq, hv),
    _fwd(2, 209, 2, hq, hv, scale="wide"), _fwd(3, 256, 1, hq, hv), _fwd(1, 255, 4, hq, hv, scale="1", out_off=2))
] + [
    # fused short backward; (2003, 50, 8, 64) is the denoiser's shape
    _bwd(2003, 50, 8, 64), _bwd(1, 1, 1, 64, scale="1"), _bwd(6, 64, 2, 64, scale="wide"), _bwd(5, 17, 3, 64, dbias=False),
    _bwd(9, 33, 3, 48), _bwd(1, 64, 1, 48, scale="wide"), _bwd(13, 15, 2, 48, scale="1"),
    _bwd(1500, 17, 4, 32), _bwd(3, 2, 5, 32, scale="1"), _bwd(7, 63, 3, 32, scale="wide"),
    # long backward: both MAXT variants of every pair, each with and without the bias sums
    _bwdl(1201, 200, 3, 48, 48),
] + [c for hq, hv in PAIRS for c in (
    _bwdl(3, 65, 2, hq, hv, scale="wide"), _bwdl(2, 208, 1, hq, hv, out_off=2), _bwdl(5, 129, 3, hq, hv, scale="1"),
    _bwdl(2, 209, 2, hq, hv), _bwdl(1, 256, 3, hq, hv, scale="wide", out_off=2), _bwdl(3, 255, 1, hq, hv, scale="1"))
]

ENV_CASES = [
    _fwd(701, 50, 8, 64, 64, env="IBM_ATTN_FWD=tc"), _fwd(1, 1, 1, 64, 64, scale="1", env="IBM_ATTN_FWD=tc"),
    _fwd(6, 64, 3, 64, 64, scale="wide", env="IBM_ATTN_FWD=tc"), _fwd(5, 17, 2, 64, 64, env="IBM_ATTN_FWD=tc"),
    _bwd(701, 50, 8, 64, env="IBM_ATTN_BWD=mma"), _bwd(1, 1, 1, 64, scale="1", env="IBM_ATTN_BWD=mma"),
    _bwd(6, 64, 2, 64, scale="wide", env="IBM_ATTN_BWD=mma"), _bwd(5, 17, 3, 64, dbias=False, env="IBM_ATTN_BWD=mma"),
] + [c for hq, hv in PAIRS for c in (_fwd(3, 200, 2, hq, hv, env="IBM_ATTN_LONG=0"),
                                     _fwd(2, 256, 1, hq, hv, scale="wide", env="IBM_ATTN_LONG=0"),
                                     _fwd(4, 65, 3, hq, hv, env="IBM_ATTN_LONG_ONE=1"),
                                     _fwd(2, 176, 2, hq, hv, scale="wide", env="IBM_ATTN_LONG_ONE=1"))]


def find(cid: str) -> Case:
    for c in CASES + ENV_CASES:
        if c.id == cid:
            return c
    raise KeyError(cid)


# ---- buffers --------------------------------------------------------------------------------------------------------
def _padded(rows, cols, ld, fill, device, col0=0):
    """(buffer [rows + 3, ld] filled with `fill`, view of rows [0, rows) and columns [col0, col0 + cols))."""
    buf = torch.full((rows + 3, ld), fill, dtype=torch.bfloat16, device=device)
    return buf, buf[:rows, col0:col0 + cols]


def make_inputs(c: Case, device="cuda", seed=0, q_zero=False, needle=False):
    """Operands of one row: every input column outside the heads, and every row past the last window, is NaN.  Outputs
    are views into sentinel-filled buffers with their own leading dimensions (and column offset out_off).
    q_zero: the uniform probe (q = 0).  needle: the needle probe (see needle_inputs)."""
    g = torch.Generator(device="cpu").manual_seed(seed * 7919 + c.T * 131 + c.hq * 17 + c.hv + c.n_win)
    rows, H = c.n_win * c.T, c.H

    def rnd(n):
        return torch.randn(rows, n, generator=g).to(torch.bfloat16).to(device)

    inp = {}
    if c.kind == "bwd":
        d = H * c.hq
        kv_off = d + 16
        ld = 2 * kv_off + d + 24
        buf, _ = _padded(rows, 0, ld, float("nan"), device)
        for j in range(3):
            buf[:rows, j * kv_off:j * kv_off + d] = rnd(d)
        inp["qkv"], inp["kv_off"] = buf, kv_off
        inp["q"], inp["k"], inp["v"] = buf[:, :d], buf[:, kv_off:kv_off + d], buf[:, 2 * kv_off:2 * kv_off + d]
    else:
        for j, (name, hd) in enumerate((("q", c.hq), ("k", c.hq), ("v", c.hv))):
            buf, view = _padded(rows, H * hd, H * hd + 8 * (j + 1), float("nan"), device)
            view.copy_(rnd(H * hd))
            inp[name] = buf
    if needle:
        needle_inputs(c, inp, g)
    if q_zero:
        inp["q"][:rows, :H * c.hq] = 0
    if c.kind != "fwd":
        buf, view = _padded(rows, H * c.hv, H * c.hv + 16, float("nan"), device)
        view.copy_(rnd(H * c.hv) if not needle else inp.pop("do_needle"))
        inp["do"] = buf
    if c.kind == "bwdl":
        o, _, _ = ao.attention_fwd_ref(inp["q"], inp["k"], inp["v"], c.n_win, c.T, H, c.hq, c.hv, c.scale_value)
        buf, view = _padded(rows, H * c.hv, H * c.hv + 8, float("nan"), device)
        view.copy_(o.to(torch.bfloat16))
        inp["o"] = buf
    return inp


def _out_geometry(c: Case):
    """{name: (ld, col0, cols)} of the output buffers of a row (the backward's fused dqkv: see out_views)."""
    H = c.H
    if c.kind == "fwd":
        return {"o_buf": (H * c.hv + 16, c.out_off, H * c.hv)}
    if c.kind == "bwd":
        return {"dqkv": (2 * (H * c.hq + 16) + H * c.hq + 24, 0, None)}
    geo = {"dq_buf": (H * c.hq + 16, c.out_off, H * c.hq), "dk_buf": (H * c.hq + 24, c.out_off, H * c.hq)}
    if c.hv >= 16:
        geo["dv_buf"] = (H * c.hv + 32, c.out_off, H * c.hv)
    return geo


def out_views(c: Case, out):
    """The output views the kernel writes (rows [0, n_win*T), the heads' columns) of a row's output buffers."""
    rows = c.n_win * c.T
    if c.kind == "bwd":
        d, kv = c.H * c.hq, c.H * c.hq + 16
        b = out["dqkv"]
        return {"dq": b[:rows, :d], "dk": b[:rows, kv:kv + d], "dv": b[:rows, 2 * kv:2 * kv + d]}
    return {name[:-4]: out[name][:rows, c0:c0 + n] for name, (ld, c0, n) in _out_geometry(c).items()}


def written_mask(c: Case, out):
    """{buffer name: bool mask of the cells the launch may write}."""
    masks = {}
    rows = c.n_win * c.T
    for name, (ld, c0, n) in _out_geometry(c).items():
        m = torch.zeros_like(out[name], dtype=torch.bool)
        if c.kind == "bwd":
            d, kv = c.H * c.hq, c.H * c.hq + 16
            for j in range(3):
                m[:rows, j * kv:j * kv + d] = True
        else:
            m[:rows, c0:c0 + n] = True
        masks[name] = m
    return masks


def _outputs(c: Case, device):
    return {name: torch.full((c.n_win * c.T + 3, ld), SENTINEL, dtype=torch.bfloat16, device=device)
            for name, (ld, _, _) in _out_geometry(c).items()}


def _bias(c: Case, n, device):
    b = torch.full((n + 8,), BIAS_SENTINEL, device=device)
    b[:n] = BIAS_INIT
    return b


def launch(c: Case, inp, with_bias=None, device="cuda"):
    """One launch of the row's entry point; returns the output buffers (and the bias accumulators when used)."""
    from inferbiomechanics_b200 import ops
    use_bias = c.dbias if with_bias is None else with_bias
    out = _outputs(c, device)
    v = out_views(c, out)
    H, s = c.H, c.scale_value
    if c.kind == "fwd":
        ops.attention_fwd(inp["q"], inp["k"], inp["v"], v["o"], c.n_win, c.T, H, c.hq, c.hv, s)
    elif c.kind == "bwd":
        kv = inp["kv_off"]
        if use_bias:
            out["dbias"] = _bias(c, 3 * kv, device)
        ops.attention_bwd(inp["qkv"], kv, inp["do"], out["dqkv"], c.n_win, c.T, H, c.hq, s, dbias=out.get("dbias"))
    else:
        if use_bias:
            out["dbq"], out["dbk"] = _bias(c, H * c.hq, device), _bias(c, H * c.hq, device)
            if c.hv >= 16:
                out["dbv"] = _bias(c, H * c.hv, device)
        ops.attention_bwd_long(inp["q"], inp["k"], inp["v"], inp["o"], inp["do"], v["dq"], v["dk"], v.get("dv"),
                               c.n_win, c.T, H, c.hq, c.hv, s, dbq=out.get("dbq"), dbk=out.get("dbk"), dbv=out.get("dbv"))
    return out


def launch_all(c: Case, inp):
    """The row's launches: a backward row with dbias runs with and then without the accumulators."""
    res = launch(c, inp)
    if c.kind != "fwd" and c.dbias:
        res["nobias"] = launch(c, inp, with_bias=False)
    return res


def profiled_launch(c: Case, inp):
    """launch_all under torch.profiler: (set of attention instantiations the launches ran, their outputs)."""
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        res = launch_all(c, inp)
        torch.cuda.synchronize()
    names = [e.name for e in prof.events()]
    names += [k.name for e in prof.events() for k in getattr(e, "kernels", [])]
    return {k for k in map(parse_kernel_name, names) if k is not None}, res


# ---- probes ---------------------------------------------------------------------------------------------------------
def needle_alpha(scale: float) -> float:
    """The power of two alpha with 2 alpha scale log2(e) >= 30: a one-bit mismatch costs a factor 2^-30."""
    return 2.0 ** math.ceil(math.log2(15.0 / (scale * ao.LOG2E)))


def needle_inputs(c: Case, inp, g):
    """For each (window, head) a permutation pi of the frames: k_j holds the 8 sign bits of j in its first 8 columns,
    q_i alpha times those of pi(i), so that query i attends to key pi(i) alone; v and dO are +-[0.5, 2) so that an
    output equals its needle to within 2^-20.  Stores pi in inp['pi'] ([n_win, H, T]) and dO in inp['do_needle']."""
    n_win, T, H, rows = c.n_win, c.T, c.H, c.n_win * c.T
    dev = inp["q"].device
    pi = torch.rand(n_win, H, T, generator=g).argsort(-1)
    bits = ((torch.arange(T).unsqueeze(-1) >> torch.arange(8)) & 1).double() * 2 - 1          # [T, 8]
    a = needle_alpha(c.scale_value)
    Kh = torch.zeros(n_win, H, T, c.hq, dtype=torch.float64)
    Kh[..., :8] = bits
    Qh = torch.zeros_like(Kh)
    Qh[..., :8] = a * bits[pi]

    def mag(n):
        return ((torch.rand(rows, n, generator=g) * 1.5 + 0.5) * (torch.randint(0, 2, (rows, n), generator=g) * 2 - 1))
    inp["q"][:rows, :H * c.hq] = ao.flat(Qh).to(torch.bfloat16).to(dev)
    inp["k"][:rows, :H * c.hq] = ao.flat(Kh).to(torch.bfloat16).to(dev)
    inp["v"][:rows, :H * c.hv] = mag(H * c.hv).to(torch.bfloat16).to(dev)
    inp["pi"] = pi.to(dev)
    inp["do_needle"] = mag(H * c.hv).to(torch.bfloat16).to(dev)
