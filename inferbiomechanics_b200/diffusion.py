"""DDPM schedule, noising and reverse sampling on libibm_b200 (builder-owned spec, DESIGN.md D-1;
the reference has no diffusion code).

  betas = linspace(1e-4, 2e-2, 1000) (fp64 → fp32 tables)          q_sample: fused kernel, optional
  x_t   = sqrt(abar_t) x0 + sqrt(1-abar_t) eps                      on-device Philox noise
  x_{t-1} = c1_t x0_hat + c2_t x_t + [t>0] sigma_t z                posterior step: fused kernel

Few-step sampling (DDIM, Song et al. 2021) walks a respaced sequence ts = round(linspace(T-1, 0, S)) with the
same kernel: each step from t to its successor p = succ[t] is linear in (x0_hat, x_t, z) with per-timestep tables
(``ddim_schedule``); eta = 1 over all T steps is the DDPM chain above, bit for bit.

The reverse loop runs the denoiser forward + one fused posterior kernel per step; the timestep lives
in device memory so two consecutive steps are captured once in a CUDA graph and replayed (sampling at
512 windows/GPU is launch-bound otherwise).  Windows are independent: multi-GPU sampling shards them
with no collective.

Classifier-free guidance (Ho & Salimans 2022) with scale s != 1 runs the forward on 2B windows per step, the B conditioned
ones and the same B with all-zero kinematics (the null condition the trainer's ``cond_drop_prob`` teaches), and one guided
step kernel combines x0_hat = u + s (c - u) before the same update; s = 0 is unconditional sampling.

Inpainting (MDM's ``p_mean_variance`` for an x0-predicting model): given known values y and a known-mask, every step
replaces the known entries of x0_hat (after the guided combination) by y before the unchanged update.  The last step of
either sampler has coef_x0 = 1, coef_xt = 0 and no noise, so the sample equals y exactly wherever the mask is set.
"""
from __future__ import annotations

import math
from typing import Callable, Optional

import numpy as np
import torch

from . import ops


def ddim_schedule(ddim_steps: int, eta: float = 0.0, num_timesteps: int = 1000, beta_start: float = 1e-4,
                  beta_end: float = 2e-2) -> dict:
    """Host tables (numpy, no GPU) of S = ``ddim_steps``-step DDIM sampling over the trained schedule (DESIGN.md D-1).

    ``ts`` (int64 [S]) = round(linspace(T-1, 0, S)): the timesteps walked, strictly decreasing from T-1.  The step from
    t = ts[i] to p = ts[i+1] (p = -1 after the last, abar[-1] := 1) is, with a = abar in fp64,
      sigma = eta sqrt((1-a_p)/(1-a_t)) sqrt(1 - a_t/a_p),   c = sqrt(max(1 - a_p - sigma^2, 0))
      x_p   = coef_x0[t] x0_hat + coef_xt[t] x_t + [t>0] sigma[t] z
      coef_x0 = sqrt(a_p) - c sqrt(a_t)/sqrt(1-a_t),   coef_xt = c/sqrt(1-a_t)
    which is sqrt(a_p) x0_hat + c eps_hat + sigma z for eps_hat = (x_t - sqrt(a_t) x0_hat)/sqrt(1-a_t).  ``coef_x0``,
    ``coef_xt``, ``sigma`` (fp32 [T]) and ``succ`` (int32 [T], = p) are indexed by timestep, 0 off the sequence.  The
    expressions are evaluated in exactly this order: at S = T and eta = 1 the fp32 tables then equal the DDPM
    posterior tables bit for bit (sigma at t >= 1; the step at t = 0 draws no noise in either)."""
    T = num_timesteps
    _check_schedule(T, None, ddim_steps, eta)
    abar = np.cumprod(1.0 - np.linspace(beta_start, beta_end, T, dtype=np.float64))
    ts = np.round(np.linspace(T - 1, 0, ddim_steps)).astype(np.int64)
    succ = np.append(ts[1:], -1)
    a_t = abar[ts]
    a_p = np.where(succ >= 0, abar[np.maximum(succ, 0)], 1.0)
    sigma = eta * np.sqrt((1.0 - a_p) / (1.0 - a_t)) * np.sqrt(1.0 - a_t / a_p)
    c = np.sqrt(np.maximum(1.0 - a_p - sigma * sigma, 0.0))
    tab = dict(coef_x0=np.sqrt(a_p) - c * np.sqrt(a_t) / np.sqrt(1.0 - a_t), coef_xt=c / np.sqrt(1.0 - a_t), sigma=sigma)
    out = {k: np.zeros(T, dtype=np.float32) for k in tab}
    for k, v in tab.items():
        out[k][ts] = v.astype(np.float32)
    out["succ"] = np.zeros(T, dtype=np.int32)
    out["succ"][ts] = succ
    out["ts"] = ts
    return out


def check_guidance_scale(guidance_scale: float) -> None:
    if not (math.isfinite(guidance_scale) and guidance_scale >= 0.0):
        raise ValueError(f"guidance_scale must be finite and >= 0 (1 = no guidance, 0 = unconditional), got {guidance_scale}")


MAX_NUM_SAMPLES = 64             # draws per window: the bound of the ensemble scoring kernel (ops.ENSEMBLE_MAX_DRAWS)


def check_num_samples(num_samples: Optional[int]) -> None:
    if num_samples is not None and not (isinstance(num_samples, int) and 1 <= num_samples <= MAX_NUM_SAMPLES):
        raise ValueError(f"num_samples must be None or an int in [1, {MAX_NUM_SAMPLES}], got {num_samples!r}")


def known_mask_words(mask: torch.Tensor, rows: int) -> torch.Tensor:
    """int32 row words of a bool known-mask (rows, 30), or (30,) for every row: bit c of word m is set iff channel c of row m
    is known (the ``known_mask`` of ``ops.posterior_step``).  A (30,) mask gives an expanded view of one word."""
    w = (mask.to(torch.int32) << torch.arange(30, dtype=torch.int32, device=mask.device)).sum(-1, dtype=torch.int32)
    return w.reshape(1).expand(rows) if mask.dim() == 1 else w.reshape(rows)


def check_known(known, known_mask, B: int, F: Optional[int], T: int, steps: Optional[int], device=None) -> bool:
    """ValueError unless (``known``, ``known_mask``) are inpainting inputs for B windows of F frames (None: not checked):
    both or neither, known fp32 (B, F, 30) (on ``device`` if given), known_mask bool (B, F, 30) or (30,), and the whole
    chain (a truncated DDPM chain stops before the step that returns the known values).  True when both are given."""
    if known is None and known_mask is None:
        return False
    if known is None or known_mask is None:
        raise ValueError("known and known_mask go together: give both or neither")
    if not isinstance(known, torch.Tensor) or known.dtype != torch.float32 or known.dim() != 3 or known.shape[0] != B \
            or known.shape[2] != 30 or (F is not None and known.shape[1] != F):
        raise ValueError(f"known must be an fp32 tensor of shape (B={B}, F={F if F is not None else 'F'}, 30)"
                         + (f", got {known.dtype} {tuple(known.shape)}" if isinstance(known, torch.Tensor) else ""))
    if device is not None and not _on(known, device):
        raise ValueError(f"known must be on {device}, got {known.device}")
    if not isinstance(known_mask, torch.Tensor) or known_mask.dtype != torch.bool or \
            tuple(known_mask.shape) not in ((30,), tuple(known.shape)):
        raise ValueError(f"known_mask must be a bool tensor of shape (30,) or {tuple(known.shape)}"
                         + (f", got {known_mask.dtype} {tuple(known_mask.shape)}" if isinstance(known_mask, torch.Tensor) else ""))
    if steps is not None and steps < T:
        raise ValueError(f"inpainting needs the whole chain: steps={steps} < {T} stops before the known values are returned")
    return True


def _on(t: torch.Tensor, device) -> bool:
    device = torch.device(device)
    return t.device.type == device.type and (device.index is None or t.device.index == device.index)


def _check_schedule(T: int, steps: Optional[int], ddim_steps: Optional[int], eta: float) -> None:
    if steps is not None and ddim_steps is not None:
        raise ValueError("give either steps (a truncated DDPM chain) or ddim_steps (a respaced DDIM sequence), not both")
    if ddim_steps is not None and not 1 <= ddim_steps <= T:
        raise ValueError(f"ddim_steps must lie in [1, {T}], got {ddim_steps}")
    if not 0.0 <= eta <= 1.0:
        raise ValueError(f"eta must lie in [0, 1], got {eta}")
    if eta != 0.0 and ddim_steps is None:
        raise ValueError("eta applies to DDIM sampling only: give ddim_steps")


class GaussianDiffusion:
    def __init__(self, num_timesteps: int = 1000, beta_start: float = 1e-4, beta_end: float = 2e-2, device="cuda"):
        self.T = num_timesteps
        self.beta_start, self.beta_end = beta_start, beta_end
        betas = np.linspace(beta_start, beta_end, num_timesteps, dtype=np.float64)
        alphas = 1.0 - betas
        abar = np.cumprod(alphas)
        abar_prev = np.concatenate([[1.0], abar[:-1]])
        post_var = betas * (1.0 - abar_prev) / (1.0 - abar)
        post_logvar = np.log(np.concatenate([post_var[1:2], post_var[1:]]))
        f = lambda a: torch.from_numpy(a.astype(np.float32)).to(device)
        self.sqrt_abar = f(np.sqrt(abar))
        self.sqrt_one_minus_abar = f(np.sqrt(1.0 - abar))
        self.coef_x0 = f(betas * np.sqrt(abar_prev) / (1.0 - abar))
        self.coef_xt = f((1.0 - abar_prev) * np.sqrt(alphas) / (1.0 - abar))
        self.sigma = f(np.exp(0.5 * post_logvar))
        self.device = torch.device(device)
        self._graphs = {}
        self._ddim = {}                 # (S, eta) -> device tables of ddim_schedule
        # reverse sampling: take the time MLP from the engine's per-timestep table (DenoiserEngine.temb_table) instead of
        # evaluating it every step; False re-runs it per step (parity check, tests/test_gpu_models.py)
        self.use_temb_table = True

    # ---- forward process -----------------------------------------------------------------------
    def q_sample(self, x0: torch.Tensor, t: torch.Tensor, eps: Optional[torch.Tensor] = None, *, xt_f32=None, xt_bf16=None,
                 bf16_ld: int = 0, seed: int = 0, offset: int = 0, eps_out=None):
        """x0 (B,F,30) fp32, t (B,) int32.  eps=None ⇒ on-device Philox(seed, offset)."""
        if xt_f32 is None and xt_bf16 is None:
            xt_f32 = torch.empty_like(x0)
        ops.q_sample(x0, eps, t, self.sqrt_abar, self.sqrt_one_minus_abar, xt_f32=xt_f32, xt_bf16=xt_bf16, bf16_ld=bf16_ld,
                     seed=seed, offset=offset, eps_out=eps_out)
        return xt_f32

    def ddim_tables(self, ddim_steps: int, eta: float = 0.0) -> dict:
        """``ddim_schedule`` of this schedule on the device (cached per (S, eta)): coef_x0 / coef_xt / sigma fp32 [T],
        succ int32 [T], ts (host numpy)."""
        key = (ddim_steps, float(eta))
        tab = self._ddim.get(key)
        if tab is None:
            h = ddim_schedule(ddim_steps, eta, self.T, self.beta_start, self.beta_end)
            tab = {k: v if k == "ts" else torch.from_numpy(v).to(self.device) for k, v in h.items()}
            self._ddim[key] = tab
        return tab

    # ---- reverse process -----------------------------------------------------------------------
    @torch.no_grad()
    def sample(self, model, B: int, *, x_T: Optional[torch.Tensor] = None, noise: Optional[Callable[[int], torch.Tensor]] = None,
               steps: Optional[int] = None, seed: int = 0, use_graph: bool = True, ddim_steps: Optional[int] = None,
               eta: float = 0.0, guidance_scale: float = 1.0, num_samples: Optional[int] = None,
               known: Optional[torch.Tensor] = None, known_mask: Optional[torch.Tensor] = None) -> torch.Tensor:
        """Reverse-sample x_0 (B,F,30) for the kinematics already packed in model.engine().xc(B, False)
        (columns 30…).  ``noise(t)`` supplies z per step for parity tests; None ⇒ on-device Philox.

        ``ddim_steps=None``: the DDPM chain; ``steps`` < T runs only its first ``steps`` steps and returns x at timestep
        T - steps (a truncated chain, not a sample).  ``ddim_steps=S``: S-step DDIM with noise scale ``eta`` in [0, 1]
        (``ddim_schedule``); eta = 0 draws no noise after x_T.  ``noise(t)`` is called with each timestep walked.

        ``guidance_scale`` s != 1: classifier-free guidance with either sampler.  The kinematics of xc(B) are copied into
        the first half of xc(2B) and the second half gets the null condition (zeros); x_T goes into both halves, each step
        runs the forward on 2B windows and the guided step kernel.  s = 1 runs the unguided loop, s = 0 samples
        unconditionally.  The result depends on s only through the prediction: x_T and the noise are those of s = 1.

        ``num_samples`` K (1..64): K independent draws per window.  The B packed conditions are copied into K consecutive
        blocks of xc(B*K) and the loop above runs on B*K windows; the result is (K, B, F, 30), draw k of window b at row
        k*B*F + b*F + f of the fp32 state (the layout ``ops.ensemble_score`` reads).  x_T and the noise are Philox draws indexed
        by element, so the draws are independent and draw 0 starts from the x_T and noise of a call without ``num_samples``.

        ``known`` (fp32 (B, F, 30) on the device) with ``known_mask`` (bool, (B, F, 30) or (30,) for every row): inpainting.
        Every step replaces the known entries of x0_hat (after the guidance combination) by ``known`` before the unchanged
        update, so the sample equals ``known`` exactly where the mask is set, in every draw; unknown entries of ``known`` are
        never read into the result.  x_T and the noise are those of a call without it.  Needs the whole chain (no
        ``steps`` < T).  The mask is packed into row words per call and both are copied into buffers of the graph cache
        entry, so calls with other values or masks replay the same graph."""
        _check_schedule(self.T, steps, ddim_steps, eta)
        check_guidance_scale(guidance_scale)
        check_num_samples(num_samples)
        words = None
        if check_known(known, known_mask, B, None, self.T, steps, self.device):
            F = model.engine().F
            if known.shape[1] != F:
                raise ValueError(f"known must have the model's F={F} frames per window, got {tuple(known.shape)}")
            known = known.reshape(B * F, 30)
            words = known_mask_words(known_mask.to(self.device), B * F)
        return self._sample(model, B, x_T=x_T, noise=noise, steps=steps, seed=seed, use_graph=use_graph, ddim_steps=ddim_steps,
                            eta=eta, guidance_scale=guidance_scale, num_samples=num_samples, known=known, words=words)

    def _sample(self, model, B: int, *, x_T, noise, steps, seed, use_graph, ddim_steps, eta, guidance_scale, num_samples,
                known: Optional[torch.Tensor], words: Optional[torch.Tensor]) -> torch.Tensor:
        """``sample`` after its checks: ``known`` fp32 (rows, 30) and ``words`` int32 (rows,) (``known_mask_words``) of the
        caller's B windows, or None; a call on B*K windows repeats them K times."""
        if num_samples is not None:
            eng = model.engine()
            src = eng.xc(B, False)
            dst = eng.xc(B * num_samples, False)
            M = src.shape[0]
            for k in range(num_samples):
                dst[k * M:(k + 1) * M].copy_(src)
            x0 = self._sample(model, B * num_samples, x_T=x_T, noise=noise, steps=steps, seed=seed, use_graph=use_graph,
                              ddim_steps=ddim_steps, eta=eta, guidance_scale=guidance_scale, num_samples=None, known=known,
                              words=words)
            return x0.view(num_samples, B, eng.F, 30)
        guided = guidance_scale != 1.0
        inpaint = known is not None
        eng = model.engine()
        F, M = eng.F, B * eng.F
        xc = eng.xc(B, False)
        if guided:
            # rows 0..M-1 conditional, M..2M-1 the same windows with all-zero kinematics
            xc2 = eng.xc(2 * B, False)
            xc2[:M].copy_(xc)
            ops.cond_dropout(xc2[M:], B, F, 30, eng.c_in, 1.0, 0, 0)
        if ddim_steps is None:
            sched = None
            ts = range(self.T - 1, self.T - 1 - (self.T if steps is None else steps), -1)
            coef_x0, coef_xt, sigma, succ = self.coef_x0, self.coef_xt, self.sigma, None
        else:
            sched = (ddim_steps, float(eta))
            tab = self.ddim_tables(ddim_steps, eta)
            ts = tab["ts"].tolist()
            coef_x0, coef_xt, sigma, succ = tab["coef_x0"], tab["coef_xt"], tab["sigma"], tab["succ"]
        # the captured launches read the schedule's tables through baked-in pointers, so each schedule has its own graph;
        # the guidance scale is a baked launch argument; inpainting reads the known values and mask words from the entry's
        # buffers, refilled per call
        key = (id(model), B, sched) if not guided else (id(model), B, sched, float(guidance_scale))
        if inpaint:
            key += ("inpaint",)
        st = self._graphs.get(key)
        if st is None or st["model"] is not model:
            # the entry holds the model (its id() cannot be recycled while cached), the schedule's tables and, below, the
            # time-MLP table the captured launches read
            st = dict(x=torch.empty(M, 30, dtype=torch.float32, device=self.device),
                      t_a=torch.zeros(1, dtype=torch.int32, device=self.device),
                      t_b=torch.zeros(1, dtype=torch.int32, device=self.device), graph=None, seed=None, model=model, table=None,
                      table_key=None, sched_tables=(coef_x0, coef_xt, sigma, succ))
            if inpaint:
                st["known"] = torch.empty(M, 30, dtype=torch.float32, device=self.device)
                st["words"] = torch.empty(M, dtype=torch.int32, device=self.device)
            self._graphs[key] = st
        x, t_a, t_b = st["x"], st["t_a"], st["t_b"]
        kn = {}
        if inpaint:
            # K = M / rows blocks of the caller's rows (num_samples), like the conditions
            reps = M // known.shape[0]
            st["known"].view(reps, -1, 30).copy_(known.unsqueeze(0).expand(reps, -1, -1))
            st["words"].view(reps, -1).copy_(words.unsqueeze(0).expand(reps, -1))
            kn = dict(known=st["known"], known_mask=st["words"])
        # the halves of the guided buffer receive the same x_T (the same Philox seed and offset, or the same rows)
        for rows in ((xc,) if not guided else (xc2[:M], xc2[M:])):
            if x_T is None:
                # x_T ~ N(0, I): the q_sample kernel with tables (0, 1) writes pure Philox noise (fp32 + bf16 rows)
                zero = torch.zeros(B, F * 30, device=self.device)
                ops.q_sample(zero, None, torch.zeros(B, dtype=torch.int32, device=self.device), torch.zeros(1, device=self.device),
                             torch.ones(1, device=self.device), xt_f32=x.view(B, F * 30), xt_bf16=rows, bf16_ld=eng.ld_in,
                             seed=seed, offset=1 << 40)
            else:
                x.copy_(x_T.reshape(M, 30))
                ops.pack_inputs([x], M, F, out_bf16=rows, frame_stride=eng.ld_in, win_extra=0, col0=0)
        n_steps = len(ts)
        t_a.fill_(self.T - 1)

        def step(t_in, t_out, z):
            if not guided:
                x0_hat = eng.forward(B, F, False, t_scalar=t_in, t_count=self.T if self.use_temb_table else 0)
                ops.posterior_step(x0_hat, 32, x, z, t_in, coef_x0, coef_xt, sigma, M, x_prev=x, xprev_bf16=xc,
                                   bf16_ld=eng.ld_in, seed=seed, offset=0, t_next=t_out, t_succ=succ, **kn)
                return
            x0_hat = eng.forward(2 * B, F, False, t_scalar=t_in, t_count=self.T if self.use_temb_table else 0)
            ops.guided_step(x0_hat, 32, x, z, t_in, coef_x0, coef_xt, sigma, M, guidance_scale, x_prev=x, xprev_bf16=xc2,
                            bf16_ld=eng.ld_in, seed=seed, offset=0, t_next=t_out, t_succ=succ, **kn)

        # DDPM runs an odd step count eagerly, as it always has; DDIM replays the graph for the even part of any S >= 2
        if noise is not None or not use_graph or (n_steps % 2 if sched is None else n_steps < 2):
            cur, nxt = t_a, t_b
            for t in ts:
                step(cur, nxt, noise(t) if noise is not None else None)
                cur, nxt = nxt, cur
            return x.view(B, F, 30).clone()

        # two steps per CUDA graph: the timestep ping-pongs between two device words.  The captured launches read the
        # per-timestep time-MLP table through a baked-in pointer: the table is re-evaluated here whenever the weights changed
        # (optimizer step, load_state_dict) and a NEW table tensor (or a new seed) forces a re-capture; the entry keeps the
        # captured table alive.
        done = 0
        table = eng.temb_table(self.T) if self.use_temb_table else None
        tkey = (getattr(eng, "_temb_key", None), None if table is None else table.data_ptr())
        if st["graph"] is None or st["seed"] != seed or st["table_key"] != tkey:
            st["table"], st["table_key"] = table, tkey
            step(t_a, t_b, None)                  # eager warm-up (real steps): allocates buffers, sets func attributes
            step(t_b, t_a, None)
            done = 2
            torch.cuda.synchronize()
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g):
                step(t_a, t_b, None)
                step(t_b, t_a, None)
            st["graph"], st["seed"] = g, seed
            done += 2                             # capture does not execute, but keep step parity simple: replay below
            done -= 2
        for _ in range((n_steps - done) // 2):
            st["graph"].replay()
        if n_steps % 2:
            step(t_a, t_b, None)                  # the last step of an odd S: the ping-pong left its timestep in t_a
        return x.view(B, F, 30).clone()

    # ---- BASELINE configs[3]: a set of windows sharded over the ranks, no collective ------------------------------
    @torch.no_grad()
    def sample_windows(self, model, cond: torch.Tensor, *, batch: int = 512, steps: Optional[int] = None, seed: int = 0,
                       rank: Optional[int] = None, world: Optional[int] = None, ddim_steps: Optional[int] = None,
                       eta: float = 0.0, guidance_scale: float = 1.0, num_samples: Optional[int] = None,
                       known: Optional[torch.Tensor] = None, known_mask: Optional[torch.Tensor] = None):
        """Reverse-sample GRF / CoP / torque / wrench trajectories for ``cond``: (N, F, C_in) fp32 packed kinematics of N
        windows (model concat order, FeedForward...py:97-108) in HOST memory (pinned for asynchronous copies).

        Windows are independent: rank r takes the contiguous range ``parallel.contiguous_shard(N, r, W)`` and walks it in
        batches of ``batch`` windows — H2D copy of the batch's conditions, one packing kernel into the denoiser's concat buffer,
        ``steps`` (default: the full schedule) CUDA-graph-replayed denoise steps, D2H copy of the trajectories — and returns
        ``(range, x0)`` with x0 a pinned host tensor (len(range), F, 30).  No collective; per-rank noise stream = seed + rank.
        The copies of batch i+1 / i-1 overlap the sampling of batch i (separate streams).  ``ddim_steps`` / ``eta`` select
        DDIM sampling and ``guidance_scale`` classifier-free guidance as in ``sample``.  ``num_samples`` K: K draws per window
        (``sample(..., num_samples=K)`` per batch, ``batch`` still counts windows) and x0 is (len(range), K, F, 30).
        ``known`` (fp32 (N, F, 30)) with ``known_mask`` (bool (N, F, 30) or (30,)), host tensors: inpainting as in ``sample``;
        the mask is packed into row words once, and each batch's values and words travel with its conditions."""
        from . import parallel
        _check_schedule(self.T, steps, ddim_steps, eta)
        check_guidance_scale(guidance_scale)
        check_num_samples(num_samples)
        inpaint = check_known(known, known_mask, cond.shape[0], None, self.T, steps)
        r, w = parallel.world()
        rank = r if rank is None else rank
        world = w if world is None else world
        eng = model.engine()
        F, C = eng.F, eng.c_in
        N = cond.shape[0]
        assert tuple(cond.shape[1:]) == (F, C) and not cond.is_cuda, "cond: host tensor (N, F, C_in)"
        if inpaint:
            check_known(known, known_mask, N, F, self.T, steps)
            if known.is_cuda or known_mask.is_cuda:
                raise ValueError("sample_windows takes known and known_mask in host memory")
            known = known.reshape(N * F, 30)
            words = known_mask_words(known_mask, N * F).contiguous().pin_memory()
        mine = parallel.contiguous_shard(N, rank, world)
        shape = (len(mine), F, 30) if num_samples is None else (len(mine), num_samples, F, 30)
        out = torch.empty(shape, dtype=torch.float32).pin_memory()
        dev = self.device
        main = torch.cuda.current_stream(dev)
        up, down = torch.cuda.Stream(dev), torch.cuda.Stream(dev)
        stage = [torch.empty(batch * F, C, dtype=torch.float32, device=dev) for _ in range(2)]
        if inpaint:
            stage_y = [torch.empty(batch * F, 30, dtype=torch.float32, device=dev) for _ in range(2)]
            stage_w = [torch.empty(batch * F, dtype=torch.int32, device=dev) for _ in range(2)]
        uploaded = [torch.cuda.Event() for _ in range(2)]
        packed = [torch.cuda.Event() for _ in range(2)]
        starts = list(range(mine.start, mine.stop, batch))

        def upload(i):
            a, b = starts[i], min(starts[i] + batch, mine.stop)
            with torch.cuda.stream(up):
                up.wait_event(packed[i & 1])
                stage[i & 1][:(b - a) * F].copy_(cond[a:b].reshape(-1, C), non_blocking=True)
                if inpaint:
                    up.wait_event(sampled[i & 1])             # batch i - 2 has read its known values and words
                    stage_y[i & 1][:(b - a) * F].copy_(known[a * F:b * F], non_blocking=True)
                    stage_w[i & 1][:(b - a) * F].copy_(words[a * F:b * F], non_blocking=True)
                uploaded[i & 1].record(up)

        sampled = [torch.cuda.Event() for _ in range(2)]
        for e in packed + sampled:
            e.record(main)
        if starts:
            upload(0)
        pending = []
        for i, a in enumerate(starts):
            b = min(a + batch, mine.stop)
            nb = b - a
            main.wait_event(uploaded[i & 1])
            buf, fs, we, col0 = eng.input_layout(nb, F, False)
            ops.pack_inputs([stage[i & 1][:nb * F]], nb * F, F, out_bf16=buf, frame_stride=fs, win_extra=we, col0=col0)
            packed[i & 1].record(main)
            if i + 1 < len(starts):
                upload(i + 1)
            kn = dict(known=stage_y[i & 1][:nb * F], words=stage_w[i & 1][:nb * F]) if inpaint else dict(known=None, words=None)
            x0 = self._sample(model, nb, x_T=None, noise=None, steps=steps, seed=seed + rank + 7919 * i, use_graph=True,
                              ddim_steps=ddim_steps, eta=eta, guidance_scale=guidance_scale, num_samples=num_samples, **kn)
            if inpaint:
                sampled[i & 1].record(main)
            if num_samples is not None:
                x0 = x0.transpose(0, 1)                       # (nb, K, F, 30): window-major for the caller
            ready = torch.cuda.Event()
            ready.record(main)
            with torch.cuda.stream(down):
                down.wait_event(ready)
                out[a - mine.start:b - mine.start].copy_(x0, non_blocking=True)
            pending.append(x0)                                # keeps the device tensor alive until the copy has run
        down.synchronize()
        return mine, out
