"""DDPM schedule, noising and reverse sampling on libibm_b200 (builder-owned spec, DESIGN.md D-1;
the reference has no diffusion code).

  betas = linspace(1e-4, 2e-2, 1000) (fp64 → fp32 tables)          q_sample: fused kernel, optional
  x_t   = sqrt(abar_t) x0 + sqrt(1-abar_t) eps                      on-device Philox noise
  x_{t-1} = c1_t x0_hat + c2_t x_t + [t>0] sigma_t z                posterior step: fused kernel

The reverse loop runs the denoiser forward + one fused posterior kernel per step; the timestep lives
in device memory so two consecutive steps are captured once in a CUDA graph and replayed (sampling at
512 windows/GPU is launch-bound otherwise).  Windows are independent: multi-GPU sampling shards them
with no collective.
"""
from __future__ import annotations

from typing import Callable, Optional

import numpy as np
import torch

from . import ops


class GaussianDiffusion:
    def __init__(self, num_timesteps: int = 1000, beta_start: float = 1e-4, beta_end: float = 2e-2, device="cuda"):
        self.T = num_timesteps
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

    # ---- reverse process -----------------------------------------------------------------------
    @torch.no_grad()
    def sample(self, model, B: int, *, x_T: Optional[torch.Tensor] = None, noise: Optional[Callable[[int], torch.Tensor]] = None,
               steps: Optional[int] = None, seed: int = 0, use_graph: bool = True) -> torch.Tensor:
        """Reverse-sample x_0 (B,F,30) for the kinematics already packed in model.engine().xc(B, False)
        (columns 30…).  ``noise(t)`` supplies z per step for parity tests; None ⇒ on-device Philox."""
        eng = model.engine()
        F, M = eng.F, B * eng.F
        xc = eng.xc(B, False)
        key = (id(model), B)
        st = self._graphs.get(key)
        if st is None or st["model"] is not model:
            # the entry holds the model (its id() cannot be recycled while cached) and, below, the time-MLP table the
            # captured launches read
            st = dict(x=torch.empty(M, 30, dtype=torch.float32, device=self.device),
                      t_a=torch.zeros(1, dtype=torch.int32, device=self.device),
                      t_b=torch.zeros(1, dtype=torch.int32, device=self.device), graph=None, seed=None, model=model, table=None,
                      table_key=None)
            self._graphs[key] = st
        x, t_a, t_b = st["x"], st["t_a"], st["t_b"]
        if x_T is None:
            # x_T ~ N(0, I): the q_sample kernel with tables (0, 1) writes pure Philox noise (fp32 + bf16 rows)
            zero = torch.zeros(B, F * 30, device=self.device)
            ops.q_sample(zero, None, torch.zeros(B, dtype=torch.int32, device=self.device), torch.zeros(1, device=self.device),
                         torch.ones(1, device=self.device), xt_f32=x.view(B, F * 30), xt_bf16=xc, bf16_ld=eng.ld_in, seed=seed,
                         offset=1 << 40)
        else:
            x.copy_(x_T.reshape(M, 30))
            ops.pack_inputs([x], M, F, out_bf16=xc, frame_stride=eng.ld_in, win_extra=0, col0=0)
        n_steps = self.T if steps is None else steps
        t_a.fill_(self.T - 1)

        def step(t_in, t_out, z):
            x0_hat = eng.forward(B, F, False, t_scalar=t_in, t_count=self.T if self.use_temb_table else 0)
            ops.posterior_step(x0_hat, 32, x, z, t_in, self.coef_x0, self.coef_xt, self.sigma, M, x_prev=x, xprev_bf16=xc,
                               bf16_ld=eng.ld_in, seed=seed, offset=0, t_next=t_out)

        if noise is not None or not use_graph or n_steps % 2:
            cur, nxt = t_a, t_b
            for i in range(n_steps):
                step(cur, nxt, noise(self.T - 1 - i) if noise is not None else None)
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
        return x.view(B, F, 30).clone()

    # ---- BASELINE configs[3]: a set of windows sharded over the ranks, no collective ------------------------------
    @torch.no_grad()
    def sample_windows(self, model, cond: torch.Tensor, *, batch: int = 512, steps: Optional[int] = None, seed: int = 0,
                       rank: Optional[int] = None, world: Optional[int] = None):
        """Reverse-sample GRF / CoP / torque / wrench trajectories for ``cond``: (N, F, C_in) fp32 packed kinematics of N
        windows (model concat order, FeedForward...py:97-108) in HOST memory (pinned for asynchronous copies).

        Windows are independent: rank r takes the contiguous range ``parallel.contiguous_shard(N, r, W)`` and walks it in
        batches of ``batch`` windows — H2D copy of the batch's conditions, one packing kernel into the denoiser's concat buffer,
        ``steps`` (default: the full schedule) CUDA-graph-replayed denoise steps, D2H copy of the trajectories — and returns
        ``(range, x0)`` with x0 a pinned host tensor (len(range), F, 30).  No collective; per-rank noise stream = seed + rank.
        The copies of batch i+1 / i-1 overlap the sampling of batch i (separate streams)."""
        from . import parallel
        r, w = parallel.world()
        rank = r if rank is None else rank
        world = w if world is None else world
        eng = model.engine()
        F, C = eng.F, eng.c_in
        N = cond.shape[0]
        assert tuple(cond.shape[1:]) == (F, C) and not cond.is_cuda, "cond: host tensor (N, F, C_in)"
        mine = parallel.contiguous_shard(N, rank, world)
        out = torch.empty(len(mine), F, 30, dtype=torch.float32).pin_memory()
        dev = self.device
        main = torch.cuda.current_stream(dev)
        up, down = torch.cuda.Stream(dev), torch.cuda.Stream(dev)
        stage = [torch.empty(batch * F, C, dtype=torch.float32, device=dev) for _ in range(2)]
        uploaded = [torch.cuda.Event() for _ in range(2)]
        packed = [torch.cuda.Event() for _ in range(2)]
        starts = list(range(mine.start, mine.stop, batch))

        def upload(i):
            a, b = starts[i], min(starts[i] + batch, mine.stop)
            with torch.cuda.stream(up):
                up.wait_event(packed[i & 1])
                stage[i & 1][:(b - a) * F].copy_(cond[a:b].reshape(-1, C), non_blocking=True)
                uploaded[i & 1].record(up)

        for e in packed:
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
            x0 = self.sample(model, nb, steps=steps, seed=seed + rank + 7919 * i)
            ready = torch.cuda.Event()
            ready.record(main)
            with torch.cuda.stream(down):
                down.wait_event(ready)
                out[a - mine.start:b - mine.start].copy_(x0, non_blocking=True)
            pending.append(x0)                                # keeps the device tensor alive until the copy has run
        down.synchronize()
        return mine, out
