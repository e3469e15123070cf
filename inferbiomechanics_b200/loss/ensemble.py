"""Probabilistic scores of an ensemble of K sampled trajectories per window (DESIGN.md §3), next to the reference report.

The denoiser returns a distribution of ground-reaction forces, not a point; one draw per window mixes the model's bias with
its sampling spread (for a calibrated model one draw's expected squared error is 2 sigma^2, the K-draw mean's sigma^2 (1 + 1/K)).
``EnsembleScorer`` accumulates, per output channel and on the device, the sums ``ops.ensemble_score`` produces for each batch
of K draws per window, and reports per channel and per quantity:

* the fair CRPS (Ferro 2014), (1/K) sum_k |x_k - y| - 1/(2K(K-1)) sum_{i,j} |x_i - x_j|, unbiased at every K;
* the ensemble-mean RMSE (the "skill") and the spread sqrt(mean s^2);
* the spread-skill ratio sqrt((K+1)/K * sum s^2 / sum (m - y)^2), 1 for a calibrated ensemble (Fortin et al. 2014);
* the mean pairwise distance between draws of one window, a per-component analogue of MDM's MultiModality;
* the element counts (CoP channels count contact rows only, like the fused loss).

All values are in the evaluator's units (N / kg, m, Nm / kg, N+Nm / kg).
"""
from __future__ import annotations

from typing import Dict, Optional

import numpy as np
import torch

from .. import ops
from .RegressionLossEvaluator import COP_FORCE_THRESHOLD

# quantity -> (channel range in a rows30 row, unit), in report order
ENSEMBLE_GROUPS = {"force": ((6, 12), "N / kg"), "cop": ((0, 6), "m"), "moment": ((12, 18), "Nm / kg"),
                   "wrench": ((18, 30), "N+Nm / kg")}
METRICS = ("crps", "rmse", "spread", "spread_skill", "pair_dist", "count")


def ensemble_metrics(sums: np.ndarray, K: int) -> Dict[str, float]:
    """The report metrics of pooled sums {crps, s^2, (m - y)^2, pair, count} (fp64 [5] in ops.ENSEMBLE_QUANTITIES order)."""
    crps, var, se, pair, n = (float(v) for v in sums)
    if n == 0:
        return dict(crps=float("nan"), rmse=float("nan"), spread=float("nan"), spread_skill=float("nan"),
                    pair_dist=float("nan"), count=0)
    ssr = float(np.sqrt((K + 1) / K * var / se)) if se > 0 else float("nan")
    return dict(crps=crps / n, rmse=float(np.sqrt(se / n)), spread=float(np.sqrt(var / n)), spread_skill=ssr,
                pair_dist=pair / n, count=int(n))


class EnsembleScorer:
    """Device-resident fp64 [5, 30] accumulator of ``ops.ensemble_score`` over the batches of one pass, with K draws per
    window.  ``score`` per batch, ``merge`` once at the end (every rank), then ``summary`` / ``print_report``."""

    def __init__(self, num_samples: int, split: str = "dev", device="cuda"):
        if not 2 <= num_samples <= ops.ENSEMBLE_MAX_DRAWS:
            raise ValueError(f"EnsembleScorer needs 2 <= num_samples <= {ops.ENSEMBLE_MAX_DRAWS}, got {num_samples}")
        self.K, self.split = num_samples, split
        self.acc = torch.zeros(len(ops.ENSEMBLE_QUANTITIES), 30, dtype=torch.float64, device=device)
        self.ws = ops.EnsembleWorkspace(device)

    def score(self, draws: torch.Tensor, labels: torch.Tensor) -> torch.Tensor:
        """draws (K, B, F, 30) fp32 as ``GaussianDiffusion.sample(..., num_samples=K)`` returns them, labels (B, Fo, 30): adds
        the batch to the accumulator and returns the ensemble mean (B, Fo, 30) for the regression evaluator."""
        if draws.shape[0] != self.K:
            raise ValueError(f"this scorer takes {self.K} draws per window, got {draws.shape[0]}")
        mean = torch.empty(labels.shape, dtype=torch.float32, device=labels.device)
        return ops.ensemble_score(draws, labels, self.acc, mean, self.ws, threshold=COP_FORCE_THRESHOLD)

    def merge(self, world: int) -> None:
        """Sums the accumulators of ``world`` data-parallel ranks (a collective: every rank calls it).  The per-rank tensors
        are gathered and added on the host in rank order, so the result does not depend on a collective's reduction order."""
        if world <= 1:
            return
        import torch.distributed as dist
        gathered = [torch.zeros_like(self.acc) for _ in range(world)]
        dist.all_gather(gathered, self.acc)
        total = np.zeros(tuple(self.acc.shape), dtype=np.float64)
        for g in gathered:
            total += g.cpu().numpy()
        self.acc.copy_(torch.from_numpy(total))

    def summary(self) -> Dict[str, Dict[str, object]]:
        """{"channels": {metric: [30 values]}, <quantity>: {metric: value}} for the quantities of ENSEMBLE_GROUPS; one D2H copy."""
        acc = self.acc.cpu().numpy()
        per = [ensemble_metrics(acc[:, c], self.K) for c in range(30)]
        out: Dict[str, Dict[str, object]] = {"channels": {m: [p[m] for p in per] for m in METRICS}}
        for q, ((a, b), _) in ENSEMBLE_GROUPS.items():
            out[q] = ensemble_metrics(acc[:, a:b].sum(axis=1), self.K)
        return out

    def print_report(self, args=None, log_to_wandb: bool = False, summary: Optional[Dict] = None, given=()) -> None:
        """``given``: quantities the sampler was given as known values (inpainting), marked "(given)"."""
        s = self.summary() if summary is None else summary
        print(f'\tEnsemble of {self.K} samples (fair CRPS, ensemble-mean RMSE, spread, spread-skill ratio, mean pairwise distance):')
        for q, (_, unit) in ENSEMBLE_GROUPS.items():
            v = s[q]
            print(f'\t{q}{" (given)" if q in given else ""}: CRPS {v["crps"]} | RMSE {v["rmse"]} | spread {v["spread"]} | spread/skill {v["spread_skill"]} | '
                  f'pair dist {v["pair_dist"]} {unit} | {v["count"]} elements')
        if log_to_wandb:
            import wandb
            wandb.log({f'{self.split}/ensemble/{q}_{m}': s[q][m] for q in ENSEMBLE_GROUPS for m in METRICS})
