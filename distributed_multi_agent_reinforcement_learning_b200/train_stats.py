"""PPO diagnostics of one training update: `MAPPO.train(..., stats=True)` leaves a `TrainStats` in `mappo.last_train_stats`.

The device reduces the per-row values of the training forward (csrc/train_stats.cu, `policy_ops.ppo_stats` per minibatch and
`ppo_stats_combine` per update) into one f64 vector of raw sums and counts (slots: include/marl_b200.h, MARL_PPO_STATS_OUT).
`TrainStats.from_sums` derives the reported values from it on the host; `allreduce_()` sums the vectors of all ranks first, so
every rank derives the same global statistics.
"""
import math

import torch

# slots of the combined vector (MARL_PPO_STATS_SUMS / MARL_PPO_STATS_OUT in include/marl_b200.h)
N_ACTIVE, ENT, KL_K1, KL_K3, CLIP, MAX_LR, MIN_LR, VCLIP, VT, VT2, RES, RES2, ADV, ADV2, HAS_V_OLD, ROWS = range(16)
MINIBATCHES, N_NORMS, NORM_MAX, NORM_LAST, CLIPPED = range(16, 21)
OUT_SLOTS = 24
_MAX_SLOTS = (MAX_LR, NORM_MAX, NORM_LAST)      # reduced over ranks with max (NORM_LAST: the largest rank's last norm)
_MIN_SLOTS = (MIN_LR,)


def _div(a, b):
    return a / b if b else math.nan


def _var(s1, s2, n):
    """Population variance from the f64 moments sum x and sum x^2 of n samples (NaN for n = 0)."""
    if not n:
        return math.nan
    m = s1 / n
    return s2 / n - m * m


def _ev(var_res, var_vt):
    """1 - Var(residual) / Var(v_target); NaN when Var(v_target) is 0 (or NaN)."""
    return 1.0 - var_res / var_vt if var_vt > 0 else math.nan


class TrainStats:
    """Statistics of one update over its active rows.  `sums` is the f64 vector [24] (on the device when it comes from `train`);
    the other attributes are host floats derived from it:

      entropy, approx_kl (the k3 estimate mean((r - 1) - log r)), approx_kl_k1 (mean(-log r)), clip_frac (share of rows with
      |r - 1| > eps), ratio_min, ratio_max; value_clip_frac (share with |value - v_old| > eps; None without a value clip);
      explained_variance (1 - Var(v_target - value) / Var(v_target), value of the training forward), rollout_explained_variance (the
      same with the rollout's v_old), adv_mean and adv_std (the raw advantage v_target - v_old; these three None without v_old);
      return_mean (mean v_target); grad_norm_max, grad_norm_last (pre-clip norms of the running accumulation) and
      clipped_minibatches (norms above max_norm), None without a gradient clip; rows (active rows), minibatches.

    Variances are population variances.  With no active row, or a constant v_target, the affected values are NaN."""

    FIELDS = ("entropy", "approx_kl", "approx_kl_k1", "clip_frac", "ratio_min", "ratio_max", "value_clip_frac", "explained_variance",
              "rollout_explained_variance", "adv_mean", "adv_std", "return_mean", "grad_norm_max", "grad_norm_last",
              "clipped_minibatches", "rows", "minibatches")

    def __init__(self, sums, eps, max_norm):
        self.sums, self.eps, self.max_norm = sums, eps, max_norm
        self._derive()

    @classmethod
    def from_sums(cls, sums, eps, max_norm):
        """sums: the combined vector (a tensor on any device, or a sequence of 24 numbers); eps: the PPO clip range the kernel
        thresholded with; max_norm: the gradient clip's max norm, or None without a gradient clip."""
        if not torch.is_tensor(sums):
            sums = torch.as_tensor(sums, dtype=torch.float64)
        if sums.dtype != torch.float64 or sums.numel() != OUT_SLOTS:
            raise ValueError(f"TrainStats: sums must be {OUT_SLOTS} float64 values, got {sums.numel()} {sums.dtype}")
        return cls(sums, eps, max_norm)

    def _derive(self):
        s = [float(x) for x in self.sums.detach().cpu().reshape(-1)]
        n = s[N_ACTIVE]
        self.rows, self.minibatches = int(n), int(s[MINIBATCHES])
        self.entropy = _div(s[ENT], n)
        self.approx_kl_k1 = _div(s[KL_K1], n)
        self.approx_kl = _div(s[KL_K3], n)
        self.clip_frac = _div(s[CLIP], n)
        self.ratio_max = math.exp(s[MAX_LR]) if n else math.nan
        self.ratio_min = math.exp(s[MIN_LR]) if n else math.nan
        var_vt = _var(s[VT], s[VT2], n)
        self.return_mean = _div(s[VT], n)
        self.explained_variance = _ev(_var(s[RES], s[RES2], n), var_vt)
        if s[HAS_V_OLD] > 0:
            var_x = _var(s[ADV], s[ADV2], n)
            self.value_clip_frac = _div(s[VCLIP], n)
            self.rollout_explained_variance = _ev(var_x, var_vt)
            self.adv_mean = _div(s[ADV], n)
            self.adv_std = math.sqrt(max(var_x, 0.0)) if n else math.nan
        else:
            self.value_clip_frac = self.rollout_explained_variance = self.adv_mean = self.adv_std = None
        if self.max_norm is not None and s[N_NORMS] > 0:
            self.grad_norm_max, self.grad_norm_last, self.clipped_minibatches = s[NORM_MAX], s[NORM_LAST], int(s[CLIPPED])
        else:
            self.grad_norm_max = self.grad_norm_last = self.clipped_minibatches = None

    def allreduce_(self):
        """Reduces `sums` over the ranks of the default process group in place (sum; max for the largest log-ratio and the gradient
        norms, min for the smallest log-ratio) and derives the values again: afterwards every rank holds the same statistics.  A no-op
        on one rank.  Counts (rows, minibatches, clipped_minibatches) then cover all ranks."""
        from . import parallel
        _, world = parallel.world()
        if world > 1:
            v = self.sums.clone()
            ext = torch.stack([v[j] for j in _MAX_SLOTS] + [-v[j] for j in _MIN_SLOTS])
            v[list(_MAX_SLOTS + _MIN_SLOTS)] = 0.0
            parallel.allreduce_sum_(v)
            parallel.allreduce_max_(ext)
            for i, j in enumerate(_MAX_SLOTS):
                v[j] = ext[i]
            for i, j in enumerate(_MIN_SLOTS):
                v[j] = -ext[len(_MAX_SLOTS) + i]
            self.sums = v
            self._derive()
        return self

    def as_dict(self):
        return {k: getattr(self, k) for k in self.FIELDS}
