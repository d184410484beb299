"""CPU checks of the PPO diagnostics: the three entry points of csrc/train_stats.cu are declared and exported, they refuse bad arguments
with MARL_EINVAL and a message before any CUDA call, `TrainStats.from_sums` derives the values worked out by hand here (no active row, a
constant v_target, no value clip, no gradient clip), and `train_loop.py` refuses --target-kl with one epoch."""
import ctypes
import math
import os
import re
import subprocess
import sys

import pytest

torch = pytest.importorskip("torch")

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
NEW = ("marl_ppo_stats_workspace_bytes", "marl_ppo_stats", "marl_ppo_stats_combine")


def test_entry_points_declared_and_exported():
    from distributed_multi_agent_reinforcement_learning_b200 import _lib
    src = open(os.path.join(ROOT, "include", "marl_b200.h")).read()
    assert re.search(r"#define MARL_PPO_STATS_SUMS 16\b", src) and re.search(r"#define MARL_PPO_STATS_OUT 24\b", src)
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    handle = ctypes.CDLL(_lib.LIB_PATH)
    for name in NEW:
        assert re.search(rf"\b{name}\s*\(", src), name
        assert hasattr(handle, name) and name in _lib.exported_symbols(), name
    L = _lib.lib()
    assert L.marl_version() == 1
    assert L.marl_ppo_stats_workspace_bytes(0) == -1 and L.marl_ppo_stats_workspace_bytes(-5) == -1
    assert L.marl_ppo_stats_workspace_bytes(1) == 16 * 8
    assert L.marl_ppo_stats_workspace_bytes(1 << 30) == 1024 * 16 * 8      # the grid is capped by a constant, not by the SM count


def _err(L):
    return L.marl_last_error_string().decode()


def test_bad_arguments_fail_loudly_without_a_gpu():
    """Every refusal happens before any CUDA call (no device here): fake, never dereferenced addresses stand in for buffers."""
    from distributed_multi_agent_reinforcement_learning_b200 import _lib
    L = _lib.lib()
    p = [0x1000 * (i + 1) for i in range(10)]       # logp, old, ent, value, v_old, v_target, active, sums, workspace
    good = dict(R=8, ptrs=[p[0], p[1], p[2], p[3], p[4], p[5], p[6]], eps=0.2, sums=p[7], ws=p[8])

    def call(R=None, ptrs=None, eps=None, sums=None, ws=None):
        a = dict(good, **{k: v for k, v in dict(R=R, ptrs=ptrs, eps=eps, sums=sums, ws=ws).items() if v is not None})
        return L.marl_ppo_stats(a["R"], *a["ptrs"], ctypes.c_float(a["eps"]), a["sums"], a["ws"], None)

    for R in (0, -1):
        assert call(R=R) == -1 and "R=" in _err(L)
    for i in (0, 1, 2, 3, 5, 6):                     # every input but v_old is required
        ptrs = list(good["ptrs"])
        ptrs[i] = None
        assert call(ptrs=ptrs) == -1 and "null pointer" in _err(L)
    assert L.marl_ppo_stats(8, *good["ptrs"], ctypes.c_float(0.2), None, p[8], None) == -1 and "null pointer" in _err(L)
    assert L.marl_ppo_stats(8, *good["ptrs"], ctypes.c_float(0.2), p[7], None, None) == -1 and "null pointer" in _err(L)
    for eps in (-0.1, math.inf, math.nan):
        assert call(eps=eps) == -1 and "eps=" in _err(L)
    with pytest.raises(_lib.MarlError, match="marl_ppo_stats"):
        _lib.check(call(R=0), "marl_ppo_stats")

    C = L.marl_ppo_stats_combine
    for n in (0, -3):
        assert C(n, p[0], p[1], ctypes.c_float(5.0), p[2], None) == -1 and "n_mb=" in _err(L)
    assert C(2, None, p[1], ctypes.c_float(5.0), p[2], None) == -1 and "null pointer" in _err(L)
    assert C(2, p[0], p[1], ctypes.c_float(5.0), None, None) == -1 and "null pointer" in _err(L)
    for mx in (0.0, -1.0, math.inf, math.nan):       # a max norm is needed only with the norms
        assert C(2, p[0], p[1], ctypes.c_float(mx), p[2], None) == -1 and "max_norm=" in _err(L)


def _sums(**kw):
    from distributed_multi_agent_reinforcement_learning_b200 import train_stats as ts
    s = [0.0] * 24
    s[ts.MAX_LR], s[ts.MIN_LR] = -math.inf, math.inf
    for k, v in kw.items():
        s[getattr(ts, k)] = v
    return s


def test_from_sums_matches_hand_worked_values():
    """Four active rows: ratio r in {1, e^0.1, e^-0.2, 1}, entropy {1, 2, 3, 2}, v_target {1, 2, 3, 4}, value {1, 1, 3, 3},
    v_old {0, 2, 2, 4}; eps 0.15 (one row clipped: |e^-0.2 - 1| > 0.15), all four rows with |value - v_old| > 0.15."""
    from distributed_multi_agent_reinforcement_learning_b200.train_stats import TrainStats
    lr = [0.0, 0.1, -0.2, 0.0]
    vt, val, vo = [1.0, 2.0, 3.0, 4.0], [1.0, 1.0, 3.0, 3.0], [0.0, 2.0, 2.0, 4.0]
    res = [a - b for a, b in zip(vt, val)]            # 0 1 0 1
    x = [a - b for a, b in zip(vt, vo)]               # 1 0 1 0
    s = _sums(N_ACTIVE=4, ENT=8.0, KL_K1=-sum(lr), KL_K3=sum(math.exp(v) - 1 - v for v in lr), CLIP=1, MAX_LR=0.1, MIN_LR=-0.2,
              VCLIP=4, VT=10.0, VT2=30.0, RES=2.0, RES2=2.0, ADV=2.0, ADV2=2.0, HAS_V_OLD=1, ROWS=6, MINIBATCHES=2, N_NORMS=2,
              NORM_MAX=7.5, NORM_LAST=4.0, CLIPPED=1)
    st = TrainStats.from_sums(s, 0.15, 5.0)
    assert st.rows == 4 and st.minibatches == 2
    assert st.entropy == 2.0
    assert st.approx_kl_k1 == pytest.approx(0.1 / 4, rel=1e-15)
    assert st.approx_kl == pytest.approx(sum(math.exp(v) - 1 - v for v in lr) / 4, rel=1e-15)
    assert st.clip_frac == 0.25 and st.value_clip_frac == 1.0
    assert st.ratio_max == math.exp(0.1) and st.ratio_min == math.exp(-0.2)
    # Var(v_target) = 7.5 - 6.25 = 1.25; Var(res) = 0.5 - 0.25 = 0.25; Var(x) = 0.25
    assert st.explained_variance == pytest.approx(1 - 0.25 / 1.25, rel=1e-15)
    assert st.rollout_explained_variance == pytest.approx(1 - 0.25 / 1.25, rel=1e-15)
    assert st.adv_mean == 0.5 and st.adv_std == 0.5 and st.return_mean == 2.5
    assert (st.grad_norm_max, st.grad_norm_last, st.clipped_minibatches) == (7.5, 4.0, 1)
    assert sum(res) == 2.0 and sum(x) == 2.0
    d = st.as_dict()
    assert list(d) == list(TrainStats.FIELDS) and d["entropy"] == 2.0
    sums64 = torch.tensor(s, dtype=torch.float64)
    assert TrainStats.from_sums(sums64, 0.15, 5.0).as_dict() == d
    assert st.allreduce_() is st and st.as_dict() == d                  # one rank: nothing to reduce


def test_from_sums_without_value_clip_or_gradient_clip():
    from distributed_multi_agent_reinforcement_learning_b200.train_stats import TrainStats
    s = _sums(N_ACTIVE=2, ENT=1.0, VT=2.0, VT2=2.0, RES=0.0, RES2=0.0, MAX_LR=0.0, MIN_LR=0.0, ROWS=2, MINIBATCHES=1)
    st = TrainStats.from_sums(s, 0.2, None)
    assert st.value_clip_frac is None and st.rollout_explained_variance is None and st.adv_mean is None and st.adv_std is None
    assert st.grad_norm_max is None and st.grad_norm_last is None and st.clipped_minibatches is None
    assert st.ratio_max == 1.0 and st.ratio_min == 1.0 and st.entropy == 0.5
    assert math.isnan(st.explained_variance)        # v_target is constant (1, 1): Var(v_target) = 0 -> NaN, not an exception
    assert st.return_mean == 1.0
    # a max norm but no norms recorded (the combine got NULL): still None
    assert TrainStats.from_sums(s, 0.2, 5.0).grad_norm_max is None


def test_from_sums_with_no_active_row():
    from distributed_multi_agent_reinforcement_learning_b200.train_stats import TrainStats
    st = TrainStats.from_sums(_sums(HAS_V_OLD=1, ROWS=5, MINIBATCHES=1, N_NORMS=1, NORM_MAX=2.0, NORM_LAST=2.0), 0.2, 5.0)
    assert st.rows == 0
    for k in ("entropy", "approx_kl", "approx_kl_k1", "clip_frac", "ratio_min", "ratio_max", "value_clip_frac", "explained_variance",
              "rollout_explained_variance", "adv_mean", "adv_std", "return_mean"):
        assert math.isnan(getattr(st, k)), k
    assert (st.grad_norm_max, st.clipped_minibatches) == (2.0, 0)


def test_from_sums_refuses_a_wrong_vector():
    from distributed_multi_agent_reinforcement_learning_b200.train_stats import TrainStats
    with pytest.raises(ValueError, match="24 float64"):
        TrainStats.from_sums([0.0] * 16, 0.2, 5.0)
    with pytest.raises(ValueError, match="24 float64"):
        TrainStats.from_sums(torch.zeros(24, dtype=torch.float32), 0.2, 5.0)


def _arg_error(*args):
    cmd = [sys.executable] + (["-s"] if sys.flags.no_user_site else []) + [os.path.join(ROOT, "tools", "train_loop.py")] + list(args)
    r = subprocess.run(cmd, cwd=ROOT, timeout=300, capture_output=True, text=True)
    assert r.returncode == 2, (r.returncode, r.stdout, r.stderr)           # argparse's error exit, before any CUDA call
    return r.stderr


def test_train_loop_refuses_target_kl_with_one_epoch():
    assert "--target-kl needs at least 2 epochs" in _arg_error("--target-kl", "0.01")                 # algo.epochs is 1
    assert "--target-kl needs at least 2 epochs" in _arg_error("--target-kl", "0.01", "--epochs", "1")
    assert "--target-kl must be a finite number" in _arg_error("--target-kl", "-1", "--epochs", "2")
    assert "--target-kl must be a finite number" in _arg_error("--target-kl", "nan", "--epochs", "2")
    assert "--epochs must be >= 1" in _arg_error("--epochs", "0")
