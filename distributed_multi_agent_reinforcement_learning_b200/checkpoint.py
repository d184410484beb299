"""Checkpoint file set of the reference driver (main.py:146-172): eight pickled modules

    actor.pth critic.pth actor_gnn.pth critic_gnn.pth actor_gru.pth critic_gru.pth actor_mean.pth critic_mean.pth

(+ the same names with `_final` at the end of training) and `recorder.npy` (rows of
(total_step, avgR, stdR, expR, objC, objA), evaluator.py).  The modules here carry the reference's sub-module names and
state_dict keys, so `torch.load(f).state_dict()` of either side's file loads into the other side's class
(evaluator.py:329-330 relies on exactly that).  Additionally every file gets a `*.state_dict.pth` twin that loads with
`weights_only=True` (no pickled classes, no omegaconf).

`save_training_state` / `load_training_state` write and read one more file: everything a run needs to continue exactly where
it stopped (optimizer moments, schedule position, reward statistics, engine tables, evaluator bookkeeping, RNG streams)."""
import collections
import os
import random

import numpy as np
import torch

from ._lib import MarlError

TRAINING_STATE_VERSION = 1

FILES = ("actor", "critic", "actor_gnn", "critic_gnn", "actor_gru", "critic_gru", "actor_mean", "critic_mean")


def _parts(mappo):
    a, c = mappo.actor, mappo.critic
    return dict(actor=a, critic=c, actor_gnn=a.shared_net, critic_gnn=c.shared_net, actor_gru=a.GRU, critic_gru=c.GRU,
                actor_mean=a.Mean, critic_mean=c.Mean)


def _detached_copy(module):
    """A CPU deep copy whose parameters own their storage (the live ones are views into the flat optimizer arena)."""
    import copy
    m = copy.deepcopy(module).cpu()
    for p in m.parameters():
        p.data = p.data.clone()
        p.grad = None
    return m


def save_checkpoint(mappo, cwd, final=False, recorder=None):
    os.makedirs(cwd, exist_ok=True)
    suffix = "_final" if final else ""
    for name, mod in _parts(mappo).items():
        m = _detached_copy(mod)
        torch.save(m, os.path.join(cwd, f"{name}{suffix}.pth"))
        torch.save(m.state_dict(), os.path.join(cwd, f"{name}{suffix}.state_dict.pth"))
    if recorder is not None:
        np.save(os.path.join(cwd, "recorder.npy"), np.asarray(recorder))


def load_state(path):
    """state_dict from either a pickled module (reference or ours) or a state_dict file."""
    try:
        obj = torch.load(path, map_location="cpu", weights_only=True)
    except Exception:
        obj = torch.load(path, map_location="cpu", weights_only=False)
    return obj.state_dict() if hasattr(obj, "state_dict") else obj


def load_checkpoint(mappo, cwd, final=False, strict=True):
    """Loads whichever of the eight files exist (whole-network files first, then the per-part files override)."""
    suffix = "_final" if final else ""
    parts = _parts(mappo)
    loaded = []
    for name in FILES:
        for ext in (".state_dict.pth", ".pth"):
            path = os.path.join(cwd, f"{name}{suffix}{ext}")
            if os.path.exists(path):
                parts[name].load_state_dict(load_state(path), strict=strict)
                loaded.append(name)
                break
    return loaded


# ---------------------------------------------------------------------------------------------------------- training state
def _cpu_state(module):
    """module.state_dict() on the CPU, keeping the version metadata: without it spectral_norm's load hook would recompute
    weight_v instead of restoring it."""
    sd = module.state_dict()
    out = collections.OrderedDict((k, v.detach().cpu().clone()) for k, v in sd.items())
    out._metadata = getattr(sd, "_metadata", None)
    return out


def _world():
    if torch.distributed.is_available() and torch.distributed.is_initialized():
        return torch.distributed.get_rank(), torch.distributed.get_world_size()
    return 0, 1


def _fingerprint(mappo, engine):
    rank, world = _world()
    return dict(N=int(mappo.cfg.env.num_defender), E=int(mappo.embedding_dim), depth=int(mappo.depth), num_layers=int(mappo.num_layers),
                action_dim=int(mappo.action_dim), n_params=int(mappo.ac_optimizer.flat_param.numel()),
                B=None if engine is None else int(engine.B), num_maps=None if engine is None else int(engine.M), rank=rank,
                world_size=world)


def save_training_state(path, mappo, engine=None, evaluator=None, extra=None):
    """Writes everything a training run carries from one iteration to the next to ONE `torch.save` file of CPU tensors and plain
    values (it loads with weights_only=True): a shape fingerprint, the actor / critic state_dicts (spectral-norm buffers included),
    the Adam state, `total_step`, the reward normaliser, the engine's state (`BatchedPursuitEnv.state_dict`), the evaluator's
    bookkeeping, the torch CPU / CUDA, Python `random` and numpy RNG states, and `extra` (the caller's loop counters).
    Take it between iterations, after `update()`.  Under torch.distributed every rank writes its own file."""
    rn = getattr(mappo, "reward_norm", None)
    np_state = np.random.get_state(legacy=False)
    st = dict(
        version=TRAINING_STATE_VERSION, meta=_fingerprint(mappo, engine),
        actor=_cpu_state(mappo.actor), critic=_cpu_state(mappo.critic), adam=mappo.ac_optimizer.state_dict(),
        total_step=int(mappo.total_step),
        reward_norm=None if rn is None else {k: getattr(rn.running_ms, k).cpu() for k in ("_n", "_mean", "_S", "_std")},
        engine=None if engine is None else engine.state_dict(),
        evaluator=None if evaluator is None else dict(recorder=[tuple(float(x) for x in row) for row in evaluator.recorder],
                                                      max_r=float(evaluator.max_r), seed=int(evaluator._seed),
                                                      total_step=int(evaluator.total_step)),
        rng=dict(torch_cpu=torch.get_rng_state(), torch_cuda=torch.cuda.get_rng_state(mappo.device), python=random.getstate(),
                 numpy=dict(bit_generator=np_state["bit_generator"], key=[int(k) for k in np_state["state"]["key"]],
                            pos=int(np_state["state"]["pos"]), has_gauss=int(np_state["has_gauss"]), gauss=float(np_state["gauss"]))),
        extra=dict(extra or {}))
    d = os.path.dirname(os.path.abspath(path))
    os.makedirs(d, exist_ok=True)
    tmp = path + ".tmp"
    torch.save(st, tmp)
    os.replace(tmp, path)          # a run interrupted while saving keeps the previous file


def load_training_state(path, mappo, engine=None, evaluator=None):
    """Restores a `save_training_state` file into freshly built objects of the same shape and returns its `extra` dict.  Every
    fingerprint field (N, E, depth, num_layers, action_dim, parameter count, B, number of maps, rank, world size) and every tensor
    shape is checked before anything is modified; a mismatch raises MarlError naming it.  Parameters are copied in place, so they
    stay views into the optimizer's flat arena."""
    st = torch.load(path, map_location="cpu", weights_only=True)
    if st.get("version") != TRAINING_STATE_VERSION:
        raise MarlError(f"{path}: training-state format {st.get('version')!r}, this build reads {TRAINING_STATE_VERSION}")
    want, have = st["meta"], _fingerprint(mappo, engine)
    for k in have:
        if engine is None and k in ("B", "num_maps"):
            continue
        if want.get(k) != have[k]:
            raise MarlError(f"{path}: {k} = {want.get(k)} in the file, {have[k]} here")
    if engine is not None and st["engine"] is None:
        raise MarlError(f"{path}: holds no engine state")
    if evaluator is not None and st["evaluator"] is None:
        raise MarlError(f"{path}: holds no evaluator state")
    rn = getattr(mappo, "reward_norm", None)
    if (rn is None) != (st["reward_norm"] is None):
        raise MarlError(f"{path}: reward normaliser {'absent' if st['reward_norm'] is None else 'present'} in the file, "
                        f"{'absent' if rn is None else 'present'} here")
    # shapes of everything below are checked before the first write
    for name, mod in (("actor", mappo.actor), ("critic", mappo.critic)):
        mine = mod.state_dict()
        if set(mine) != set(st[name]):
            raise MarlError(f"{path}: {name} state_dict keys differ: {sorted(set(mine) ^ set(st[name]))[:4]}")
        for k, v in mine.items():
            if tuple(v.shape) != tuple(st[name][k].shape):
                raise MarlError(f"{path}: {name}.{k} is {tuple(st[name][k].shape)}, here {tuple(v.shape)}")
    n = mappo.ac_optimizer.flat_param.numel()
    if st["adam"]["exp_avg"].numel() != n or st["adam"]["exp_avg_sq"].numel() != n:
        raise MarlError(f"{path}: Adam state of {st['adam']['exp_avg'].numel()} elements, here {n}")
    if engine is not None:
        for k in engine._STATE:
            src, dst = st["engine"].get(k), getattr(engine, k)
            if src is None or src.dtype != dst.dtype or (k != "target_tape" and tuple(src.shape) != tuple(dst.shape)):
                raise MarlError(f"{path}: engine {k} does not match this engine ({None if src is None else tuple(src.shape)} vs "
                                f"{tuple(dst.shape)})")
    with torch.no_grad():
        mappo.actor.load_state_dict(st["actor"])
        mappo.critic.load_state_dict(st["critic"])
    mappo.ac_optimizer.load_state_dict(st["adam"])
    mappo.total_step = int(st["total_step"])
    if rn is not None:
        for k, v in st["reward_norm"].items():
            getattr(rn.running_ms, k).copy_(v)
    if engine is not None:
        engine.load_state_dict(st["engine"])
    if evaluator is not None:
        ev = st["evaluator"]
        evaluator.recorder = [tuple(r) for r in ev["recorder"]]
        evaluator.max_r, evaluator._seed, evaluator.total_step = float(ev["max_r"]), int(ev["seed"]), int(ev["total_step"])
    rng = st["rng"]
    torch.set_rng_state(rng["torch_cpu"])
    torch.cuda.set_rng_state(rng["torch_cuda"], mappo.device)
    py = rng["python"]
    random.setstate((py[0], tuple(py[1]), py[2]))
    nps = rng["numpy"]
    np.random.set_state(dict(bit_generator=nps["bit_generator"], state=dict(key=np.asarray(nps["key"], dtype=np.uint32), pos=nps["pos"]),
                             has_gauss=nps["has_gauss"], gauss=nps["gauss"]))
    return dict(st["extra"])
