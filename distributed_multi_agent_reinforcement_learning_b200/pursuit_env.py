"""Pursuit-evasion environment: the batched B200 engine and the reference-compatible facade.

* `BatchedPursuitEnv` — B environments resident in HBM (SoA of [B,N,4] fp64 states, bit-packed maps and sensor
  tables), stepped by the sm_100a kernels behind the C-ABI (include/marl_b200.h).  This is the engine the
  rollout uses; nothing in it touches the host per step.
* `Pursuit_Env` — drop-in for the reference class of the same name
  (environment/pursuit_evasion_game/pursuit_env.py:56-229 and the identical top-level pursuit_env.py): same
  constructor, `reset/step/get_state/communicate/sensor/attacker_step/demon`, same return types (Python lists,
  ints, bool, None) and attributes (`num_defender, max_steps, time_step, collision, target,
  boundary_map.obstacle_agent, occupied_map, defender_list, attacker_list`).  It is a B=1 view of the engine.

There is no CPU fallback: constructing either class without the CUDA library / a CUDA device raises.
"""
import math
from types import SimpleNamespace

import numpy as np
import torch

from . import _lib, maps
from .config import env_params_dict


def _dev_i32(a, device):
    return torch.from_numpy(np.ascontiguousarray(a, dtype=np.int32)).to(device)


class BatchedPursuitEnv:
    """B independent pursuit-evasion environments on one GPU.

    Memory (HBM) per env at N=8, O=176, 60x55: state 256 B + evader 32 B + path 2 KB; per map: occupancy 480 B,
    inflated 480 B, raser table 3300 x 24 B = 79 KB (bit-packed; the reference's dense float list is 4.6 MB).
    """

    PATH_CAP = 512

    def __init__(self, cfg, num_envs, device="cuda:0", num_maps=None):
        if not torch.cuda.is_available():
            raise _lib.MarlError("BatchedPursuitEnv needs a CUDA device (no CPU fallback)")
        self.lib = _lib.lib()
        self.cfg = cfg
        self.device = torch.device(device)
        self.params = _lib.EnvParams.from_dict(env_params_dict(cfg))
        p = self.params
        self.B, self.N, self.O = int(num_envs), p.N, p.O
        self.M = int(num_maps) if num_maps else self.B
        B, N, M, dev = self.B, self.N, self.M, self.device
        f64, i32, u8 = torch.float64, torch.int32, torch.uint8
        self.p_state = torch.zeros(B, N, 4, dtype=f64, device=dev)
        self.e_state = torch.zeros(B, 4, dtype=f64, device=dev)
        self.target = torch.zeros(B, 2, dtype=i32, device=dev)
        self.path = torch.zeros(B, self.PATH_CAP, 2, dtype=torch.int16, device=dev)
        self.path_len = torch.zeros(B, dtype=i32, device=dev)
        self.time_step = torch.zeros(B, dtype=i32, device=dev)
        self.collision = torch.zeros(B, dtype=u8, device=dev)
        self.done = torch.zeros(B, dtype=u8, device=dev)
        self.reward = torch.zeros(B, N, dtype=i32, device=dev)
        self.can_apply = torch.zeros(B, N, dtype=u8, device=dev)
        self.evader_status = torch.zeros(B, dtype=i32, device=dev)
        self.map_id = torch.arange(B, dtype=i32, device=dev) % M
        self.grid_bits = torch.zeros(M, p.W, p.HW, dtype=i32, device=dev)
        self.inflated_bits = torch.zeros(M, p.W, p.HW, dtype=i32, device=dev)
        self.boundary_bits = torch.zeros(M, p.W, p.HW, dtype=i32, device=dev)
        self.boundary_count = torch.zeros(M, dtype=i32, device=dev)
        self.boundary_xy = torch.zeros(M, p.O, 2, dtype=i32, device=dev)
        self.raser_bits = torch.zeros(M, p.W * p.H, p.OW, dtype=i32, device=dev)
        self.action_table = torch.from_numpy(maps.action_table(cfg.defender.vmax)).to(dev)
        self.beam_dir = torch.from_numpy(maps.beam_directions(int(cfg.sensor.num_beams))).to(dev)
        self.target_tape = torch.zeros(B, 1, 2, dtype=i32, device=dev)
        self.tape_pos = torch.zeros(B, dtype=i32, device=dev)
        # observation outputs (packed canonical + optional dense fp32 in the reference layout)
        self.p_adj_bits = torch.zeros(B, N, p.NW, dtype=i32, device=dev)
        self.e_adj = torch.zeros(B, N, dtype=u8, device=dev)
        self.o_adj_bits = torch.zeros(B, N, p.OW, dtype=i32, device=dev)
        self._dense = None
        # per-env Welford state (DHGN/normalization.py)
        self.wf_n = torch.zeros(B, dtype=torch.int64, device=dev)
        self.wf_mean = torch.zeros(B, N, dtype=f64, device=dev)
        self.wf_S = torch.zeros(B, N, dtype=f64, device=dev)
        self.wf_std = torch.zeros(B, N, dtype=f64, device=dev)
        self.r_norm = torch.zeros(B, N, dtype=torch.float32, device=dev)
        self.launches = 0

    # ---------------------------------------------------------------------------------------------- set-up
    def _pp(self):
        import ctypes
        return ctypes.byref(self.params)

    def set_maps(self, grids, inflated=None):
        """grids: u8 [M,W,H] occupancy.  Uploads bit-packed maps and builds the sensor tables on the GPU."""
        grids = np.asarray(grids, dtype=np.uint8)
        assert grids.shape == (self.M, self.params.W, self.params.H), grids.shape
        if inflated is None:
            inflated = maps.dilate(grids, 2)
        self.grid_bits.copy_(torch.from_numpy(maps.pack_grid(grids)))
        self.inflated_bits.copy_(torch.from_numpy(maps.pack_grid(inflated)))
        self.build_sensor_tables()
        self.maps_set = True

    def build_sensor_tables(self):
        _lib.check(self.lib.marl_raser_map_build(
            self._pp(), self.M, _lib.ptr(self.grid_bits), _lib.ptr(self.beam_dir), _lib.ptr(self.boundary_bits),
            _lib.ptr(self.boundary_count), _lib.ptr(self.boundary_xy), _lib.ptr(self.raser_bits), _lib.stream_ptr()),
            "marl_raser_map_build")
        self.launches += 1

    def set_state(self, p_state=None, e_state=None, target=None, map_id=None, time_step=None):
        if p_state is not None:
            self.p_state.copy_(torch.as_tensor(np.asarray(p_state, dtype=np.float64)).reshape(self.B, self.N, 4))
        if e_state is not None:
            self.e_state.copy_(torch.as_tensor(np.asarray(e_state, dtype=np.float64)).reshape(self.B, 4))
        if target is not None:
            self.target.copy_(torch.as_tensor(np.asarray(target, dtype=np.int32)).reshape(self.B, 2))
        if map_id is not None:
            self.map_id.copy_(torch.as_tensor(np.asarray(map_id, dtype=np.int32)).reshape(self.B))
        if time_step is not None:
            self.time_step.fill_(int(time_step))

    def load_host_state(self, p_state=None, e_state=None, target=None, reset_reward_norm=False):
        """Start-of-episode state from HOST tensors (pinned memory makes the copies asynchronous): p_state f64 [B,N,4], e_state f64
        [B,4], target i32 [B,2]; clears the episode bookkeeping (time step, flags, evader path, target-tape cursor) and, on request,
        the running reward statistics.  Everything is queued on the current stream - no synchronisation."""
        for name, src in (("p_state", p_state), ("e_state", e_state), ("target", target)):
            if src is not None:
                dst = getattr(self, name)
                if src.dtype != dst.dtype or src.numel() != dst.numel():
                    raise _lib.MarlError(f"load_host_state: {name} must be {dst.dtype} with {dst.numel()} elements")
                dst.copy_(src.view(dst.shape), non_blocking=True)
        self.start_episode()
        self.tape_pos.zero_()
        if reset_reward_norm:
            for t in (self.wf_n, self.wf_mean, self.wf_S, self.wf_std):
                t.zero_()

    def set_target_tape(self, tape):
        """tape: int [B,L,2] candidate targets consumed by mid-episode init_target (base_env.py:52-70)."""
        tape = np.asarray(tape, dtype=np.int32).reshape(self.B, -1, 2)
        if tape.shape[1] == 0:
            tape = np.zeros((self.B, 1, 2), np.int32)
            self._tape_len = 0
        else:
            self._tape_len = tape.shape[1]
        self.target_tape = torch.from_numpy(tape).to(self.device)
        self.tape_pos.zero_()

    _tape_len = 0
    maps_set = False    # whether the maps were ever set (set_maps / MapPool.install, a "generate" reset, reset, load_state_dict)
    MAP_MODES = ("generate", "keep", "draw")

    def reset(self, seed=0):
        """Fresh episode for every env (host generation, reference rules; one map per pool slot)."""
        rng = maps.GenRng(seed)
        grids = np.zeros((self.M, self.params.W, self.params.H), np.uint8)
        infl = np.zeros_like(grids)
        per_map = []
        for m in range(self.M):
            r = maps.reset_one(self.cfg, rng)
            grids[m], infl[m] = r["grid"], r["inflated"]
            per_map.append(r)
        self.set_maps(grids, infl)
        mid = np.arange(self.B) % self.M
        ps = np.stack([per_map[m]["p_state"] for m in mid])
        es = np.stack([per_map[m]["e_state"] for m in mid])
        tg = np.stack([per_map[m]["target"] for m in mid])
        if self.B > self.M:   # envs sharing a map still get their own placement
            for b in range(self.M, self.B):
                m = mid[b]
                work = infl[m].copy()
                tg[b] = maps.draw_target(infl[m], rng)
                pxy, cells = maps.place_pursuers(work, self.N, float(self.cfg.defender.comm_range), rng)
                ps[b, :, :2] = pxy
                es[b, :2] = maps.place_evader(work, cells, float(self.cfg.defender.sen_range), rng)
        self.set_state(ps, es, tg, mid, time_step=0)
        self.start_episode()

    def reset_device(self, seed=0, tape_len=16, tape="torch", maps="generate"):
        """Fresh episode for every env, generated ON THE GPU (csrc/reset_kernels.cu): maps, sensor tables, targets, pursuers,
        evaders and the candidate-target tape.  Same placement rules as `reset` / the reference, per-env counter RNG streams.

        tape: "torch" draws the tape [B, tape_len, 2] with a torch.Generator seeded from `seed`; "device" draws it with
        marl_target_tape_generate (env b's own counter stream of (seed, b), the same distribution).  Everything else is the same in
        both modes.  When tape_len is unchanged the tape is written into the existing `target_tape` storage, so a CUDA graph that
        reads it keeps reading the current episode's tape.
        seed: a host int, or (tape="device" only) a one-element int64 device tensor holding the seed's u64 bit pattern, read when the
        kernels run: then every launch is graph-capturable (no generator, no host read, no allocation after the first call).
        maps: "generate" generates all M maps and builds their sensor tables; "keep" keeps the M maps the engine holds (e.g. a pool
        installed with MapPool.install) and the map assignment `map_id`, and draws the placements and the tape only; "draw" is "keep"
        after marl_map_draw gives every env a map drawn uniformly from the M held ones (env b's own stream of (seed, b), written into
        `map_id` in place).  "keep" / "draw" need maps that were set (set_maps, MapPool.install, a "generate" reset, reset or
        load_state_dict): MarlError otherwise, before any CUDA call."""
        import ctypes
        if maps not in self.MAP_MODES:
            raise ValueError(f"reset_device: maps={maps!r}: 'generate', 'keep' or 'draw'")
        if maps != "generate" and not self.maps_set:
            raise _lib.MarlError(f"reset_device(maps={maps!r}) keeps the engine's maps, but they were never set (install a pool with "
                                 "MapPool.install, call set_maps, or reset with maps='generate' first)")
        if tape not in ("torch", "device"):
            raise ValueError(f"tape={tape!r}: 'torch' or 'device'")
        on_device = isinstance(seed, torch.Tensor)
        if on_device and tape != "device":
            raise _lib.MarlError("reset_device: a device-resident seed needs tape='device' (the torch tape is drawn from a host seed)")
        if tape == "device" and int(tape_len) < 1:
            raise _lib.MarlError(f"reset_device: tape_len={tape_len}; the device tape has at least one entry")
        p, mc = self.params, self.cfg.map
        self._reset_buffers()
        if on_device:
            if seed.dtype != torch.int64 or seed.numel() != 1 or not seed.is_cuda:
                raise _lib.MarlError("reset_device: a device seed is one int64 element on the engine's device")
            seed_arg, gen, place, sfx = _lib.ptr(seed), self.lib.marl_map_generate_dseed, self.lib.marl_env_reset_place_dseed, "_dseed"
            draw = self.lib.marl_map_draw_dseed
        else:
            seed_arg = ctypes.c_uint64(int(seed) & 0xFFFFFFFFFFFFFFFF)
            gen, place, sfx = self.lib.marl_map_generate, self.lib.marl_env_reset_place, ""
            draw = self.lib.marl_map_draw
        if maps == "generate":
            _lib.check(gen(self._pp(), self.M, int(mc.num_obstacle_block), ctypes.c_double(float(mc.center[0])),
                           ctypes.c_double(float(mc.center[1])), ctypes.c_double(float(mc.variance)), seed_arg, _lib.ptr(self.grid_bits),
                           _lib.ptr(self.inflated_bits), _lib.stream_ptr()), "marl_map_generate" + sfx)
            self.build_sensor_tables()
            self.maps_set = True
        elif maps == "draw":
            _lib.check(draw(self._pp(), self.B, self.M, seed_arg, _lib.ptr(self.map_id), _lib.stream_ptr()), "marl_map_draw" + sfx)
        _lib.check(place(self._pp(), self.B, self.M, _lib.ptr(self.inflated_bits), _lib.ptr(self.map_id), seed_arg, ctypes.c_double(4.0),
                         2, 200000, _lib.ptr(self.p_state), _lib.ptr(self.e_state), _lib.ptr(self.target), _lib.ptr(self._reset_scratch),
                         _lib.ptr(self.reset_fail), _lib.stream_ptr()), "marl_env_reset_place" + sfx)
        self.launches += 1 + (maps != "keep")      # the map generation or draw, and the placement (the table build counts itself)
        shape = (self.B, int(tape_len), 2)
        if tuple(self.target_tape.shape) != shape or not self.target_tape.is_contiguous():
            self.target_tape = torch.empty(shape, dtype=torch.int32, device=self.device)
        if tape == "device":
            if not on_device:
                self._seed_word.fill_(_lib.u64_bits(seed))
                seed = self._seed_word
            _lib.check(self.lib.marl_target_tape_generate(self._pp(), self.B, int(tape_len), _lib.ptr(seed), _lib.ptr(self.target_tape),
                                                          _lib.stream_ptr()), "marl_target_tape_generate")
            self.launches += 1
        else:
            g = torch.Generator(device=self.device).manual_seed(int(seed) & 0x7FFFFFFFFFFFFFFF)
            self.target_tape.copy_(torch.stack([torch.randint(0, p.W, (self.B, tape_len), generator=g, device=self.device),
                                                torch.randint(0, p.H, (self.B, tape_len), generator=g, device=self.device)], dim=-1))
        self._tape_len = int(tape_len)
        self.tape_pos.zero_()
        self.start_episode()

    def _reset_buffers(self):
        """The device reset's scratch rows, failure flags and seed word (allocated once)."""
        if getattr(self, "_reset_scratch", None) is None:
            p = self.params
            self._reset_scratch = torch.empty(self.B, p.W, p.HW, dtype=torch.int32, device=self.device)
            self.reset_fail = torch.zeros(self.B, dtype=torch.int32, device=self.device)
            self._seed_word = torch.zeros(1, dtype=torch.int64, device=self.device)

    def start_episode(self):
        self.time_step.zero_()
        self.collision.zero_()
        self.done.zero_()
        self.path_len.zero_()
        self.evader_status.zero_()

    # ---------------------------------------------------------------------------------------------- kernels
    def dense_views(self):
        if self._dense is None:
            B, N, O, dev = self.B, self.N, self.O, self.device
            self._dense = (torch.zeros(B, N, N, dtype=torch.float32, device=dev),
                           torch.zeros(B, N, 1, dtype=torch.float32, device=dev),
                           torch.zeros(B, N, O, dtype=torch.float32, device=dev))
        return self._dense

    def observe(self, dense=False, lo=0, hi=None):
        """communicate() + sensor() for all envs (or envs [lo, hi)).  Packed words always; dense fp32 (reference layout) on
        request (whole batch only)."""
        d = self.dense_views() if dense else (None, None, None)
        hi = self.B if hi is None else hi
        sl = slice(lo, hi)
        assert not dense or (lo == 0 and hi == self.B)
        _lib.check(self.lib.marl_env_observe(
            self._pp(), hi - lo, self.M, _lib.ptr(self.p_state[sl]), _lib.ptr(self.e_state[sl]), _lib.ptr(self.grid_bits),
            _lib.ptr(self.raser_bits), _lib.ptr(self.map_id[sl]), _lib.ptr(self.p_adj_bits[sl]), _lib.ptr(self.e_adj[sl]),
            _lib.ptr(self.o_adj_bits[sl]), _lib.ptr(d[0]), _lib.ptr(d[1]), _lib.ptr(d[2]), _lib.stream_ptr()),
            "marl_env_observe")
        self.launches += 1
        return d if dense else (self.p_adj_bits, self.e_adj, self.o_adj_bits)

    def evader_step(self, e_tape2=None):
        """attacker_step() for all envs (A* replanning every `difficulty` steps + waypoint following).
        e_tape2: optional f64 [2,B,4] receiving the evader state before/after (feeds rollout(K=1))."""
        _lib.check(self.lib.marl_evader_step(
            self._pp(), self.B, self.M, _lib.ptr(self.e_state), _lib.ptr(self.p_state), _lib.ptr(self.target),
            _lib.ptr(self.path), _lib.ptr(self.path_len), self.PATH_CAP, _lib.ptr(self.time_step),
            _lib.ptr(self.grid_bits), _lib.ptr(self.inflated_bits), _lib.ptr(self.map_id),
            _lib.ptr(self.target_tape), self._tape_len, _lib.ptr(self.tape_pos), _lib.ptr(self.evader_status),
            _lib.ptr(e_tape2), _lib.stream_ptr()), "marl_evader_step")
        self.launches += 1

    def step(self, action):
        """Pursuit_Env.step for all envs.  action: int32 [B,N] device tensor."""
        if action.dtype != torch.int32 or action.device != self.device:
            action = action.to(device=self.device, dtype=torch.int32)
        action = action.contiguous()
        _lib.check(self.lib.marl_env_step(
            self._pp(), self.B, self.M, _lib.ptr(self.p_state), _lib.ptr(self.e_state), _lib.ptr(action),
            _lib.ptr(self.grid_bits), _lib.ptr(self.map_id), _lib.ptr(self.action_table), _lib.ptr(self.reward),
            _lib.ptr(self.can_apply), _lib.ptr(self.collision), _lib.ptr(self.time_step), _lib.ptr(self.done),
            _lib.stream_ptr()), "marl_env_step")
        self.launches += 1
        return self.reward, self.done

    def normalize_reward(self, update=True):
        """Normalization(shape=N)(r) per env (DHGN/normalization.py:25-35) on the last step's rewards."""
        _lib.check(self.lib.marl_welford_update(
            self.B, self.N, _lib.ptr(self.reward), _lib.ptr(self.wf_n), _lib.ptr(self.wf_mean), _lib.ptr(self.wf_S),
            _lib.ptr(self.wf_std), _lib.ptr(self.r_norm), 1 if update else 0, _lib.stream_ptr()),
            "marl_welford_update")
        self.launches += 1
        return self.r_norm

    def rollout(self, arena, K, t0=0, e_tape=None, action_tape=None, seed=0, sync_evader=True):
        """K fused env-only iterations (observe -> evader tape -> step -> reward-norm -> store) in ONE launch.
        arena: RolloutArena.  e_tape f64 [K+1,B,4]; action_tape i32 [K,B,N] or None (counter-based uniform)."""
        assert e_tape is not None and tuple(e_tape.shape) == (K + 1, self.B, 4) and e_tape.dtype == torch.float64
        if action_tape is not None:
            assert tuple(action_tape.shape) == (K, self.B, self.N) and action_tape.dtype == torch.int32
        import ctypes
        rec = arena.records()
        _lib.check(self.lib.marl_rollout_steps(
            self._pp(), self.B, self.M, arena.T, t0, K, _lib.ptr(self.p_state), _lib.ptr(e_tape),
            _lib.ptr(action_tape), ctypes.c_uint64(seed), _lib.ptr(self.grid_bits), _lib.ptr(self.raser_bits),
            _lib.ptr(self.map_id), _lib.ptr(self.action_table), _lib.ptr(self.wf_n), _lib.ptr(self.wf_mean),
            _lib.ptr(self.wf_S), _lib.ptr(self.wf_std), _lib.ptr(self.collision), _lib.ptr(self.time_step),
            ctypes.byref(rec), _lib.stream_ptr()), "marl_rollout_steps")
        self.launches += 1
        if sync_evader:
            self.e_state.copy_(e_tape[K])

    def evader_replan(self, lo=0, hi=None, stream=None):
        """Evader.replan for every env in [lo, hi) whose time_step is a multiple of `difficulty`."""
        hi = self.B if hi is None else hi
        sl = slice(lo, hi)
        _lib.check(self.lib.marl_evader_replan(
            self._pp(), hi - lo, self.M, _lib.ptr(self.e_state[sl]), _lib.ptr(self.p_state[sl]),
            _lib.ptr(self.target[sl]), _lib.ptr(self.path[sl]), _lib.ptr(self.path_len[sl]), self.PATH_CAP,
            _lib.ptr(self.time_step[sl]), _lib.ptr(self.grid_bits), _lib.ptr(self.map_id[sl]),
            _lib.ptr(self.evader_status[sl]), _lib.stream_ptr(stream)), "marl_evader_replan")
        self.launches += 1

    def _closed_chunk(self, arena, rec_ptrs, lo, hi, t, chunk, action_tape, k, seed, stream):
        """One marl_rollout_closed launch for envs [lo, hi) and arena time index t."""
        import ctypes
        sl = slice(lo, hi)
        rec = _lib.RolloutRecords()
        for f, (base, row_bytes) in rec_ptrs.items():
            setattr(rec, f, None if base is None else base + lo * row_bytes)
        tape = None
        if action_tape is not None:
            tape = action_tape[k].data_ptr() + lo * self.N * 4      # [K,B,N] int32, env-offset, B_stride time stride
        _lib.check(self.lib.marl_rollout_closed(
            self._pp(), hi - lo, self.B, lo, self.M, arena.T, t, chunk, _lib.ptr(self.p_state[sl]),
            _lib.ptr(self.e_state[sl]), _lib.ptr(self.target[sl]), _lib.ptr(self.path[sl]), _lib.ptr(self.path_len[sl]),
            self.PATH_CAP, _lib.ptr(self.inflated_bits), _lib.ptr(self.target_tape[sl]), self._tape_len,
            _lib.ptr(self.tape_pos[sl]), _lib.ptr(self.evader_status[sl]), tape, ctypes.c_uint64(seed),
            _lib.ptr(self.grid_bits), _lib.ptr(self.raser_bits), _lib.ptr(self.map_id[sl]), _lib.ptr(self.action_table),
            _lib.ptr(self.wf_n[sl]), _lib.ptr(self.wf_mean[sl]), _lib.ptr(self.wf_S[sl]), _lib.ptr(self.wf_std[sl]),
            _lib.ptr(self.collision[sl]), _lib.ptr(self.time_step[sl]), ctypes.byref(rec), _lib.stream_ptr(stream)),
            "marl_rollout_closed")
        self.launches += 1

    def rollout_closed(self, arena, K, t0=0, action_tape=None, seed=0, env_t0=0, groups=1):
        """K closed-loop env iterations with the A* evader on the GPU.  The evader's per-step move is fused into the
        rollout kernel; replanning is one launch per `difficulty` steps, so K steps are 2*ceil(K/difficulty) launches
        per group.  `env_t0` is the (lock-step) env time_step at entry.

        groups > 1 splits the envs into that many contiguous sub-batches, each running its own launch chain on its own
        CUDA stream: a search that takes 100x longer than the median (A* is a long-tailed workload) then only holds
        up its own sub-batch while the other chains keep the SMs busy.  Results are identical for any grouping.
        Nothing touches the host, so the whole thing can be captured in a CUDA graph (EpisodeGraph)."""
        assert arena.B == self.B
        if action_tape is not None:
            assert tuple(action_tape.shape) == (K, self.B, self.N) and action_tape.dtype == torch.int32
            assert action_tape.is_contiguous()
        D = self.params.difficulty
        rec_ptrs = arena.record_pointers()
        groups = max(1, min(int(groups), self.B))
        bounds = [(g * self.B // groups, (g + 1) * self.B // groups) for g in range(groups)]

        def chain(lo, hi, stream):
            k = 0
            while k < K:
                ts = env_t0 + k
                if ts % D == 0:
                    self.evader_replan(lo, hi, stream)
                chunk = min(D - ts % D, K - k)
                self._closed_chunk(arena, rec_ptrs, lo, hi, t0 + k, chunk, action_tape, k, seed, stream)
                k += chunk

        if groups == 1:
            chain(0, self.B, None)
            return
        main = torch.cuda.current_stream()
        if len(getattr(self, "_streams", [])) < groups:
            self._streams = [torch.cuda.Stream(device=self.device) for _ in range(groups)]
        fork = torch.cuda.Event()
        fork.record(main)
        for (lo, hi), st in zip(bounds, self._streams):
            st.wait_event(fork)
            chain(lo, hi, st)
            done = torch.cuda.Event()
            done.record(st)
            main.wait_event(done)

    def snapshot(self):
        """Device-side copy of everything an episode mutates (for replaying identical episodes)."""
        names = ("p_state", "e_state", "target", "path", "path_len", "time_step", "collision", "done", "tape_pos",
                 "evader_status", "wf_n", "wf_mean", "wf_S", "wf_std")
        return {n: getattr(self, n).clone() for n in names}

    def restore(self, snap):
        for n, t in snap.items():
            getattr(self, n).copy_(t)

    # everything that persists from one training iteration to the next: the snapshot (Welford statistics included), the map
    # assignment, the target tape and the map / sensor tables (a pool installed once with MapPool.install survives a resume)
    _STATE = ("p_state", "e_state", "target", "path", "path_len", "time_step", "collision", "done", "tape_pos", "evader_status",
              "wf_n", "wf_mean", "wf_S", "wf_std", "map_id", "target_tape", "grid_bits", "inflated_bits", "boundary_bits",
              "boundary_count", "boundary_xy", "raser_bits")

    def state_dict(self):
        """CPU copies of the engine's persistent tensors, plus the target-tape length."""
        sd = {n: getattr(self, n).cpu() for n in self._STATE}
        sd["tape_len"] = int(self._tape_len)
        return sd

    def load_state_dict(self, sd):
        """Inverse of `state_dict`.  Every tensor is checked against this engine's shapes and dtypes before any is written (the
        target tape may have another length); raises MarlError naming the first mismatch."""
        for n in self._STATE:
            if n not in sd:
                raise _lib.MarlError(f"engine state: {n} missing")
            src, dst = sd[n], getattr(self, n)
            same = tuple(src.shape) == tuple(dst.shape) or (n == "target_tape" and src.dim() == 3 and src.shape[0] == self.B
                                                             and src.shape[2] == 2)
            if not same or src.dtype != dst.dtype:
                raise _lib.MarlError(f"engine state: {n} is {tuple(src.shape)} {src.dtype}, this engine's is {tuple(dst.shape)} {dst.dtype}")
        for n in self._STATE:
            if n == "target_tape" and tuple(sd[n].shape) != tuple(self.target_tape.shape):
                self.target_tape = sd[n].to(self.device).contiguous()
            else:
                getattr(self, n).copy_(sd[n])
        self._tape_len = int(sd["tape_len"])
        self.maps_set = True


class EpisodeGraph:
    """One whole closed-loop episode (2*ceil(T/difficulty) kernel launches) captured in a CUDA graph, so replaying
    an episode costs one host call."""

    def __init__(self, env, arena, T, seed=0, groups=1):
        self.env, self.arena, self.T, self.groups = env, arena, T, groups
        snap = env.snapshot()
        env.rollout_closed(arena, T, 0, seed=seed, groups=groups)   # eager warm-up (also sets kernel attributes)
        torch.cuda.synchronize()
        env.restore(snap)
        self.graph = torch.cuda.CUDAGraph()
        side = torch.cuda.Stream()
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):
            with torch.cuda.graph(self.graph, stream=side):
                env.rollout_closed(arena, T, 0, seed=seed, groups=groups)
        torch.cuda.current_stream().wait_stream(side)
        torch.cuda.synchronize()
        env.restore(snap)
        D = env.params.difficulty
        self.launches_per_replay = 2 * ((T + D - 1) // D) * max(1, min(groups, env.B))

    def replay(self):
        self.graph.replay()


class RolloutArena:
    """Time-major rollout storage [T,B,N,...] in HBM (DESIGN.md §3): one env-step of all envs is one contiguous
    slab, so the per-step stores of the rollout kernel are fully coalesced, and the GRU's [T, B*N, ...] view is
    free.  The reference's ReplayBuffer tensors ([B,T,...], DHGN/replay_buffer.py:28-40) are zero-copy permuted
    views (`reference_view`).  Adjacency is bit-packed (32x smaller than the reference's fp32 0/1 matrices)
    unless `dense=True` asks for the reference's fp32 layout as well."""

    def __init__(self, params, B, T, device, dense=False):
        N, O, NW, OW = params.N, params.O, params.NW, params.OW
        f32, i32, u8 = torch.float32, torch.int32, torch.uint8
        z = lambda *s, dtype=f32: torch.zeros(*s, dtype=dtype, device=device)
        self.B, self.T, self.N, self.O = B, T, N, O
        self.p_state_f32 = z(T, B, N, 4)
        self.e_state_f32 = z(T, B, 1, 4)
        self.p_adj_bits = z(T, B, N, NW, dtype=i32)
        self.e_adj = z(T, B, N, dtype=u8)
        self.o_adj_bits = z(T, B, N, OW, dtype=i32)
        self.a_n = z(T, B, N)
        self.r = z(T, B, N)
        self.raw_reward = z(T, B, N, dtype=i32)
        self.active = z(T, B, N)
        self.p_adj_f32 = z(T, B, N, N) if dense else None
        self.e_adj_f32 = z(T, B, N, 1) if dense else None
        self.o_adj_f32 = z(T, B, N, O) if dense else None

    def records(self):
        rec = _lib.RolloutRecords()
        for f in _lib.RolloutRecords.FIELDS:
            t = getattr(self, f)
            setattr(rec, f, t.data_ptr() if t is not None else None)
        return rec

    def record_pointers(self):
        """field -> (device base pointer or None, bytes per env row of one time slab)."""
        out = {}
        for f in _lib.RolloutRecords.FIELDS:
            t = getattr(self, f)
            out[f] = (None, 0) if t is None else (t.data_ptr(), t[0, 0].numel() * t.element_size())
        return out

    def nbytes(self):
        return sum(getattr(self, f).numel() * getattr(self, f).element_size()
                   for f in _lib.RolloutRecords.FIELDS if getattr(self, f) is not None)

    def reference_view(self, key):
        """[B,T,...] view with the reference ReplayBuffer key names (p_state, e_state, a_n, r, active, p_adj,
        e_adj, o_adj — the last three need dense=True)."""
        name = {"p_state": "p_state_f32", "e_state": "e_state_f32", "p_adj": "p_adj_f32", "e_adj": "e_adj_f32",
                "o_adj": "o_adj_f32"}.get(key, key)
        t = getattr(self, name)
        if t is None:
            raise KeyError(f"{key}: arena was created without dense=True")
        return t.transpose(0, 1)


# ---------------------------------------------------------------------------------------------------- facade
class _AgentView:
    """defender_list / attacker_list element: attribute view of one agent's host-side state."""

    def __init__(self, env, kind, idx):
        self._env, self._kind, self._idx = env, kind, idx
        self.theta = 0.0

    def _row(self):
        return self._env._host_p[self._idx] if self._kind == "defender" else self._env._host_e

    x = property(lambda s: float(s._row()[0]), lambda s, v: s._env._poke(s._kind, s._idx, 0, v))
    y = property(lambda s: float(s._row()[1]), lambda s, v: s._env._poke(s._kind, s._idx, 1, v))
    vx = property(lambda s: float(s._row()[2]), lambda s, v: s._env._poke(s._kind, s._idx, 2, v))
    vy = property(lambda s: float(s._row()[3]), lambda s, v: s._env._poke(s._kind, s._idx, 3, v))


class Pursuit_Env:
    """Reference-compatible single environment (B=1 view of BatchedPursuitEnv).

    `reset()` draws from the global `random` / `np.random` streams in the reference's order, so identical seeds
    give the reference's initial state.  Mid-episode target resampling also uses `random.randint`
    (pursuit_env.py:98-100 -> base_env.py:63-70)."""

    def __init__(self, cfg, device="cuda:0"):
        self.cfg = cfg
        self.map_config, self.env_config = cfg.map, cfg.env
        self.defender_config, self.attacker_config, self.sensor_config = cfg.defender, cfg.attacker, cfg.sensor
        self.num_defender = int(cfg.env.num_defender)
        self.num_attacker = int(cfg.env.num_attacker)
        self.num_target = int(cfg.env.num_target)
        self.max_steps = int(cfg.env.max_steps)
        self.step_size = cfg.env.step_size
        self.time_step = 0
        self.n_episode = 0
        self.collision = False
        self.engine = BatchedPursuitEnv(cfg, 1, device=device, num_maps=1)
        self.defender_list = [_AgentView(self, "defender", i) for i in range(self.num_defender)]
        self.attacker_list = [_AgentView(self, "attacker", 0)]
        self._host_p = np.zeros((self.num_defender, 4))
        self._host_e = np.zeros(4)
        self.target = [(0, 0)]

    # -- host mirrors ------------------------------------------------------------------------------------
    def _pull(self):
        self._host_p = self.engine.p_state[0].cpu().numpy()
        self._host_e = self.engine.e_state[0].cpu().numpy()

    def _poke(self, kind, idx, col, v):
        if kind == "defender":
            self.engine.p_state[0, idx, col] = float(v)
        else:
            self.engine.e_state[0, col] = float(v)
        self._pull()

    def reset(self):
        self.time_step = 0
        self.n_episode += 1
        self.collision = False
        r = maps.reset_one(self.cfg, maps.RefRng())
        eng = self.engine
        eng.set_maps(r["grid"][None], r["inflated"][None])
        eng.set_state(r["p_state"][None], r["e_state"][None], r["target"][None], np.zeros(1, np.int32), time_step=0)
        eng.start_episode()
        eng.set_target_tape(np.zeros((1, 0, 2), np.int32))
        self._inflated = r["inflated"]
        self.target = [tuple(int(v) for v in r["target"])]
        n_b = int(eng.boundary_count[0].item())
        if n_b > eng.O:
            raise _lib.MarlError(f"map has {n_b} boundary cells > map.num_max_obstacle={eng.O}")
        bxy = eng.boundary_xy[0, :n_b].cpu().numpy()
        self._n_boundary = n_b
        grid = r["grid"].astype(np.float64)
        self.occupied_map = SimpleNamespace(grid_map=grid, boundaries=tuple(self.map_config.map_size),
                                            obstacles=[tuple(int(v) for v in c) for c in np.argwhere(grid == 1)])
        self.inflated_map = SimpleNamespace(grid_map=r["inflated"].astype(np.float64), boundaries=tuple(self.map_config.map_size))
        self.boundary_map = SimpleNamespace(
            grid_map=maps.unpack_words(eng.boundary_bits[0].cpu().numpy(), self.engine.params.H).astype(bool),
            obstacles=[[int(x), int(y)] for x, y in bxy], obstacle_agent=[[int(x), int(y), 0, 0] for x, y in bxy],
            boundaries=tuple(self.map_config.map_size))
        self._pull()

    # -- whole-episode hand-off to the batched rollout (MAPPO.explore_env) -----------------------------------------
    def begin_batched_episode(self, tape_len=64):
        """Pre-draws candidate targets from the global `random` stream for the device-side evader; the stream is put
        back in `end_batched_episode` so that exactly as many draws are consumed as the reference would have made."""
        import random
        W, H = self.map_config.map_size
        self._rng_state = random.getstate()
        tape = [(random.randint(0, W - 1), random.randint(0, H - 1)) for _ in range(tape_len)]
        random.setstate(self._rng_state)
        self.engine.set_target_tape(np.asarray(tape, np.int32).reshape(1, tape_len, 2))

    def end_batched_episode(self):
        import random
        eng = self.engine
        status = int(eng.evader_status[0].item())
        if status:
            raise _lib.MarlError(f"evader status {status} (search overflow or target tape exhausted)")
        W, H = self.map_config.map_size
        for _ in range(int(eng.tape_pos[0].item())):          # replay the draws the episode actually consumed
            random.randint(0, W - 1), random.randint(0, H - 1)
        self.time_step = int(eng.time_step[0].item())
        self.collision = bool(eng.collision[0].item())
        self.target = [tuple(int(v) for v in eng.target[0].cpu().numpy())]
        self._pull()

    def get_state(self, agent_type):
        if agent_type == "defender":
            return [[float(v) for v in row] for row in self._host_p]
        return [[float(v) for v in self._host_e]]

    def get_agent_state(self, agent):
        return [agent.x, agent.y, agent.vx, agent.vy]

    def communicate(self):
        p_adj, _, _ = self.engine.observe(dense=True)
        return p_adj[0].cpu().numpy().astype(np.float64).tolist()

    def sensor(self):
        _, e_adj, o_adj = self.engine.observe(dense=True)
        o = o_adj[0, :, :self._n_boundary].cpu().numpy().astype(np.float64).tolist()
        e = [[int(v)] for v in e_adj[0, :, 0].cpu().numpy()]
        return o, e

    def attacker_step(self):
        import random
        eng = self.engine
        eng.evader_status.zero_()
        eng.evader_step()
        status = int(eng.evader_status[0].item())
        if status & ~_lib.EV_TAPE_EXHAUSTED:
            raise _lib.MarlError(f"evader search overflow (status {status})")
        if status & _lib.EV_TAPE_EXHAUSTED:   # target reached: resample like base_env.py:52-70
            W, H = self.map_config.map_size
            while True:
                t = (random.randint(0, W - 1), random.randint(0, H - 1))
                if not self._inflated[t[0], t[1]]:
                    break
            self.target = [t]
            eng.target.copy_(torch.tensor([list(t)], dtype=torch.int32))
        self._pull()
        n = int(eng.path_len[0].item())
        path = eng.path[0, :n].cpu().numpy()
        return [[(int(x), int(y)) for x, y in path]]

    def step(self, action):
        act = torch.as_tensor(np.asarray(action, dtype=np.int64).reshape(1, -1).astype(np.int32), device=self.engine.device)
        reward, done = self.engine.step(act)
        self.time_step += 1
        self._pull()
        self.collision = bool(self.engine.collision[0].item())
        return [int(v) for v in reward[0].cpu().numpy()], bool(done[0].item()), None

    def demon(self):
        """Scripted chaser (pursuit_env.py:211-229): the discrete action closest to the bearing of the evader."""
        table = [[np.cos(i * np.pi / 4), np.sin(i * np.pi / 4)] for i in range(8)] + [[0.0, 0.0]]
        ex, ey = self._host_e[0], self._host_e[1]
        out = []
        for x, y, _, _ in self._host_p:
            rad = np.linalg.norm([x - ex, y - ey])
            if math.isclose(rad, 0.0, abs_tol=0.01):
                want = [0.0, 0.0]
            else:
                phi = np.sign(ey - y) * np.arccos((ex - x) / (rad + 1e-3))
                want = [np.cos(phi), np.sin(phi)]
            d = [np.linalg.norm((a[0] - want[0], a[1] - want[1])) for a in table]
            out.append(d.index(min(d)))
        return out

    def get_done(self):
        pass
