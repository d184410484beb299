"""Evaluator path of the reference (evaluator.py:20-201), without Ray.

* `evaluate(env, actor, cfg)` — one deterministic (arg-max) episode of the actor in a `Pursuit_Env`, step by step through the
  reference-facing facade (`get_state / communicate / sensor / attacker_step / step`, `actor.choose_action`); returns
  `[episode_reward, last_step_index]` exactly like evaluator.py:107-201.  Every network / env operation is one of our kernels.
* `Evaluator` — the bookkeeping of `EvaluatorProc` (evaluator.py:20-103): `run`, `evaluate_and_save`, `recorder` rows
  `(total_step, avg_r, std_r, exp_r, *logging_tuple)`, "save when the average return does not get worse".  Its episodes are
  ONE batched arg-max rollout of `num_cpus_eval` independent environments on the GPU (`MAPPO.rollout_batched(deterministic=
  True, actor_only=True)`: the actor alone, fed with its own previous embeddings exactly as `evaluate` does) instead of
  `num_cpus_eval` Ray tasks.  With a map pool (`Evaluator(..., pool=, pool_indices=)`) the episodes are played on a fixed
  held-out set of maps, so successive evaluations are comparable.
"""
import time

import numpy as np
import torch

from .mappo_parallel import AttributeDataset, EmbeddingDataset
from .pursuit_env import BatchedPursuitEnv, RolloutArena


def evaluate(env, actor, cfg):
    """evaluator.py:107-201.  env: Pursuit_Env facade; actor: SharedActor.  Returns [episode_reward, step]."""
    dev = next(actor.parameters()).device
    algo = cfg.algo
    env.reset()
    n = env.num_defender
    hidden = torch.zeros(algo.num_layers, n, algo.rnn_hidden_dim, dtype=torch.float32, device=dev)
    history = EmbeddingDataset(attribute=[torch.zeros(n, algo.embedding_dim, dtype=torch.float32, device=dev)
                                          for _ in range(algo.depth)], adjacent=None, depth=algo.depth)
    current = torch.zeros(n, algo.embedding_dim, dtype=torch.float32, device=dev)
    obstacles = torch.as_tensor(env.boundary_map.obstacle_agent, dtype=torch.float32, device=dev)
    episode_reward, step = 0, 0
    with torch.no_grad():
        for step in range(env.max_steps):
            pursuers = torch.as_tensor(env.get_state(agent_type="defender"), dtype=torch.float32, device=dev)
            evader = torch.as_tensor(env.get_state(agent_type="attacker"), dtype=torch.float32, device=dev)
            p_adj = torch.as_tensor(env.communicate(), dtype=torch.float32, device=dev)
            o_adj, e_adj = env.sensor()
            o_adj = torch.as_tensor(o_adj, dtype=torch.float32, device=dev)
            e_adj = torch.as_tensor(e_adj, dtype=torch.float32, device=dev)
            env.attacker_step()                                   # the evader moves before the pursuers act (evaluator.py:143)
            attributes = AttributeDataset(attribute=[pursuers, evader, obstacles], adjacent=[p_adj, e_adj, o_adj])
            history.update(embedding=current, adjacent=p_adj)
            actions, hidden, current = actor.choose_action(attributes, history, hidden, deterministic=True)
            current = current.squeeze(0)
            rewards, done, _ = env.step(actions.detach().cpu().numpy())
            episode_reward += sum(rewards)
            if done:
                break
    return [episode_reward, step]


class Evaluator:
    """EvaluatorProc (evaluator.py:20-103) as a plain object.  `agent` is a MAPPO built with agent_type "Evaluator"."""

    def __init__(self, cfg, num_cpus_eval, agent, device=None, seed=0, pool=None, pool_indices=None):
        """pool / pool_indices: evaluate on a fixed held-out set of maps, maps `pool_indices` of a MapPool (default: all of it).  The
        engine then holds exactly those M maps, installed once (verify=True) on first use, and every evaluation keeps them: env b plays
        map b % M, and only the placements and the target tape come from the evaluation's seed.  Without a pool, every evaluation
        generates new maps."""
        self.cfg, self.agent, self.num_cpus_eval = cfg, agent, int(num_cpus_eval)
        self.pool = pool
        self.pool_indices = None
        if pool is not None:
            idx = np.arange(len(pool)) if pool_indices is None else np.asarray(pool_indices, dtype=np.int64).reshape(-1)
            if idx.size == 0:
                raise ValueError("Evaluator: pool_indices selects no map")
            self.pool_indices = idx
        elif pool_indices is not None:
            raise ValueError("Evaluator: pool_indices without a pool")
        self.device = torch.device(device) if device is not None else agent.device
        self.total_step = 0
        self.start_time = time.time()
        self.break_step = cfg.algo.max_train_steps
        self.recorder = []                 # (total_step, avg_r, std_r, exp_r, *logging_tuple)
        self.max_r = -np.inf
        self._seed = int(seed)
        self._engine = None

    def run(self, actor_weights, critic_weights, total_step, exp_r, logging_tuple):
        """evaluator.py:48-60: returns [if_train, saved] with saved = [actor, critic, recorder] or []."""
        with torch.no_grad():
            self.agent.actor.set_weights(actor_weights)
            self.agent.critic.set_weights(critic_weights)
            saved = self.evaluate_and_save(total_step, exp_r, logging_tuple)
        return [self.total_step <= self.break_step, saved]

    def evaluate_and_save(self, new_total_step, exp_r, logging_tuple):
        self.total_step = new_total_step
        rs = self.get_rewards_and_step()
        returns, steps = rs[:, 0], rs[:, 1]
        avg_r, std_r = returns.mean().item(), returns.std().item()
        self.recorder.append((self.total_step, avg_r, std_r, exp_r, *logging_tuple))
        self.last = dict(avg_r=avg_r, std_r=std_r, avg_s=steps.mean().item(), std_s=steps.std().item())
        prev = self.max_r
        self.max_r = max(self.max_r, avg_r)
        return [self.agent.actor, self.agent.critic, self.recorder] if avg_r >= prev else []

    def get_recorder(self):
        return self.recorder

    def get_rewards_and_step(self):
        """[num_cpus_eval, 2] float32: (episode return, last step index) of independent arg-max episodes (evaluator.py:91-103),
        all of them in one batched rollout on the device."""
        cfg, B = self.cfg, self.num_cpus_eval
        if self._engine is None:
            M = B if self.pool is None else len(self.pool_indices)
            eng = BatchedPursuitEnv(cfg, B, device=self.device, num_maps=M)
            if self.pool is not None:        # env b plays held-out map b % M (the engine's initial map_id), in every evaluation
                self.pool.install(eng, self.pool_indices, verify=True)
            self._engine = eng
            self._arena = RolloutArena(self._engine.params, B, int(cfg.env.max_steps), self._engine.device)
        eng, T = self._engine, int(cfg.env.max_steps)
        self._seed += 1
        eng.reset_device(seed=self._seed, tape_len=64, maps="generate" if self.pool is None else "keep")
        self.agent.rollout_batched(eng, self._arena, T, seed=self._seed, deterministic=True, actor_only=True)
        ret = self._arena.raw_reward[:T].sum(dim=(0, 2)).to(torch.float32)
        steps = torch.full((B,), float(T - 1), dtype=torch.float32, device=ret.device)   # `done` fires at step index T-1
        return torch.stack([ret, steps], dim=1).cpu()
