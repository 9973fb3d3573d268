"""``ShardedDroneEnv`` -- S independent ``BatchedDroneEnv`` shards of ONE GPU stepped as a single stream of
launches, with the launch path that reaches the HBM roofline built in: CUDA graphs over parallel chains.

Why shards.  One ``DroneGame.step`` for 1 M envs is a ~24 us launch that streams 153 MB.  Two things keep a plain
loop of such launches off the roofline: (a) the host cost of a launch (a Python call per step races the GPU), and
(b) the fill / drain of every launch when each one depends on the previous (same buffers).  Environments are
independent (``DroneGame`` instances share nothing, game_engine.py:14-57), so a GPU's envs can be cut into S shards
whose steps need no mutual ordering: shard s runs on chain ``s % chains``; kernels of different chains overlap, which
hides the drain of one launch behind the fill of the next, and consecutive launches of a schedule are captured once
into a CUDA graph and replayed, which removes the per-launch host cost.  This replaces the reference's per-step loop
over its game instances (/root/reference/delivery_drone/socket_server.py:115-124; Actor_Critic_PPO.ipynb
c16:L42-108), for both kinds of caller:

  * ``step_all(actions)`` -- policy in the loop: the caller writes this step's packed actions for every shard into
    the static buffer ``self.actions [S, N]`` (or passes them) and all S shards advance one step: S launches on the
    chains, one graph replay.
  * ``run(k)`` -- actions from a device-resident trace (BASELINE.json configs[1] "fixed action trace", configs[2]
    "synthetic random actions"): launch j of the env's life (``self.t`` counts them) steps shard ``j % S`` with trace
    row ``(j // S) % L``.  The schedule has period ``S * L`` launches; a call's k launches are one piece (or pieces of
    one period each), a piece is identified by (offset in the period, length) and replays cached graphs -- one per
    chain -- so ANY k, 20 or 12,000, runs from graphs, and the result is bit-identical to stepping the shards eagerly
    in that order (tested).  ``run`` / ``step_all`` return as soon as the work is enqueued on the env's own chain
    streams; ``join()`` orders the caller's stream behind it.

``env_kw`` goes to every shard's ``BatchedDroneEnv`` (``obs_dtype=torch.bfloat16``, ``param_sets=[...]`` etc.): the
observation format and the parameter-set pointers are part of each shard's resolved step launch, so the graphs replay
them like any other argument.

Global env ids are contiguous over the shards (``env_id_base + s * N + i``), so a ShardedDroneEnv of S x N envs is the
same set of trajectories as one BatchedDroneEnv of S * N envs (Philox is keyed by the global id).
"""
from __future__ import annotations

from collections import OrderedDict
from typing import Dict, List, Optional

import torch

from . import _native as nv
from .env import BatchedDroneEnv


def schedule_pieces(t: int, k: int, num_shards: int, trace_len: int):
    """The trace schedule as plain integers: launches t .. t+k-1 of an env's life, cut into pieces of at most one
    period (S * L launches).  Yields ``(offset_in_period, length, [(shard, trace_row), ...])`` per piece; launch j
    steps shard ``j % S`` with trace row ``(j // S) % L``.  (offset, length) identifies a piece: its job list
    depends on nothing else, which is what makes the graph cache of ``ShardedDroneEnv.run`` exact."""
    S, L = int(num_shards), int(trace_len)
    period = S * L
    t, k = int(t), int(k)
    while k > 0:
        off = t % period
        seg = min(k, period)
        yield off, seg, [((off + j) % S, ((off + j) // S) % L) for j in range(seg)]
        t += seg
        k -= seg


class ShardedDroneEnv:
    def __init__(self, num_shards: int, envs_per_shard: int, device="cuda", chains: int = 2, trace_len: int = 16,
                 use_graphs: bool = True, max_graphs: int = 256, env_id_base: int = 0, launch_flags: int = nv.LAUNCH_PDL,
                 **env_kw):
        if num_shards < 1 or chains < 1 or trace_len < 1:
            raise ValueError("num_shards, chains and trace_len must be >= 1")
        self.device = torch.device(device)
        if self.device.type != "cuda":
            raise ValueError("ShardedDroneEnv runs on a CUDA device only (there is no CPU fallback)")
        if self.device.index is None:
            self.device = torch.device("cuda", torch.cuda.current_device())
        self.S, self.N, self.L = int(num_shards), int(envs_per_shard), int(trace_len)
        self.C = max(1, min(int(chains), self.S))
        self.use_graphs = bool(use_graphs)
        self.max_graphs = int(max_graphs)
        self.shards: List[BatchedDroneEnv] = [
            BatchedDroneEnv(self.N, device=self.device, env_id_base=int(env_id_base) + s * self.N,
                            launch_flags=launch_flags, **env_kw) for s in range(self.S)]
        self.num_envs = self.S * self.N
        self.t = 0                                              # launches so far (the position in the trace schedule)
        self.trace: Optional[torch.Tensor] = None               # uint8 [L, S, N]
        self.actions = torch.zeros(self.S, self.N, dtype=torch.uint8, device=self.device)   # static input of step_all
        self._chains = [torch.cuda.Stream(self.device) for _ in range(self.C)]
        self._graphs: "OrderedDict[tuple, list]" = OrderedDict()   # piece key -> one CUDAGraph (or None) per chain
        self.graph_replays = 0
        self.eager_launches = 0
        self._dirty = False                                     # chain streams hold work the caller's stream has not joined

    # ---- set-up -------------------------------------------------------------------------------------------
    def reset(self, want_obs: bool = True) -> None:
        self.join()
        for e in self.shards:
            e.reset(want_obs=want_obs)
        self.t = 0

    def set_trace(self, trace: torch.Tensor) -> None:
        """``trace``: uint8 [L, S, N] packed actions (DD_ACT_* bits) on this device; row (j // S) % L of shard j % S is
        what launch j of ``run`` reads.  Replaces the trace and drops the graphs captured over the old one."""
        if trace.dtype != torch.uint8 or tuple(trace.shape) != (self.L, self.S, self.N) or trace.device != self.device:
            raise ValueError(f"trace must be a uint8 tensor of shape {(self.L, self.S, self.N)} on {self.device}")
        self.join()
        self.trace = trace.contiguous()
        self._drop_graphs("run")

    def random_trace(self) -> torch.Tensor:
        """Fill the trace with the synthetic random policy (p = 0.5 per thruster, examples/random_agent.py:27-31): the
        same Philox bits ``rollout(policy='random')`` draws in-kernel for steps 0 .. L-1 of every env."""
        tr = torch.empty(self.L, self.S, self.N, dtype=torch.uint8, device=self.device)
        for s, e in enumerate(self.shards):
            tr[:, s].copy_(e.random_actions(self.L, t0=0))
        self.set_trace(tr)
        return tr

    # ---- the launch schedule -------------------------------------------------------------------------------
    # Shard s lives on chain stream s % C for its whole life, so each shard's launches are stream-ordered whatever
    # piece / graph they come from.  A piece of the schedule is ONE CUDA GRAPH PER CHAIN (that chain's launches of the
    # piece, back to back, programmatic dependent launch between them); the chains are never joined to each other --
    # only to the caller's stream: forked from it when a piece is enqueued (cheap: an event), joined back by join().
    # A join per piece would drain both chains at every graph boundary: ~1 us per step at 20-launch pieces (measured).
    def _fork(self) -> None:
        cur = torch.cuda.current_stream(self.device)
        for ch in self._chains:
            ch.wait_stream(cur)
        self._dirty = True

    def join(self) -> None:
        """Make the caller's current stream wait for everything this env has enqueued on its chain streams.  Called by
        every method of this class that hands tensors back; call it yourself before touching ``shards[s]`` buffers
        (``.obs``, ``.reward`` ...) or calling ``shards[s]`` methods directly after ``run`` / ``step_all``."""
        if self._dirty:
            cur = torch.cuda.current_stream(self.device)
            for ch in self._chains:
                cur.wait_stream(ch)
            self._dirty = False

    def _emit_chain(self, c: int, jobs, want_obs: bool) -> None:
        """Enqueue chain c's part of ``jobs`` = [(shard, actions uint8[N]) ...] on the CURRENT stream, in order."""
        for s, act in jobs:
            if s % self.C == c:
                self.shards[s].step_raw(act, want_obs=want_obs)

    def _play(self, key: tuple, make_jobs, want_obs: bool) -> None:
        """``make_jobs()`` builds the job list; it is only called when the piece is not in the graph cache."""
        self._fork()
        if not self.use_graphs:
            jobs = make_jobs()
            for c in range(self.C):
                with torch.cuda.stream(self._chains[c]):
                    self._emit_chain(c, jobs, want_obs)
            self.eager_launches += len(jobs)
            return
        gs = self._graphs.get(key)
        if gs is None:
            gs = self._capture(make_jobs(), want_obs)
            self._graphs[key] = gs
            while len(self._graphs) > self.max_graphs:
                self._retire(self._graphs.popitem(last=False)[1])
        else:
            self._graphs.move_to_end(key)
        for c, g in enumerate(gs):
            if g is not None:
                with torch.cuda.stream(self._chains[c]):
                    g.replay()
                self.graph_replays += 1

    def _capture(self, jobs, want_obs: bool):
        for s in {s for s, _ in jobs}:                      # resolve the step plans outside the capture
            e = self.shards[s]
            if e._needs_reset:
                raise RuntimeError("call reset() before stepping")
            if (want_obs, True) not in e._plans:
                e._make_plan(want_obs, True)
        gs = []
        for c in range(self.C):
            if not any(s % self.C == c for s, _ in jobs):
                gs.append(None)
                continue
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g, stream=self._chains[c]):
                self._emit_chain(c, jobs, want_obs)
            gs.append(g)
        return gs

    def _retire(self, graphs) -> None:
        """A captured graph may still be executing: wait for the chains before its executable is destroyed (rare path)."""
        for ch in self._chains:
            ch.synchronize()
        del graphs

    def _drop_graphs(self, kind: Optional[str] = None) -> None:
        keys = [k for k in self._graphs if kind is None or k[0] == kind]
        if keys:
            for ch in self._chains:
                ch.synchronize()
        for k in keys:
            del self._graphs[k]

    # ---- stepping ---------------------------------------------------------------------------------------------
    def run(self, k: int, want_obs: bool = True) -> None:
        """Advance the trace schedule by ``k`` launches (see the module docstring)."""
        if self.trace is None:
            raise RuntimeError("call set_trace() / random_trace() before run()")
        for off, seg, jobs in schedule_pieces(self.t, k, self.S, self.L):   # a piece may wrap around the period
            self._play(("run", off, seg, want_obs), lambda: [(s, self.trace[row, s]) for s, row in jobs], want_obs)
            self.t += seg

    def step_all(self, actions: Optional[torch.Tensor] = None, want_obs: bool = True):
        """One step of EVERY shard.  ``actions``: uint8 [S, N] packed actions, copied into the static buffer
        ``self.actions`` (or write that buffer yourself and pass None).  Returns the lists of per-shard output
        tensors ``(obs, reward, step_flags)`` (the shards' own buffers, overwritten by the next step)."""
        if actions is not None:
            if tuple(actions.shape) != (self.S, self.N) or actions.dtype != torch.uint8:
                raise ValueError(f"actions must be uint8 of shape {(self.S, self.N)}")
            self.actions.copy_(actions, non_blocking=True)
        self._play(("all", want_obs), lambda: [(s, self.actions[s]) for s in range(self.S)], want_obs)
        self.join()
        return ([e.obs for e in self.shards], [e.reward for e in self.shards], [e.step_flags for e in self.shards])

    @property
    def max_steps(self) -> int:
        return self.shards[0].max_steps

    @max_steps.setter
    def max_steps(self, v: Optional[int]) -> None:
        """Curriculum knob for every shard; the captured graphs embed the old value and are dropped."""
        self.join()
        for e in self.shards:
            e.max_steps = v
        self._drop_graphs()

    @property
    def params(self) -> "nv.DDParams":
        """A copy of the physics parameters of the shards (``BatchedDroneEnv.params``)."""
        return self.shards[0].params

    @params.setter
    def params(self, p: "nv.DDParams") -> None:
        """New physics parameters for every shard; the captured graphs embed the old constants and are dropped.  Set
        them here, not on one shard: the graphs of this class would keep replaying a shard's old launches."""
        self.join()
        for e in self.shards:
            e.params = p
        self._drop_graphs()

    def set_param_sets(self, sets, index: Optional[torch.Tensor] = None, resample: bool = False) -> None:
        """Per-env parameter sets for every shard (``BatchedDroneEnv.set_param_sets``); ``index``: ``[S, N]`` (None:
        env i of each shard runs under set ``i % len(sets)``).  The captured graphs are dropped.  Afterwards in-place
        edits of ``shards[s].param_index`` reach the graphs as they are (they hold its pointer; ``join()`` first)."""
        if index is not None and tuple(index.shape) != (self.S, self.N):
            raise ValueError(f"index must have shape {(self.S, self.N)}")
        self.join()
        for s, e in enumerate(self.shards):
            e.set_param_sets(sets, None if index is None else index[s], resample)
        self._drop_graphs()

    # ---- statistics / state -------------------------------------------------------------------------------------
    def stats_tensor(self) -> torch.Tensor:
        self.join()
        out = self.shards[0].stats_tensor().clone()
        for e in self.shards[1:]:
            out += e.stats_tensor()
        return out

    def reset_stats(self) -> None:
        self.join()
        for e in self.shards:
            e.reset_stats()

    def stats(self, reduce: bool = False) -> Dict[str, float]:
        from .distributed import allreduce_stats, stats_dict
        w = self.stats_tensor()
        if reduce:
            w = allreduce_stats(w)
        return stats_dict(w)

    @property
    def graphs_cached(self) -> int:
        return len(self._graphs)
