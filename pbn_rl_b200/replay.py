"""Device-resident replay ring for the batched env (SURVEY.md 8f-1).

The reference stores one ``Transition(state, target, action, reward, next_state, done)`` per env
step in a python list and samples with ``random.sample`` (bdq_model/memory.py:22-70); every policy
update then rebuilds float tensors from the tuples (bdq_model/__init__.py:100-109).  With 2^20 env
instances per step that path is the bottleneck, so here the transitions stay *packed* in HBM
(28 B per transition at N <= 64, bins = 3) and one gather+unpack kernel produces exactly the tensors
``update_policy`` consumes.  All device work goes through the C-ABI (``pbn_replay_*``); torch only
lends memory and draws the sample indices.
"""
from __future__ import annotations

import ctypes as C
from typing import Dict, Optional

import torch

from . import _cabi
from ._cabi import check

__all__ = ["DeviceReplay", "DevicePrioritizedReplay"]


class DeviceReplay:
    """Ring of ``capacity`` packed transitions next to a :class:`VecPBNEnv`.

    Protocol per env step (the two halves of ``memory.store``)::

        replay.observe()                 # before env.step: (state, target) of every instance
        env.step(actions, final_state=nxt)
        replay.commit(actions, nxt)      # after: (action, reward, done, next_state)

    or simply ``replay.step(actions)`` which does the three calls.
    """

    def __init__(self, env, capacity: int):
        if capacity < env.num_envs:
            raise ValueError("capacity %d < num_envs %d: one step would overwrite itself" % (capacity, env.num_envs))
        self.env = env
        self.capacity = int(capacity)
        dev, w, b = env.device, env.n_words, env.bins
        c = self.capacity
        self.state = torch.zeros((c, w), dtype=torch.int64, device=dev)
        self.next_state = torch.zeros((c, w), dtype=torch.int64, device=dev)
        self.target_id = torch.full((c,), -1, dtype=torch.int32, device=dev)
        self.actions = torch.zeros((c, b), dtype=torch.uint8, device=dev)
        self.reward = torch.zeros((c,), dtype=torch.float32, device=dev)
        self.done = torch.zeros((c,), dtype=torch.uint8, device=dev)
        self._r = _cabi.Replay()
        self._r.state, self._r.next_state = self.state.data_ptr(), self.next_state.data_ptr()
        self._r.target_id, self._r.actions = self.target_id.data_ptr(), self.actions.data_ptr()
        self._r.reward, self._r.done = self.reward.data_ptr(), self.done.data_ptr()
        self._r.capacity = c
        self.head = 0          # next slot to write
        self.size = 0          # transitions stored (<= capacity)
        self._pending = False
        self._final = torch.zeros((env.num_envs, w), dtype=torch.int64, device=dev)

    def __len__(self) -> int:
        return self.size

    @property
    def bytes_per_transition(self) -> int:
        return 16 * self.env.n_words + 4 + self.env.bins + 4 + 1

    def observe(self) -> None:
        env = self.env
        check(env.lib.pbn_replay_observe(env._h, C.byref(self._r), self.head, env.state.data_ptr(),
                                         env.target_id.data_ptr(), env.num_envs, env._stream()))
        self._pending = True

    def commit(self, actions: Optional[torch.Tensor], next_state: torch.Tensor) -> None:
        if not self._pending:
            raise RuntimeError("commit() without observe()")
        env = self.env
        actions = env._check_actions(actions)
        check(env.lib.pbn_replay_commit(env._h, C.byref(self._r), self.head,
                                        None if actions is None else actions.data_ptr(), env.reward.data_ptr(),
                                        env.terminated.data_ptr(), env.truncated.data_ptr(), next_state.data_ptr(),
                                        env.num_envs, env._stream()))
        self.head = (self.head + env.num_envs) % self.capacity
        self.size = min(self.capacity, self.size + env.num_envs)
        self._pending = False

    def step(self, actions: Optional[torch.Tensor]):
        """observe -> env.step -> commit.  Returns what ``env.step`` returns."""
        self.observe()
        actions = self.env._check_actions(actions)
        out = self.env.step(actions, final_state=self._final)
        self.commit(actions, self._final)
        return out

    def sample(self, batch_size: int, generator: Optional[torch.Generator] = None,
               index: Optional[torch.Tensor] = None) -> Dict[str, torch.Tensor]:
        """``memory.sample(batch_size)`` + the tensor building of ``update_policy``: returns
        ``obs`` [2,B,N] (states, targets), ``next_obs`` [2,B,N] (next states, targets) float32,
        ``actions`` [B,bins,1] int64, ``reward`` [B,1], ``done`` [B,1] float32 and the ``index`` used."""
        env = self.env
        if index is None:
            if self.size == 0:
                raise RuntimeError("the replay ring is empty")
            index = torch.randint(0, self.size, (batch_size,), device=env.device, generator=generator)
        index = index.to(device=env.device, dtype=torch.int64).contiguous()
        b, n = int(index.numel()), env.n_genes
        obs = torch.empty((2, b, n), dtype=torch.float32, device=env.device)
        nxt = torch.empty((2, b, n), dtype=torch.float32, device=env.device)
        act = torch.empty((b, env.bins, 1), dtype=torch.int64, device=env.device)
        rew = torch.empty((b, 1), dtype=torch.float32, device=env.device)
        done = torch.empty((b, 1), dtype=torch.float32, device=env.device)
        check(env.lib.pbn_replay_sample(env._h, C.byref(self._r), index.data_ptr(), b, obs.data_ptr(), nxt.data_ptr(),
                                        act.data_ptr(), rew.data_ptr(), done.data_ptr(), env._stream()))
        return {"obs": obs, "next_obs": nxt, "actions": act, "reward": rew, "done": done, "index": index}


class DevicePrioritizedReplay(DeviceReplay):
    """:class:`DeviceReplay` with proportional prioritised sampling (the reference's PER over a sum / min segment
    tree, SURVEY.md section 2 rows 13-14), the trees on the device next to the ring (``pbn_per_*``; contract in
    include/pbn_b200.h).

    ``commit()`` also enters the new transitions at the running maximum priority; ``sample(batch, beta)`` draws
    ``batch`` slots by stratified proportional sampling and returns the parent's tensors plus ``weight`` [B,1], the
    importance weights ``(pmin / p) ** beta`` (already divided by their maximum over the ring);
    ``update_priorities(index, td_error)`` sets ``p = (|td| + eps) ** alpha``.  Nothing synchronises the host, so
    sample -> gather -> update can be captured in a CUDA graph; ``beta`` is a host float of each call, so a captured
    graph keeps the value it was captured with (anneal it by re-capturing, or sample eagerly).
    """

    def __init__(self, env, capacity: int, alpha: float = 0.6, eps: float = 1e-6):
        super().__init__(env, capacity)
        if not eps > 0:
            raise ValueError("eps=%r must be > 0" % eps)
        if not alpha >= 0:
            raise ValueError("alpha=%r must be >= 0" % alpha)
        self.alpha, self.eps = float(alpha), float(eps)
        nf = int(env.lib.pbn_per_tree_floats(self.capacity))
        if nf < 0:
            check(nf)
        self.leaves_pow2 = nf // 5
        self.tree = torch.empty((nf,), dtype=torch.float32, device=env.device)
        self.max_p_buf = torch.empty((1,), dtype=torch.float32, device=env.device)
        self._p = _cabi.Per()
        self._p.tree, self._p.max_p = self.tree.data_ptr(), self.max_p_buf.data_ptr()
        self._p.capacity, self._p.alpha = self.capacity, self.alpha
        check(env.lib.pbn_per_init(env._h, C.byref(self._p), env._stream()))

    def commit(self, actions: Optional[torch.Tensor], next_state: torch.Tensor) -> None:
        head = self.head
        super().commit(actions, next_state)
        self.push(head, self.env.num_envs)

    def push(self, head: int, n: int) -> None:
        """Slots ``(head + e) % capacity``, ``e < n``, get priority ``max_p ** alpha`` (what ``commit()`` does after
        storing the transitions)."""
        env = self.env
        check(env.lib.pbn_per_push(env._h, C.byref(self._p), head, n, env._stream()))

    def sample(self, batch_size: int, beta: float = 0.4, generator: Optional[torch.Generator] = None,
               u: Optional[torch.Tensor] = None) -> Dict[str, torch.Tensor]:
        """``u`` ([B] float32 in [0, 1)) fixes the draw; by default ``torch.rand`` with ``generator``."""
        env = self.env
        if self.size == 0:
            raise RuntimeError("the replay ring is empty")
        if u is None:
            u = torch.rand((batch_size,), dtype=torch.float32, device=env.device, generator=generator)
        u = u.to(device=env.device, dtype=torch.float32).contiguous()
        b = int(u.numel())
        index = torch.empty((b,), dtype=torch.int64, device=env.device)
        weight = torch.empty((b, 1), dtype=torch.float32, device=env.device)
        check(env.lib.pbn_per_sample(env._h, C.byref(self._p), u.data_ptr(), b, float(beta), index.data_ptr(),
                                     weight.data_ptr(), env._stream()))
        out = super().sample(b, index=index)
        out["weight"] = weight
        return out

    def update_priorities(self, index: torch.Tensor, td_error: torch.Tensor) -> None:
        """New priorities for ring slots ``index`` from TD errors; the last occurrence of a repeated slot wins,
        indices outside ``[0, capacity)`` are ignored, NaN counts as 0 and +-inf as 1e30."""
        env = self.env
        index = index.to(device=env.device, dtype=torch.int64).contiguous()
        td = td_error.to(device=env.device, dtype=torch.float32).reshape(-1).contiguous()
        if td.numel() != index.numel():
            raise ValueError("index has %d entries, td_error %d" % (index.numel(), td.numel()))
        check(env.lib.pbn_per_update(env._h, C.byref(self._p), index.data_ptr(), td.data_ptr(), int(index.numel()),
                                     self.eps, env._stream()))

    # ---- read accessors (views of the device trees; layout in include/pbn_b200.h)
    def leaves(self) -> torch.Tensor:
        """Priorities ``p`` of the ``capacity`` slots (sum-tree leaves)."""
        L = self.leaves_pow2
        return self.tree[L:L + self.capacity]

    def levels(self):
        """``[(sum, min)]`` per binary level, leaves (all ``L`` of them) first, root last."""
        L, out = self.leaves_pow2, []
        n = L
        while n >= 1:
            out.append((self.tree[n:2 * n], self.tree[2 * L + n:2 * L + 2 * n]))
            n //= 2
        return out

    def total(self) -> float:
        return float(self.tree[1].item())

    def pmin(self) -> float:
        return float(self.tree[2 * self.leaves_pow2 + 1].item())

    def max_p(self) -> float:
        return float(self.max_p_buf.item())
