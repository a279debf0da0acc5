"""Batched PBN environment: E independent env instances stepped by one kernel launch.

This is the batched surface of the drop-in (SURVEY.md section 8b): the per-instance gym API
of the reference (``env.reset()`` / ``env.step(a)``, bdq_model/__init__.py:161-204) is
served by :mod:`pbn_rl_b200.gym_env` on top of this class with ``num_envs=1``; throughput
work uses it directly.  All tensors are torch CUDA tensors owned by Python; the extension
only sees raw pointers and the current CUDA stream.
"""
from __future__ import annotations

import ctypes as C
from typing import Dict, Optional, Sequence, Tuple, Union

import numpy as np
import torch

from . import _cabi
from ._cabi import NetDesc, StepArgs, check
from .attractors import AttractorSet
from .network import PBNNetwork

__all__ = ["VecPBNEnv", "survival_table", "pair_thresholds", "make_desc", "precompile", "jit_source"]


def survival_table(p: float, n_genes: int) -> np.ndarray:
    """``S[j] = floor((1-p)^j * 2^32)`` clamped to u32 -- the geometric-skip table of the
    perturbation stream (include/pbn_b200.h, "Random streams")."""
    out = np.zeros(n_genes + 1, dtype=np.uint32)
    for j in range(n_genes + 1):
        out[j] = min(int(((1.0 - p) ** j) * 4294967296.0), 0xFFFFFFFF)
    return out


def pair_thresholds(weights: np.ndarray) -> np.ndarray:
    """A x A non-negative (source, target) weights -> cumulative u32 thresholds [A*A]."""
    w = np.asarray(weights, dtype=np.float64).reshape(-1)
    if (w < 0).any() or w.sum() <= 0:
        raise ValueError("pair weights must be non-negative with a positive sum")
    cum = np.cumsum(w / w.sum())
    thr = np.minimum(np.rint(cum * 4294967296.0), 4294967295.0).astype(np.uint64).astype(np.uint32)
    last = int(np.nonzero(w)[0][-1])
    thr[last:] = 0xFFFFFFFF
    return thr


def make_desc(network: PBNNetwork, bins: int = 3, horizon: int = 20, perturb_p: float = 0.0,
              perturb_mode: str = "A", r_success: float = 5.0, r_step: float = 0.0, r_action: float = -1.0,
              seed: int = 0x5EED, device: int = 0, kernel: str = "auto", r_wrong: float = 0.0):
    """Fill a ``pbn_net_desc`` for ``network``; returns ``(desc, keepalive)`` -- the host arrays the
    descriptor points into must outlive the C call."""
    arr = network.descriptor_arrays()
    d = NetDesc()
    d.n_genes = network.n_genes
    d.n_funcs = network.n_functions
    d.func_offset = arr["func_offset"].ctypes.data
    d.func_arity = arr["func_arity"].ctypes.data
    d.func_inputs = arr["func_inputs"].ctypes.data
    d.func_lut = arr["func_lut"].ctypes.data
    d.func_cum = arr["func_cum"].ctypes.data
    d.survival = None  # computed by the library from perturb_p
    d.bins = int(bins)
    d.horizon = int(horizon)
    d.perturb_mode = _cabi.PERT_MODES[perturb_mode]
    d.perturb_p = float(perturb_p)
    d.r_success, d.r_step, d.r_action = float(r_success), float(r_step), float(r_action)
    d.r_wrong = float(r_wrong)
    d.seed = int(seed) & 0xFFFFFFFFFFFFFFFF
    d.device = int(device)
    d.kernel = _cabi.KERNEL_KINDS[kernel]
    d.n_wide = int(arr["wide_inputs"].shape[0])
    if d.n_wide:
        d.wide_inputs = arr["wide_inputs"].ctypes.data
        d.wide_lut_offset = arr["wide_lut_offset"].ctypes.data
        d.wide_lut = arr["wide_lut"].ctypes.data
    return d, arr


def precompile(network: PBNNetwork, bins: int = 3) -> None:
    """Generate + NVRTC-compile the sliced-kernel specialisations of ``network`` into the on-disk
    cubin cache (works without a GPU).  Raises PbnError if the network is not eligible."""
    d, keep = make_desc(network, bins=bins)
    check(_cabi.lib().pbn_jit_precompile(C.byref(d)))
    del keep


def jit_source(network: PBNNetwork, bins: int = 3, injected: bool = False) -> str:
    """The CUDA source generated for ``network`` (predictor functions as LOP3 trees)."""
    d, keep = make_desc(network, bins=bins)
    lib = _cabi.lib()
    n = lib.pbn_jit_source(C.byref(d), int(injected), None, 0)
    if n < 0:
        check(int(n))
    buf = C.create_string_buffer(int(n) + 1)
    lib.pbn_jit_source(C.byref(d), int(injected), buf, int(n) + 1)
    del keep
    return buf.value.decode()


def _ptr(t: Optional[torch.Tensor]) -> Optional[int]:
    return None if t is None else t.data_ptr()


class VecPBNEnv:
    """``num_envs`` PBN env instances resident on one GPU.

    Parameters mirror the reference's ``gym.make`` kwargs where they exist (``horizon``,
    train_BDQ.py:50) and expose every constant the reference tree does not pin (SURVEY.md 8c):
    ``perturb_p`` / ``perturb_mode`` (A: Shmulevich, a perturbed step skips the update; B:
    update then flip; C: per-gene), the reward constants (``r_success`` on reaching the target, ``r_step`` per
    step, ``r_action`` per flipped gene, ``r_wrong`` for ending a step in an attractor that is not the target --
    upstream gym-PBN's shape is +5 / -1 per action / -2, SURVEY.md 8c) and the Philox ``seed``.
    ``env_offset`` is the global id of env 0 (a multiple of 1024): shards of one logical batch
    on several GPUs draw exactly the randomness the single-GPU batch would.
    ``device_counter=True`` keeps the Philox step counter in device memory (incremented by each
    step launch), so steps captured in a CUDA graph keep advancing their random streams on
    every replay.  ``pdl=True`` (implies ``device_counter``) launches the steps with programmatic
    dependent launch: each step draws its state-independent selection planes under the tail of the
    previous kernel; the device counter is then advanced explicitly with :meth:`advance_counter`
    at the end of a captured sequence instead of by every launch.
    ``chain=True`` (needs ``resident``; implies ``pdl``) additionally chains the steps of a sequence tile by tile
    (``PBN_STEP_CHAIN``): a step's tile waits only for the same tile of the previous step, so consecutive steps
    overlap on the device.  Only for open-loop sequences: the action buffers of all steps of a sequence must be
    complete before its first step is enqueued, and nothing else may be enqueued between its steps.
    ``resident=True`` (sliced kernel) keeps the env state on the device as bit-planes between steps
    (``pbn_resident_import`` / ``pbn_step`` with ``args.resident``): the fastest form of :meth:`step`.
    ``state`` / ``target_id`` / ``t`` stay available as row-format tensors -- reading them exports the
    planes, and the next step imports them again, so touch them at the boundary, not per step;
    :meth:`step` then returns ``None`` in place of the state words.  Results are bit-identical to
    ``resident=False``.
    """

    def __init__(self, network: PBNNetwork, num_envs: int, attractors: Optional[AttractorSet] = None,
                 device: Union[str, torch.device, int] = "cuda:0", seed: int = 0x5EED, horizon: int = 20,
                 bins: int = 3, perturb_p: float = 0.0, perturb_mode: str = "A", r_success: float = 5.0,
                 r_step: float = 0.0, r_action: float = -1.0, kernel: str = "auto", env_offset: int = 0,
                 auto_reset: bool = False, pair_weights: Optional[np.ndarray] = None,
                 device_counter: bool = False, pdl: bool = False, resident: bool = False, chain: bool = False,
                 r_wrong: float = 0.0):
        self._h = None
        self.lib = _cabi.lib()  # raises if the CUDA extension is not built: no fallback
        if not torch.cuda.is_available():
            raise RuntimeError("pbn_rl_b200 needs a CUDA device (B200, sm_100a); there is no CPU path")
        self.device = torch.device(device if not isinstance(device, int) else "cuda:%d" % device)
        if self.device.type != "cuda":
            raise ValueError("device must be a CUDA device")
        if self.device.index is None:
            self.device = torch.device("cuda", torch.cuda.current_device())
        self.network = network
        self.num_envs = int(num_envs)
        self.n_genes = network.n_genes
        self.n_words = network.n_words
        self.bins = int(bins)
        self.horizon = int(horizon)
        self.auto_reset = bool(auto_reset)
        self.env_offset = int(env_offset)
        self.seed = int(seed) & 0xFFFFFFFFFFFFFFFF
        self.step_ctr = 0
        self.perturb_p = float(perturb_p)
        self.perturb_mode = perturb_mode
        self.r_success, self.r_step, self.r_action = float(r_success), float(r_step), float(r_action)
        self.r_wrong = float(r_wrong)

        d, self._keep = make_desc(network, bins=self.bins, horizon=self.horizon, perturb_p=self.perturb_p,
                                  perturb_mode=perturb_mode, r_success=r_success, r_step=r_step,
                                  r_action=r_action, seed=self.seed, device=self.device.index, kernel=kernel,
                                  r_wrong=r_wrong)
        h = C.c_void_p()
        check(self.lib.pbn_create(C.byref(d), C.byref(h)))
        self._h = h
        self.kernel = {1: "scalar", 2: "sliced"}[self.lib.pbn_kernel_kind(self._h)]

        e, w = self.num_envs, self.n_words
        dev = self.device
        self._state = torch.zeros((e, w), dtype=torch.int64, device=dev)
        self._target_id = torch.full((e,), -1, dtype=torch.int32, device=dev)
        self.source_id = torch.full((e,), -1, dtype=torch.int32, device=dev)
        self._t = torch.zeros((e,), dtype=torch.int16, device=dev)  # uint16 payload
        self.resident = bool(resident)
        self._res = None            # the plane-resident block
        self._planes_fresh = False  # the block holds the current env state
        self._rows_fresh = True     # the row-format tensors hold the current env state
        if self.resident:
            if self.kernel != "sliced":
                raise ValueError("resident=True needs the sliced kernel (network not eligible: kernel=%s)" % self.kernel)
            nw = int(self.lib.pbn_resident_words(self._h, max(e, 1)))
            self._res = torch.zeros((nw,), dtype=torch.int32, device=dev)
        self.reward = torch.zeros((e,), dtype=torch.float32, device=dev)
        self.terminated = torch.zeros((e,), dtype=torch.uint8, device=dev)
        self.truncated = torch.zeros((e,), dtype=torch.uint8, device=dev)
        self.stats_buf = torch.zeros((_cabi.N_STATS,), dtype=torch.int64, device=dev)
        self.chain = bool(chain)
        if self.chain and not resident:
            raise ValueError("chain=True needs resident=True")
        pdl = bool(pdl) or self.chain
        self.pdl = bool(pdl)
        self.step_ctr_dev = torch.zeros((1,), dtype=torch.int64, device=dev) if (device_counter or pdl) else None
        self._pos = 0  # position inside a PDL sequence (host part of the step counter)
        self._reset_ctr = 0
        self.attractors: Optional[AttractorSet] = None
        self._host = None
        if attractors is not None:
            self.set_attractors(attractors, pair_weights)

    # ------------------------------------------------------------------ lifecycle
    def close(self) -> None:
        if getattr(self, "_h", None):
            self.lib.pbn_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _stream(self) -> int:
        return torch.cuda.current_stream(self.device).cuda_stream

    # ------------------------------------------------------------------ row-format view of plane-resident state
    def _rows(self) -> None:
        """Make the row-format tensors current (exports the resident block if it is newer) and treat them as
        modified by the caller: the next resident step imports them again."""
        if self.resident:
            if not self._rows_fresh:
                check(self.lib.pbn_resident_export(self._h, _ptr(self._res), _ptr(self._state), _ptr(self._target_id),
                                                   _ptr(self._t), self.num_envs, self._stream()))
                self._rows_fresh = True
            self._planes_fresh = False

    def _planes(self) -> None:
        """Make the resident block current (imports the row-format tensors if they are newer)."""
        if not self._planes_fresh:
            if self.pdl and self._pos:
                self.advance_counter()   # an import restarts the sequence: its next step is launched fully serialised
            check(self.lib.pbn_resident_import(self._h, _ptr(self._res), _ptr(self._state),
                                               _ptr(self._target_id) if self.attractors is not None else None,
                                               _ptr(self._t), self.num_envs, self._stream()))
            self._planes_fresh = True

    @property
    def state(self) -> torch.Tensor:
        self._rows()
        return self._state

    @property
    def target_id(self) -> torch.Tensor:
        self._rows()
        return self._target_id

    @property
    def t(self) -> torch.Tensor:
        self._rows()
        return self._t

    @property
    def launches(self) -> int:
        out = C.c_uint64()
        check(self.lib.pbn_launch_count(self._h, C.byref(out)))
        return out.value

    # ------------------------------------------------------------------ tables
    def set_attractors(self, attractors: AttractorSet, pair_weights: Optional[np.ndarray] = None) -> None:
        """Upload / replace the attractor table (``env.all_attractors`` may grow during
        training, bdq_model/__init__.py:182-184) and the (source, target) sampling weights
        (the curriculum of ``env.rework_probas``)."""
        if attractors.n_genes != self.n_genes:
            raise ValueError("attractor states have %d genes, network has %d" % (attractors.n_genes, self.n_genes))
        self._rows()  # the target planes of a resident block are built from the table: re-import after the change
        offs, care, val = attractors.tables()
        care = np.ascontiguousarray(care)
        val = np.ascontiguousarray(val)
        thr = None
        if pair_weights is not None:
            pw = np.asarray(pair_weights, dtype=np.float64)
            if pw.shape != (len(attractors), len(attractors)):
                raise ValueError("pair_weights must be [A, A]")
            thr = pair_thresholds(pw)
        check(self.lib.pbn_update_attractors(
            self._h, offs.ctypes.data, care.ctypes.data, val.ctypes.data, len(attractors),
            None if thr is None else thr.ctypes.data, self._stream()))
        self.attractors = attractors
        self.pair_weights = pair_weights
        if self._host is not None:
            self._host.pop("args", None)  # cached step_host arguments depend on the table's presence

    # ------------------------------------------------------------------ env API
    def reset(self, mask: Optional[torch.Tensor] = None) -> Tuple[torch.Tensor, torch.Tensor]:
        """``env.reset()`` for every instance (or those with ``mask != 0``): returns
        ``(state_words [E,W] int64, target_id [E] int32)``."""
        if mask is not None:
            mask = mask.to(device=self.device, dtype=torch.uint8).contiguous()
        if self.step_ctr_dev is None:
            ctr = self.step_ctr
            self.step_ctr += 1
        else:  # explicit resets draw from their own half of the 48-bit counter space
            ctr = (1 << 47) | self._reset_ctr
            self._reset_ctr += 1
        check(self.lib.pbn_reset(self._h, _ptr(self.state), _ptr(self.target_id), _ptr(self.source_id),
                                 _ptr(self.t), _ptr(mask), ctr, self.env_offset, self.num_envs,
                                 self._stream()))
        return self.state, self.target_id

    def _args(self, actions: Optional[torch.Tensor], final_state: Optional[torch.Tensor], stats: bool,
              rows: bool = False) -> StepArgs:
        a = StepArgs()
        a.actions = _ptr(actions)
        a.source_id = _ptr(self.source_id)
        if self.resident and final_state is None and not rows:
            self._planes()
            self._rows_fresh = False
            a.resident = _ptr(self._res)
        else:
            a.state = _ptr(self.state)
            a.target_id = _ptr(self._target_id) if self.attractors is not None else None
            a.t = _ptr(self._t)
        a.reward = _ptr(self.reward)
        a.terminated = _ptr(self.terminated)
        a.truncated = _ptr(self.truncated)
        a.final_state = _ptr(final_state)
        a.stats = _ptr(self.stats_buf) if stats else None
        a.step_ctr_dev = _ptr(self.step_ctr_dev)
        a.step_ctr = self.step_ctr
        a.env_offset = self.env_offset
        a.n_envs = self.num_envs
        a.flags = (_cabi.STEP_AUTORESET if self.auto_reset else 0) | (_cabi.STEP_PDL if self.pdl else 0)
        if self.chain and not rows and final_state is None:
            a.flags |= _cabi.STEP_CHAIN
        if self.pdl:
            a.step_ctr = self._pos
        return a

    def _check_actions(self, actions: Optional[torch.Tensor]) -> Optional[torch.Tensor]:
        if actions is None:
            return None
        if actions.dtype != torch.uint8 or actions.device != self.device or not actions.is_contiguous():
            actions = actions.to(device=self.device, dtype=torch.uint8).contiguous()
        if actions.numel() != self.num_envs * self.bins:
            raise ValueError("actions must hold num_envs*bins = %d bytes" % (self.num_envs * self.bins))
        return actions

    def step(self, actions: Optional[torch.Tensor], final_state: Optional[torch.Tensor] = None,
             stats: bool = True):
        """One ``env.step`` for every instance.  ``actions``: uint8 ``[E, bins]`` with values in
        ``[0, N]`` (0 = no-op, k flips gene k-1), or ``None`` for an uncontrolled update
        (``env.step([])``).  Returns ``(state, reward, terminated, truncated)`` -- views of the
        env's own tensors, overwritten by the next call."""
        actions = self._check_actions(actions)
        a = self._args(actions, final_state, stats)
        check(self.lib.pbn_step(self._h, C.byref(a), self._stream()))
        if self.step_ctr_dev is None:
            self.step_ctr += 1
        elif self.pdl:
            self._pos += 1
        return (None if a.resident else self._state), self.reward, self.terminated, self.truncated

    def step_injected(self, actions: Optional[torch.Tensor], sel: torch.Tensor,
                      pert_mask: Optional[torch.Tensor] = None, final_state: Optional[torch.Tensor] = None,
                      stats: bool = True):
        """The same step with injected predictor choices ``sel`` (uint8 ``[E, N]``) and
        perturbation masks ``pert_mask`` (int64 ``[E, W]``): the deterministic core the parity
        tests compare bit for bit with the oracle."""
        actions = self._check_actions(actions)
        sel = sel.to(device=self.device, dtype=torch.uint8).contiguous()
        if sel.numel() != self.num_envs * self.n_genes:
            raise ValueError("sel must be [E, N]")
        if pert_mask is not None:
            pert_mask = pert_mask.to(device=self.device, dtype=torch.int64).contiguous()
            if pert_mask.numel() != self.num_envs * self.n_words:
                raise ValueError("pert_mask must be [E, W]")
        a = self._args(actions, final_state, stats)
        a.flags &= ~_cabi.STEP_CHAIN
        a.sel = _ptr(sel)
        a.pert_mask = _ptr(pert_mask)
        check(self.lib.pbn_step_injected(self._h, C.byref(a), self._stream()))
        if self.step_ctr_dev is None:
            self.step_ctr += 1
        return (None if a.resident else self._state), self.reward, self.terminated, self.truncated

    def rollout(self, n_steps: int, stats: bool = True, recorder=None, stride: int = 1) -> torch.Tensor:
        """``n_steps`` uncontrolled updates of every instance (``env.step([])`` ``n_steps`` times,
        graph_classifier/__init__.py:148) in one launch: the states stay on chip as bit-planes between the
        updates (``pbn_rollout``).  Only ``state`` changes -- bit-identical to ``n_steps`` calls of
        ``step(None)`` -- counters, targets, rewards and flags are left alone and nothing is reset.  Networks
        the sliced kernel does not take fall back to a loop of steps.

        ``recorder`` (a :class:`pbn_rl_b200.discover.StateRecorder` of this env): the states after every update
        ``s`` (``s = 1..n_steps``) with ``s % stride == 0`` are also counted into it, inside the same launch
        (``pbn_rollout_record``); the updates themselves are the same.  The step-loop fallback calls
        ``recorder.add()`` after every ``stride``-th step instead."""
        n_steps = int(n_steps)
        stride = int(stride)
        if recorder is not None:
            if stride < 1:
                raise ValueError("stride must be >= 1")
            if recorder.env is not self:
                raise ValueError("the recorder belongs to another env")
        if n_steps <= 0:
            return self.state
        if self.step_ctr_dev is not None:
            raise RuntimeError("rollout() needs the host-side step counter (device_counter=False, pdl=False)")
        if self.kernel != "sliced":
            saved = (self.t.clone(), self.target_id.clone(), self.auto_reset)
            self.auto_reset = False
            for s in range(1, n_steps + 1):
                self.step(None, stats=stats)
                if recorder is not None and s % stride == 0:
                    recorder.add()
            self.t.copy_(saved[0])
            self.target_id.copy_(saved[1])
            self.auto_reset = saved[2]
            return self.state
        st = _ptr(self.stats_buf) if stats else None
        if recorder is None:
            check(self.lib.pbn_rollout(self._h, _ptr(self.state), n_steps, self.step_ctr, self.env_offset, self.num_envs,
                                       st, self._stream()))
        else:
            check(self.lib.pbn_rollout_record(self._h, _ptr(self.state), n_steps, self.step_ctr, self.env_offset,
                                              self.num_envs, stride, recorder._proj_ptr, recorder.k,
                                              _ptr(recorder.gene_on), _ptr(recorder.hist), st, self._stream()))
            recorder.n += self.num_envs * (n_steps // stride)
        self.step_ctr += n_steps
        return self.state

    def advance_counter(self) -> None:
        """Close a sequence of ``pdl`` steps: add the number of steps taken since the last call to the
        device step counter (one tiny serialised launch) and restart the host-side positions.  When the
        sequence is captured in a CUDA graph, capture this call as its last node."""
        if not self.pdl:
            return
        check(self.lib.pbn_advance_counter(self._h, _ptr(self.step_ctr_dev), self._pos, self._stream()))
        self._pos = 0

    # ------------------------------------------------------------------ host-buffer path (end-to-end API)
    def _host_buffers(self) -> Dict[str, torch.Tensor]:
        if self._host is None:
            e, w = self.num_envs, self.n_words
            pin = dict(pin_memory=True)
            self._host = {
                "actions": torch.empty((e, self.bins), dtype=torch.uint8, **pin),
                "state": torch.empty((e, w), dtype=torch.int64, **pin),
                "reward": torch.empty((e,), dtype=torch.float32, **pin),
                "terminated": torch.empty((e,), dtype=torch.uint8, **pin),
                "truncated": torch.empty((e,), dtype=torch.uint8, **pin),
                "d_actions": torch.empty((e, self.bins), dtype=torch.uint8, device=self.device),
            }
        return self._host

    def pinned_actions(self) -> torch.Tensor:
        """A page-locked uint8 ``[E, bins]`` host tensor: actions written here (or into any other pinned
        tensor of that shape) go to the device without an intermediate host copy in :meth:`step_host`."""
        return torch.empty((self.num_envs, self.bins), dtype=torch.uint8, pin_memory=True)

    def reward_table(self) -> np.ndarray:
        """fp32 ``[2, bins + 1]``: ``reward = table[terminated, n_flips]`` with ``n_flips`` the number of distinct action
        values in ``1..N`` of the env -- exactly the values :meth:`step` writes (``pbn_reward_table``).  Lets a host
        caller of ``step_host(compact="packed")`` derive rewards without moving them over PCIe."""
        out = np.zeros(2 * (self.bins + 1), dtype=np.float32)
        check(self.lib.pbn_reward_table(self._h, out.ctypes.data, out.size))
        return out.reshape(2, self.bins + 1)

    def pinned_actions16(self) -> torch.Tensor:
        """A page-locked int16 ``[E]`` host tensor for packed actions ``a0 | a1 << 5 | a2 << 10`` (bins = 3, N <= 30)."""
        return torch.empty((self.num_envs,), dtype=torch.int16, pin_memory=True)

    @staticmethod
    def pack_actions16(actions) -> np.ndarray:
        """uint8 ``[E, 3]`` actions -> the packed 16-bit form ``step_host`` takes as ``actions16``."""
        a = np.asarray(actions, dtype=np.uint16).reshape(-1, 3)
        return (a[:, 0] | (a[:, 1] << 5) | (a[:, 2] << 10)).astype(np.uint16)

    def step_host(self, actions_host, chunks: int = 0, compact=False, actions16=None) -> Dict[str, np.ndarray]:
        """``step`` with HOST buffers, the call a user of the reference's CPU env makes per step
        (``pbn_step_host``): uploads ``actions_host`` (uint8 ``[E, bins]``: a pinned torch tensor is used
        in place, anything else is first copied into a pinned buffer; ``None`` = no interventions), steps,
        and streams state / reward / terminated / truncated into pinned host buffers returned as
        numpy views (valid until the next call).  ``compact=True`` returns the same information in
        fewer PCIe bytes: ``state32`` (uint32, networks with N <= 32), ``reward`` and ``done``
        (``terminated | truncated << 1``); ``compact="packed"`` (N <= 30) returns one uint32 per env,
        ``packed = state | terminated << 30 | truncated << 31`` -- the reward follows from the caller's own actions and
        the terminated bit through :meth:`reward_table`.  ``actions16`` (instead of ``actions_host``): a pinned int16
        ``[E]`` tensor of packed actions (:meth:`pack_actions16`), 2 instead of 3 bytes per env.  The batch is
        cut into ``chunks`` lanes, each of which uploads, steps and downloads its slice on its own stream, so that the
        lanes' transfers and kernels overlap (0 = library default); blocks until the results are there."""
        hb = self._host_buffers()
        key = "io_packed" if compact == "packed" else ("io_compact" if compact else "io")
        if key not in hb:
            io = _cabi.HostIO()
            io.actions_dev = hb["d_actions"].data_ptr()
            if compact == "packed":
                if self.n_genes > 30:
                    raise ValueError("packed host results need N <= 30")
                hb["packed"] = torch.empty((self.num_envs,), dtype=torch.int32, pin_memory=True)
                io.packed = hb["packed"].data_ptr()
                hb["views_packed"] = {"packed": hb["packed"].numpy().view(np.uint32)}
            elif compact:
                io.reward = hb["reward"].data_ptr()
                if self.n_genes > 32:
                    raise ValueError("compact host results need N <= 32 (state32)")
                hb["state32"] = torch.empty((self.num_envs,), dtype=torch.int32, pin_memory=True)
                hb["done"] = torch.empty((self.num_envs,), dtype=torch.uint8, pin_memory=True)
                io.state32 = hb["state32"].data_ptr()
                io.done = hb["done"].data_ptr()
                hb["views_compact"] = {"state32": hb["state32"].numpy().view(np.uint32), "reward": hb["reward"].numpy(),
                                       "done": hb["done"].numpy()}
            else:
                io.reward = hb["reward"].data_ptr()
                io.state = hb["state"].data_ptr()
                io.terminated = hb["terminated"].data_ptr()
                io.truncated = hb["truncated"].data_ptr()
                hb["views"] = {k: hb[k].numpy() for k in ("state", "reward", "terminated", "truncated")}
            hb[key] = io
        io = hb[key]
        io.actions, io.actions16 = None, None
        if actions16 is not None:
            # (the checks cost a driver query per call -- is_pinned -- so a buffer that passed them is remembered)
            if hb.get("a16_checked") is not actions16:
                if not (isinstance(actions16, torch.Tensor) and actions16.is_pinned() and actions16.dtype == torch.int16
                        and actions16.is_contiguous() and actions16.numel() == self.num_envs):
                    raise ValueError("actions16 must be a pinned contiguous int16 tensor with one entry per env")
                hb["a16_checked"] = actions16
            if "d_actions16" not in hb:
                hb["d_actions16"] = torch.empty((self.num_envs,), dtype=torch.int16, device=self.device)
            io.actions16 = actions16.data_ptr()
            io.actions16_dev = hb["d_actions16"].data_ptr()
        elif actions_host is None:
            pass
        elif isinstance(actions_host, torch.Tensor) and actions_host.is_pinned() and actions_host.dtype == torch.uint8 \
                and actions_host.is_contiguous() and actions_host.numel() == self.num_envs * self.bins:
            io.actions = actions_host.data_ptr()
        else:
            src = hb["actions"]
            src.numpy()[...] = np.asarray(actions_host, dtype=np.uint8).reshape(self.num_envs, self.bins)
            io.actions = src.data_ptr()
        io.n_chunks = int(chunks)
        self._rows()  # the host-buffer path works on the row-format tensors
        a = hb.get("args")
        if a is None:
            a = hb["args"] = self._args(None, None, True, rows=True)
            # with a device counter the library advances it after the step, so the arguments stay the same from call
            # to call (the packed form replays them as one captured graph)
            a.flags &= ~_cabi.STEP_PDL
        if self._pos:
            self.advance_counter()   # close the PDL sequence: the device counter then holds the whole count
        a.step_ctr = self.step_ctr
        check(self.lib.pbn_step_host(self._h, C.byref(a), C.byref(io), self._stream()))
        if self.step_ctr_dev is None:
            self.step_ctr += 1
        return hb["views_packed" if compact == "packed" else ("views_compact" if compact else "views")]

    @property
    def host_bytes_per_step(self) -> Tuple[int, int]:
        """(host->device, device->host) bytes moved by one :meth:`step_host`."""
        e = self.num_envs
        return e * self.bins, e * (8 * self.n_words + 4 + 1 + 1)

    @property
    def host_bytes_per_step_packed(self) -> Tuple[int, int]:
        """The same for ``step_host(actions16=..., compact="packed")``: 2 bytes up, one uint32 down per env."""
        e = self.num_envs
        return e * 2, e * 4

    @property
    def host_bytes_per_step_compact(self) -> Tuple[int, int]:
        """The same for ``step_host(..., compact=True)``: uint32 state + fp32 reward + done byte."""
        e = self.num_envs
        return e * self.bins, e * (4 + 4 + 1)

    # ------------------------------------------------------------------ state access
    def set_state(self, state: Union[torch.Tensor, np.ndarray], packed: Optional[bool] = None) -> None:
        """``env.graph.setState`` for all instances: ``[E, N]`` 0/1 values or packed ``[E, W]`` words."""
        st = torch.as_tensor(state)
        if packed is None:
            packed = st.dtype in (torch.int64, torch.uint64) and st.shape[-1] == self.n_words and self.n_genes != self.n_words
        if packed:
            self.state.copy_(st.to(torch.int64).reshape(self.num_envs, self.n_words))
        else:
            bits = st.to(device=self.device, dtype=torch.uint8).reshape(self.num_envs, self.n_genes).contiguous()
            check(self.lib.pbn_pack(self._h, _ptr(bits), _ptr(self.state), self.num_envs, self._stream()))

    def set_target(self, target_id: Union[int, torch.Tensor, np.ndarray]) -> None:
        if isinstance(target_id, int):
            self.target_id.fill_(target_id)
        else:
            self.target_id.copy_(torch.as_tensor(target_id).to(torch.int32).reshape(self.num_envs))

    def unpack(self, words: Optional[torch.Tensor] = None, dtype: torch.dtype = torch.uint8) -> torch.Tensor:
        """Packed words -> ``[E, N]`` uint8 or float32 (the agent's input layer, bdq_model/__init__.py:92)."""
        words = self.state if words is None else words.to(device=self.device, dtype=torch.int64).contiguous()
        e = words.shape[0]
        out = torch.empty((e, self.n_genes), dtype=dtype, device=self.device)
        kind = {torch.uint8: _cabi.UNPACK_U8, torch.float32: _cabi.UNPACK_F32}[dtype]
        check(self.lib.pbn_unpack(self._h, _ptr(words), _ptr(out), kind, e, self._stream()))
        return out

    def observe(self, out: Optional[torch.Tensor] = None) -> torch.Tensor:
        """The agent's network input for all instances in one kernel: float32 ``[2, E, N]`` =
        (state bits, bits of the target attractor's first state with ``'*'`` -> 0) -- what
        ``predict`` builds per instance with ``np.stack((state, target))`` (bdq_model/__init__.py:92-93)."""
        if out is None:
            out = torch.empty((2, self.num_envs, self.n_genes), dtype=torch.float32, device=self.device)
        check(self.lib.pbn_observe(self._h, _ptr(self.state), _ptr(self.target_id) if self.attractors is not None else None,
                                   _ptr(out), self.num_envs, self._stream()))
        return out

    def attractor_ids(self, words: Optional[torch.Tensor] = None) -> torch.Tensor:
        """Index of the attractor containing each state (-1: none): ``is_attracting_state`` /
        ``state_attractor_id`` of the reference env."""
        if self.attractors is None:
            raise RuntimeError("no attractor table")
        words = self.state if words is None else words.to(device=self.device, dtype=torch.int64).contiguous()
        e = words.shape[0]
        out = torch.empty((e,), dtype=torch.int32, device=self.device)
        check(self.lib.pbn_attractor_id(self._h, _ptr(words), _ptr(out), e, self._stream()))
        return out

    def stats(self, reset: bool = False) -> Dict[str, int]:
        """Episode statistics accumulated on the device since the last reset of the counters."""
        vals = self.stats_buf.cpu().tolist()
        if reset:
            self.stats_buf.zero_()
        return dict(zip(_cabi.STAT_NAMES[:7], vals[:7]))
