"""ctypes binding of libmpcb200.so (include/mpcb200.h).

This is the only way the package computes an MPC solve: there is NO CPU fallback.
If the shared library is missing it is built with nvcc (diplomjourney_b200.build);
if that is impossible, or no CUDA device is present, a RuntimeError is raised.
"""
from __future__ import annotations

import ctypes as C
import math
import operator
import os

import numpy as np

from . import build as _build

MODE_FULL, MODE_HELD = 0, 1
COST_MM, COST_TREE = 0, 1
ALGO_AUTO, ALGO_LEAFWALK, ALGO_PREFIX = 0, 1, 2
FLAG_SLOW = 1
FLAG_SKIP = 2
MAX_H = 8

_ERR = {-1: "invalid argument", -2: "CUDA error", -3: "no grid set", -4: "empty control grid",
        -5: "tree too large", -6: "no CUDA device", -7: "NCCL error"}


class MpcbError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__(f"libmpcb200: {_ERR.get(code, code)}: {msg}")
        self.code = code


class Stats(C.Structure):
    _fields_ = [("units", C.c_int64), ("leaves_per_solve", C.c_int64), ("segments", C.c_int64),
                ("refine_segments", C.c_int64), ("refine_candidates", C.c_int64), ("pruned_units", C.c_int64),
                ("algo", C.c_int32), ("kernel_launches", C.c_int32), ("stage2_units", C.c_int64)]


class LoopParams(C.Structure):
    """mpcb_loop_params (include/mpcb200.h)."""
    _fields_ = [("L", C.c_double), ("delta_t", C.c_double), ("delta_v", C.c_double), ("delta_beta", C.c_double),
                ("v_max", C.c_double), ("v_min", C.c_double), ("beta_limit", C.c_double), ("half_v", C.c_double),
                ("half_beta", C.c_double), ("eps", C.c_double), ("n_v", C.c_int32), ("n_beta", C.c_int32),
                ("cost_kind", C.c_int32), ("H", C.c_int32), ("max_ticks", C.c_int32), ("reserved", C.c_int32)]

    @classmethod
    def from_config(cls, cfg, cost_kind=COST_TREE, H=3, max_ticks=512):
        """Window constants computed exactly as math_model_tree.py:239-256 computes them."""
        half_v = (cfg.v_acc_max * cfg.delta_t) / cfg.delta_v
        half_b = (math.degrees(cfg.beta_acc_max) * cfg.delta_t) / math.degrees(cfg.delta_beta)
        return cls(L=cfg.L, delta_t=cfg.delta_t, delta_v=cfg.delta_v, delta_beta=cfg.delta_beta, v_max=cfg.v_max,
                   v_min=cfg.v_min, beta_limit=cfg.beta_max + math.radians(cfg.eps_beta), half_v=half_v,
                   half_beta=half_b, eps=cfg.eps, n_v=1 + 2 * int(half_v), n_beta=1 + 2 * int(half_b),
                   cost_kind=cost_kind, H=H, max_ticks=max_ticks, reserved=0)


LOOP_ON_TARGET, LOOP_STALLED, LOOP_MAX_TICKS, LOOP_NO_LEAF = 0, 1, 2, 3
LOOP_RUNNING = -1


class HeldCtrl(C.Structure):
    """mpcb_held_ctrl (include/mpcb200.h): one robot's online controller between two steps, in device memory."""
    _fields_ = [("pose", C.c_double * 5), ("line", C.c_double * 4), ("threshold", C.c_double), ("prev", C.c_double * 2),
                ("opt", C.c_double * (3 * MAX_H)), ("command", C.c_double * 2), ("slow_steps", C.c_int32), ("m", C.c_int32),
                ("ticks", C.c_int32), ("status", C.c_int32), ("recursive", C.c_int32), ("have_traj", C.c_int32),
                ("pending", C.c_int32), ("reserved", C.c_int32)]


class LoopEvent(C.Structure):
    """mpcb_loop_event (include/mpcb200.h): one operator event of a closed-loop script."""
    _fields_ = [("tick", C.c_int32), ("kind", C.c_int32), ("a", C.c_double), ("b", C.c_double)]


EVENT_NEW_TARGET, EVENT_TURN_LEFT, EVENT_TURN_RIGHT = 1, 2, 3


class LoopTrace(C.Structure):
    """mpcb_loop_trace (include/mpcb200.h): where the next closed-loop call writes its per-tick trace."""
    _fields_ = [("pred", C.c_void_p), ("control", C.c_void_p), ("cost", C.c_void_p)]

_lib = None
_dp, _i64p, _u8p, _fp = C.POINTER(C.c_double), C.POINTER(C.c_int64), C.POINTER(C.c_uint8), C.POINTER(C.c_float)


def library_path() -> str:
    return _build.LIB


def load():
    """Load (building first if needed) libmpcb200.so. Raises if it cannot be had."""
    global _lib
    if _lib is not None:
        return _lib
    path = _build.build_library()       # returns at once unless a source is newer than the library (or MPCB_LIB is set)
    lib = C.CDLL(path)
    vp = C.c_void_p
    lib.mpcb_version.restype = C.c_int
    lib.mpcb_device_count.restype = C.c_int
    lib.mpcb_create.argtypes = [C.c_int, C.POINTER(vp)]
    lib.mpcb_destroy.argtypes = [vp]
    lib.mpcb_last_error.argtypes = [vp]
    lib.mpcb_last_error.restype = C.c_char_p
    lib.mpcb_stream.argtypes = [vp]
    lib.mpcb_stream.restype = vp
    lib.mpcb_sync.argtypes = [vp]
    lib.mpcb_set_grid.argtypes = [vp, _dp, C.c_int, _dp, C.c_int, C.c_double, C.c_double, C.c_double]
    lib.mpcb_set_option.argtypes = [vp, C.c_char_p, C.c_double]
    solve = [vp, C.c_int, C.c_int, C.c_int, C.c_int64, vp, vp, vp, vp, vp, C.c_int64, C.c_int64, vp, vp, vp, vp]
    lib.mpcb_solve_batch_host.argtypes = solve
    lib.mpcb_solve_batch_device.argtypes = solve
    lib.mpcb_dump_leaves_host.argtypes = [vp, C.c_int, C.c_int, C.c_int, C.c_int, _dp, _dp, _dp, C.c_uint8,
                                          C.c_int64, C.c_int64, _fp, _dp]
    lib.mpcb_get_stats.argtypes = [vp, C.POINTER(Stats)]
    loop = [vp, C.POINTER(LoopParams), C.c_int64, vp, vp, vp, vp, vp, vp, vp, vp]
    lib.mpcb_held_closed_loop_host.argtypes = loop
    lib.mpcb_held_closed_loop_device.argtypes = loop
    lib.mpcb_held_closed_loop_events_host.argtypes = loop[:8] + [vp, C.c_int32, C.c_double] + loop[8:] + [vp]
    lib.mpcb_held_closed_loop_actual_host.argtypes = loop[:8] + [vp, C.c_int32, C.c_double, vp] + loop[8:] + [vp]
    lib.mpcb_held_closed_loop_actual_device.argtypes = lib.mpcb_held_closed_loop_actual_host.argtypes
    lib.mpcb_held_closed_loop_seeded_host.argtypes = loop[:8] + [vp, C.c_int32, C.c_double, vp, C.c_int32, vp] + loop[8:] + [vp]
    lib.mpcb_rng_seed_device.argtypes = [vp, C.c_int64, vp, C.c_int32, vp]
    lib.mpcb_held_closed_loop_pcg64_host.argtypes = lib.mpcb_held_closed_loop_actual_host.argtypes
    lib.mpcb_held_closed_loop_pcg64_device.argtypes = lib.mpcb_held_closed_loop_actual_host.argtypes
    lib.mpcb_held_closed_loop_pcg64_seeded_host.argtypes = loop[:8] + [vp, C.c_int32, C.c_double, vp, C.c_int32, C.c_int32,
                                                                       vp, C.c_int32, vp] + loop[8:] + [vp]
    lib.mpcb_pcg64_seed_device.argtypes = [vp, C.c_int64, vp, C.c_int32, C.c_int32, vp, C.c_int32, vp]
    lib.mpcb_held_tick_host.argtypes = [vp, vp, C.c_int, vp, C.c_int, C.c_double, C.c_double, C.c_double, C.c_int, C.c_int,
                                        vp, vp, vp, C.c_double, C.c_int, vp, vp, vp, vp]
    win = [vp, C.POINTER(LoopParams), C.c_int64, vp, vp, vp, vp, vp, vp, vp, vp, vp, vp, vp]
    lib.mpcb_solve_held_windows_host.argtypes = win
    lib.mpcb_solve_held_windows_device.argtypes = win
    lib.mpcb_full_closed_loop_host.argtypes = [vp, C.c_int, C.c_int, C.c_int64, vp, vp, vp, vp, C.c_double, C.c_int, vp, vp, vp]
    lib.mpcb_full_closed_loop_device.argtypes = lib.mpcb_full_closed_loop_host.argtypes
    lib.mpcb_set_loop_trace.argtypes = [vp, C.POINTER(LoopTrace)]
    lib.mpcb_held_ctrl_init_device.argtypes = [vp, C.POINTER(LoopParams), C.c_int64, vp, vp, vp, vp, vp, vp]
    lib.mpcb_held_ctrl_step_device.argtypes = [vp, C.POINTER(LoopParams), C.c_int64, vp, vp, vp, C.c_int32, C.c_double,
                                               vp, vp]
    split = [vp, vp, C.c_int, C.c_int, C.c_int64, vp, vp, vp, vp, vp, vp, vp, vp]
    lib.mpcb_solve_tree_split_host.argtypes = split
    lib.mpcb_solve_tree_split_device.argtypes = split
    lib.mpcb_allreduce_min.argtypes = [vp, vp, vp, vp]
    lib.mpcb_nccl_unique_id.argtypes = [vp]
    lib.mpcb_nccl_comm_create.argtypes = [vp, C.c_int, C.c_int, vp, C.POINTER(vp)]
    lib.mpcb_nccl_comm_destroy.argtypes = [vp]
    _lib = lib
    return lib


def _arr(a, dtype, shape=None):
    a = np.ascontiguousarray(a, dtype=dtype)
    if shape is not None:
        a = a.reshape(shape)
    return a


def _ptr(a):
    return None if a is None else a.ctypes.data_as(C.c_void_p)


MAX_KEY_LEN = 4096
_SEED_RANGE = "Seed must be between 0 and 2**32 - 1"


def seed_keys(seeds, n):
    """numpy's legacy seeds of ``n`` generators in the form mpcb_rng_seed_device takes them.  ``seeds`` [n] holds one
    integer seed per generator, as RandomState(seeds[i]); [n][K] holds one key of K words per generator, as
    RandomState(list(seeds[i])) -- also for K == 1 (numpy squeezes a one-element *array* to an integer seed, but
    RandomState(5) and RandomState([5]) are different streams, and here the shape decides).  Returns
    (uint32 array, key_len), key_len = 0 for integer seeds.  Raises numpy's errors for what RandomState would refuse."""
    try:
        a = np.asarray(seeds)
    except ValueError:
        raise ValueError("seeds must be [N] integer seeds or [N][K] keys of one length K") from None
    if a.ndim not in (1, 2):
        raise ValueError(f"seeds must be [N] integer seeds or [N][K] keys (each key 1-d), got shape {a.shape}")
    if a.shape[0] != n:
        raise ValueError(f"seeds holds {a.shape[0]} rows for {n} robots")
    if a.ndim == 2 and a.shape[1] == 0 and n:
        raise ValueError("Seed must be non-empty")
    if a.ndim == 2 and a.shape[1] > MAX_KEY_LEN:
        raise ValueError(f"keys of {a.shape[1]} words: at most {MAX_KEY_LEN} per generator")
    if a.size and a.dtype == object:
        try:
            vals = [operator.index(x) for x in a.ravel()]
        except TypeError:
            raise TypeError("seeds must be integers") from None
        if any(v < 0 or v > 0xFFFFFFFF for v in vals):
            raise ValueError(_SEED_RANGE)
        a = np.array(vals, np.int64).reshape(a.shape)
    elif a.size and a.dtype.kind not in "iu":
        raise TypeError(f"seeds must be integers, not {a.dtype}")
    if a.size and (a.min() < 0 or a.max() > 0xFFFFFFFF):
        raise ValueError(_SEED_RANGE)
    return np.ascontiguousarray(a, dtype=np.uint32), (a.shape[1] if a.ndim == 2 else 0)


PCG64_WORDS = 6
_U64 = (1 << 64) - 1


def pcg64_record(bit_generator):
    """[6] uint64 record of a numpy PCG64 bit generator (or of its ``.state`` dict) in the form the PCG64 entries take
    it: state >> 64, state mod 2^64, inc >> 64, inc mod 2^64, has_uint32, uinteger."""
    st = bit_generator if isinstance(bit_generator, dict) else bit_generator.state
    if st.get("bit_generator") != "PCG64":
        raise TypeError(f"not a PCG64 state: {st.get('bit_generator')!r}")
    s, inc = int(st["state"]["state"]), int(st["state"]["inc"])
    return np.array([s >> 64, s & _U64, inc >> 64, inc & _U64, int(st["has_uint32"]), int(st["uinteger"])], np.uint64)


def pcg64_state(record):
    """numpy's PCG64 ``state`` dict of one [6] record (the inverse of ``pcg64_record``)."""
    r = [int(x) for x in record]
    return {"bit_generator": "PCG64", "state": {"state": (r[0] << 64) | r[1], "inc": (r[2] << 64) | r[3]},
            "has_uint32": r[4], "uinteger": r[5]}


def _words(x):
    """SeedSequence's 32-bit little-endian words of a non-negative integer (0 -> one word) or of a sequence of them."""
    if not isinstance(x, (int, np.integer)):
        out = []
        for v in x:
            out += _words(v)
        return out
    x = operator.index(x)
    if x < 0:
        raise ValueError("expected non-negative integer")
    w = []
    while True:
        w.append(x & 0xFFFFFFFF)
        x >>= 32
        if not x:
            return w


def pcg64_seed_words(seeds, n):
    """The seeds of ``n`` Generator(PCG64) streams in the form mpcb_pcg64_seed_device takes them: returns (entropy
    uint32, entropy_stride, spawn uint32 [n][K] or None).

    * ``seeds`` an ``np.random.SeedSequence``: robot i gets ``default_rng(seeds.spawn(n)[i])`` -- the shared entropy
      (stride 0) and per robot the spawn key ``seeds.spawn_key + (seeds.n_children_spawned + i,)``.  ``seeds`` is not
      advanced here.
    * ``seeds`` [n] non-negative integers: robot i gets ``default_rng(seeds[i])`` -- one entropy row per robot.

    Raises what numpy raises for a negative integer, refuses a pool_size other than 4 and integer rows whose word counts
    cannot share one stride (integers of different lengths above 2^128)."""
    if isinstance(seeds, np.random.SeedSequence):
        if seeds.pool_size != 4:
            raise ValueError(f"SeedSequence pool_size {seeds.pool_size}: the PCG64 seeding works with pool_size 4")
        ent = _words(seeds.entropy)
        base = _words(seeds.spawn_key)
        first = seeds.n_children_spawned
        if first + n > 2 ** 32:                 # numpy counts children in 32 bits
            raise ValueError(f"{first} + {n} children: more than 2^32 spawned from one SeedSequence")
        if len(ent) > MAX_KEY_LEN or len(base) + 1 > MAX_KEY_LEN:
            raise ValueError(f"more than {MAX_KEY_LEN} seed words")
        keys = np.empty((n, len(base) + 1), np.uint32)
        keys[:, :-1] = base
        keys[:, -1] = np.arange(first, first + n, dtype=np.uint64)
        return np.array(ent, np.uint32), 0, (keys if n else None)
    if isinstance(seeds, np.random.Generator) or isinstance(seeds, np.random.BitGenerator):
        raise TypeError("seeds must be a SeedSequence or integer seeds, not a generator")
    a = list(seeds)
    if len(a) != n:
        raise ValueError(f"seeds holds {len(a)} rows for {n} robots")
    try:
        rows = [_words(operator.index(s)) for s in a]
    except TypeError:
        raise TypeError("seeds must be integers or a SeedSequence") from None
    E = max([4] + [len(r) for r in rows])
    if E > 4 and any(len(r) != E for r in rows):
        raise ValueError("integer seeds above 2^128 must all have the same number of 32-bit words")
    if E > MAX_KEY_LEN:
        raise ValueError(f"more than {MAX_KEY_LEN} seed words")
    ent = np.zeros((n, E), np.uint32)     # zero words up to the pool size do not change the stream
    for i, r in enumerate(rows):
        ent[i, :len(r)] = r
    return ent, E, None


def _event_script(events):
    """(mpcb_loop_event array or None, count) of a script [(tick, kind, a, b), ...]."""
    if not events:
        return None, 0
    ev = (LoopEvent * len(events))()
    for i, (tick, kind, a, b) in enumerate(events):
        ev[i] = LoopEvent(int(tick), int(kind), float(a), float(b))
    return ev, len(events)


class Solver:
    """One device, one stream, one control grid at a time (mpcb_handle)."""

    def __init__(self, device: int = 0):
        self.lib = load()
        h = C.c_void_p()
        rc = self.lib.mpcb_create(int(device), C.byref(h))
        if rc != 0:
            raise MpcbError(rc, "mpcb_create failed (a CUDA device is required; there is no CPU fallback)")
        self.h = h
        self.device = int(device)
        self.S = 0
        self.grid = None
        self._owner = None
        self._tick = None

    def close(self):
        if getattr(self, "h", None):
            self.lib.mpcb_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _ck(self, rc):
        if rc != 0:
            raise MpcbError(rc, (self.lib.mpcb_last_error(self.h) or b"").decode())

    # ---- configuration
    def set_grid(self, vector_v, vector_beta, L, delta_t, v_min=0.0):
        v = _arr(vector_v, np.float64).ravel()
        b = _arr(vector_beta, np.float64).ravel()
        self._ck(self.lib.mpcb_set_grid(self.h, v.ctypes.data_as(_dp), v.size, b.ctypes.data_as(_dp), b.size,
                                        float(L), float(delta_t), float(v_min)))
        self.S = v.size * b.size
        self.grid = (v, b, float(L), float(delta_t), float(v_min))
        self._owner = None      # whoever cached "my grid is set on this solver" must set it again

    def set_option(self, name: str, value: float):
        self._ck(self.lib.mpcb_set_option(self.h, name.encode(), float(value)))

    @property
    def stream(self) -> int:
        return int(self.lib.mpcb_stream(self.h) or 0)

    def sync(self):
        self._ck(self.lib.mpcb_sync(self.h))

    def set_loop_trace(self, pred=0, control=0, cost=0):
        """mpcb_set_loop_trace: the NEXT closed-loop call on this solver writes its per-tick trace to these addresses --
        pred [N][max_ticks][H][3], control [N][max_ticks][2], cost [N][max_ticks] float64, each 0 = not wanted; host
        memory for the host entries, device memory (e.g. torch.Tensor.data_ptr()) for the device ones.  That call
        consumes the trace whether it succeeds or fails; all three 0 clears it."""
        self._ck(self.lib.mpcb_set_loop_trace(self.h, C.byref(LoopTrace(int(pred) or None, int(control) or None,
                                                                         int(cost) or None))))

    def _host_trace(self, N, max_ticks, H):
        """Arrays for a host entry's trace, attached to the next call (immediately before it: nothing may raise
        between this and the call, or the trace would outlive the arrays)."""
        tr = dict(pred=np.full((N, max_ticks, H, 3), np.nan), control=np.full((N, max_ticks, 2), np.nan),
                  cost=np.full((N, max_ticks), np.nan))
        self.set_loop_trace(*(tr[k].ctypes.data for k in ("pred", "control", "cost")))
        return tr

    def stats(self) -> dict:
        s = Stats()
        self._ck(self.lib.mpcb_get_stats(self.h, C.byref(s)))
        return {k: getattr(s, k) for k, _ in Stats._fields_}

    # ---- solves
    def solve(self, mode, cost, H, state, target, origin, threshold=None, flags=None, i0_range=None):
        """Host-buffer batch solve (mpcb_solve_batch_host). Arrays: state[N,3], target[N,2], origin[N,2]."""
        st = _arr(state, np.float64)
        st = st.reshape(-1, st.shape[-1])[:, :3].copy() if st.ndim > 1 else st[:3].reshape(1, 3).copy()
        N = st.shape[0]
        tg = _arr(target, np.float64, (-1, 2))
        og = _arr(origin, np.float64, (-1, 2))
        if tg.shape[0] == 1 and N > 1:
            tg = np.repeat(tg, N, 0)
        if og.shape[0] == 1 and N > 1:
            og = np.repeat(og, N, 0)
        if tg.shape[0] != N or og.shape[0] != N:
            raise ValueError("state/target/origin batch sizes differ")
        thr = None if threshold is None else _arr(np.broadcast_to(np.asarray(threshold, np.float64), (N,)), np.float64)
        fl = None if flags is None else _arr(np.broadcast_to(np.asarray(flags, np.uint8), (N,)), np.uint8)
        lo, hi = (0, -1) if i0_range is None else (int(i0_range[0]), int(i0_range[1]))
        cost_o = np.empty(N, np.float64)
        idx_o = np.empty(N, np.int64)
        traj_o = np.empty((N, H, 3), np.float64)
        ctl_o = np.empty((N, 2), np.float64)
        self._ck(self.lib.mpcb_solve_batch_host(self.h, mode, cost, H, N, _ptr(st), _ptr(tg), _ptr(og), _ptr(thr),
                                                _ptr(fl), lo, hi, _ptr(cost_o), _ptr(idx_o), _ptr(traj_o), _ptr(ctl_o)))
        return dict(cost=cost_o, index=idx_o, traj=traj_o, first_control=ctl_o)

    def solve_device(self, mode, cost, H, N, state, target, origin, threshold, flags, out_cost, out_index,
                     out_traj, out_ctl, i0_range=None):
        """Device-pointer batch solve (mpcb_solve_batch_device); arguments are raw device addresses
        (e.g. torch.Tensor.data_ptr()) or 0/None. Enqueues on self.stream, does not synchronise."""
        lo, hi = (0, -1) if i0_range is None else (int(i0_range[0]), int(i0_range[1]))
        vp = lambda x: C.c_void_p(int(x)) if x else None
        self._ck(self.lib.mpcb_solve_batch_device(self.h, mode, cost, H, int(N), vp(state), vp(target), vp(origin),
                                                  vp(threshold), vp(flags), lo, hi, vp(out_cost), vp(out_index),
                                                  vp(out_traj), vp(out_ctl)))

    def solve_tree_split(self, comm: "NcclComm", cost, H, state, target, origin, threshold=None):
        """ONE FULL tree per solve shared by the ranks of ``comm`` (mpcb_solve_tree_split_host): collective call,
        every rank passes the same arguments and gets the whole tree's result (global leaf indices)."""
        st = _arr(state, np.float64)
        st = st.reshape(-1, st.shape[-1])[:, :3].copy() if st.ndim > 1 else st[:3].reshape(1, 3).copy()
        N = st.shape[0]
        tg = _arr(np.broadcast_to(_arr(target, np.float64, (-1, 2)), (N, 2)), np.float64)
        og = _arr(np.broadcast_to(_arr(origin, np.float64, (-1, 2)), (N, 2)), np.float64)
        thr = None if threshold is None else _arr(np.broadcast_to(np.asarray(threshold, np.float64), (N,)), np.float64)
        cost_o, idx_o = np.empty(N, np.float64), np.empty(N, np.int64)
        traj_o, ctl_o = np.empty((N, H, 3), np.float64), np.empty((N, 2), np.float64)
        self._ck(self.lib.mpcb_solve_tree_split_host(self.h, comm.comm, cost, H, N, _ptr(st), _ptr(tg), _ptr(og),
                                                     _ptr(thr), _ptr(cost_o), _ptr(idx_o), _ptr(traj_o), _ptr(ctl_o)))
        return dict(cost=cost_o, index=idx_o, traj=traj_o, first_control=ctl_o)

    def solve_tree_split_device(self, comm: "NcclComm", cost, H, N, state, target, origin, threshold, out_cost,
                                out_index, out_traj, out_ctl):
        """Device-pointer flavour (mpcb_solve_tree_split_device): enqueues the solve of this rank's share, the
        16-byte all-gather and the finalisation on self.stream; does not synchronise."""
        vp = lambda x: C.c_void_p(int(x)) if x else None
        self._ck(self.lib.mpcb_solve_tree_split_device(self.h, comm.comm, cost, H, int(N), vp(state), vp(target),
                                                       vp(origin), vp(threshold), vp(out_cost), vp(out_index),
                                                       vp(out_traj), vp(out_ctl)))

    def held_tick(self, vector_v, vector_beta, L, delta_t, v_min, cost, H, state, target, origin, threshold=math.inf,
                  flags=0):
        """One online tick in one call (mpcb_held_tick_host): the control window lists of this tick and ONE HELD
        solve.  The lean path of math_model_tree.predictive_control: preallocated buffers, no per-call numpy work
        beyond turning the two window lists into arrays.  Returns (cost, index, traj[H,3], (v, beta))."""
        buf = self._tick
        if buf is None or buf["H"] != H:
            buf = self._tick = dict(H=H, inp=np.empty(7), cost=np.empty(1), index=np.empty(1, np.int64),
                                    traj=np.empty((H, 3)), ctl=np.empty(2))
            buf["ptr"] = tuple(C.c_void_p(buf[k].ctypes.data) for k in ("cost", "index", "traj", "ctl"))
            base = buf["inp"].ctypes.data
            buf["in_ptr"] = (C.c_void_p(base), C.c_void_p(base + 24), C.c_void_p(base + 40))
        v = np.asarray(vector_v, dtype=np.float64)
        b = np.asarray(vector_beta, dtype=np.float64)
        inp = buf["inp"]
        inp[0], inp[1], inp[2] = state[0], state[1], state[2]
        inp[3], inp[4] = target[0], target[1]
        inp[5], inp[6] = origin[0], origin[1]
        self._ck(self.lib.mpcb_held_tick_host(self.h, C.c_void_p(v.ctypes.data), v.size, C.c_void_p(b.ctypes.data), b.size,
                                              L, delta_t, v_min, cost, H, *buf["in_ptr"], float(threshold), int(flags),
                                              *buf["ptr"]))
        self.S = v.size * b.size
        self.grid = (v, b, float(L), float(delta_t), float(v_min))
        self._owner = None
        return float(buf["cost"][0]), int(buf["index"][0]), buf["traj"], (float(buf["ctl"][0]), float(buf["ctl"][1]))

    def solve_held_windows(self, params: "LoopParams", state, v_beta, target, origin, threshold=None, flags=None):
        """One online tick of N robots, each with its OWN acceleration window built on the device around its current
        (v, beta) (mpcb_solve_held_windows_host).  state[N,3], v_beta[N,2], target[N,2], origin[N,2].
        Returns dict(cost, index, traj, first_control, shape[N,2] = (nV, nB))."""
        st = _arr(state, np.float64)
        st = st.reshape(-1, st.shape[-1])[:, :3].copy()
        N = st.shape[0]
        vb = _arr(np.broadcast_to(_arr(v_beta, np.float64, (-1, 2)), (N, 2)), np.float64)
        tg = _arr(np.broadcast_to(_arr(target, np.float64, (-1, 2)), (N, 2)), np.float64)
        og = _arr(np.broadcast_to(_arr(origin, np.float64, (-1, 2)), (N, 2)), np.float64)
        thr = None if threshold is None else _arr(np.broadcast_to(np.asarray(threshold, np.float64), (N,)), np.float64)
        fl = None if flags is None else _arr(np.broadcast_to(np.asarray(flags, np.uint8), (N,)), np.uint8)
        H = params.H
        cost_o, idx_o = np.empty(N, np.float64), np.empty(N, np.int64)
        traj_o, ctl_o = np.empty((N, H, 3), np.float64), np.empty((N, 2), np.float64)
        shape_o = np.empty((N, 2), np.int32)
        self._ck(self.lib.mpcb_solve_held_windows_host(self.h, C.byref(params), N, _ptr(st), _ptr(vb), _ptr(tg), _ptr(og),
                                                       _ptr(thr), _ptr(fl), _ptr(cost_o), _ptr(idx_o), _ptr(traj_o),
                                                       _ptr(ctl_o), _ptr(shape_o)))
        return dict(cost=cost_o, index=idx_o, traj=traj_o, first_control=ctl_o, shape=shape_o)

    def held_closed_loop(self, params: "LoopParams", init, target, origin, first_threshold=None, slow_steps=None,
                         events=None, radius_u_turn=0.0, rng_state=None, seeds=None, return_rng_state=True,
                         pcg_state=None, pcg_seeds=None, trace=False):
        """Whole closed loops of the online controller for a batch of robots on the device
        (mpcb_held_closed_loop_host / _events_host). ``events``: an operator script [(tick, kind, a, b), ...] with kind
        EVENT_NEW_TARGET (a, b = the new target) or EVENT_TURN_LEFT / _RIGHT (a = distance), applied to every robot
        after the tick it names; ``radius_u_turn`` = L / sin(beta_max) for the turns.
        ``rng_state`` [N][625] uint32 (per robot numpy RandomState key[624] + pos): the "actual" run with actuator noise
        (mpcb_held_closed_loop_actual_host); the input is not modified.
        ``seeds`` [N] integer seeds or [N][K] keys (see ``seed_keys``): the actual run with the generators of
        RandomState(seeds[i]), seeded on the device (mpcb_held_closed_loop_seeded_host); not together with
        ``rng_state``.  ``return_rng_state=False`` leaves the seeded generators' final states on the device.
        ``pcg_state`` [N][6] uint64 (per robot numpy Generator(PCG64) state, see ``pcg64_record``): the actual run with
        numpy's Generator stream in place of RandomState's (mpcb_held_closed_loop_pcg64_host); the input is not modified.
        ``pcg_seeds`` a SeedSequence or [N] integer seeds (see ``pcg64_seed_words``): the generators of
        default_rng(pcg_seeds.spawn(N)[i]) resp. default_rng(pcg_seeds[i]), seeded on the device
        (mpcb_held_closed_loop_pcg64_seeded_host); a SeedSequence is advanced as spawn(N) advances it.
        Returns dict(log[N,max_ticks,5], ticks[N], status[N], final[N,6] = x_t, y_t, x_0, y_0, steps_for_slowing, m),
        with ``rng_state`` or ``seeds`` also the generators' states after the run (``pcg_state`` with the PCG64 ones).
        ``trace=True`` adds what every tick logs besides the 5-list (see ``mpcb_set_loop_trace``): pred[N,max_ticks,H,3]
        (the poses of optimal_trajectory), control[N,max_ticks,2] (the commanded v, beta, before actuator noise) and
        cost[N,max_ticks] (the accepted leaf's cost, NaN on a tick that accepted none); NaN after a robot's last tick."""
        if sum(x is not None for x in (rng_state, seeds, pcg_state, pcg_seeds)) > 1:
            raise ValueError("rng_state, seeds, pcg_state and pcg_seeds each give the generators: pass one of them")
        ini = _arr(init, np.float64, (-1, 5))
        N = ini.shape[0]
        tg = _arr(np.broadcast_to(np.asarray(target, np.float64).reshape(-1, 2), (N, 2)), np.float64)
        og = _arr(np.broadcast_to(np.asarray(origin, np.float64).reshape(-1, 2), (N, 2)), np.float64)
        thr = None if first_threshold is None else _arr(np.broadcast_to(np.asarray(first_threshold, np.float64), (N,)), np.float64)
        sl = None if slow_steps is None else _arr(np.broadcast_to(np.asarray(slow_steps, np.int32), (N,)), np.int32)
        log = np.full((N, params.max_ticks, 5), np.nan)
        ticks = np.empty(N, np.int32)
        status = np.empty(N, np.int32)
        ev, n_ev = _event_script(events)
        final = np.empty((N, 6))
        tr = {}
        arm = (lambda: tr.update(self._host_trace(N, params.max_ticks, params.H))) if trace else (lambda: None)
        if pcg_seeds is not None or pcg_state is not None:
            common = (self.h, C.byref(params), N, _ptr(ini), _ptr(tg), _ptr(og), _ptr(thr), _ptr(sl), ev, n_ev,
                      float(radius_u_turn))
            if pcg_seeds is not None:
                ent, stride, spawn = pcg64_seed_words(pcg_seeds, N)
                ps = np.empty((N, PCG64_WORDS), np.uint64) if return_rng_state else None
                arm()
                self._ck(self.lib.mpcb_held_closed_loop_pcg64_seeded_host(
                    *common, _ptr(ent), ent.shape[-1], stride, _ptr(spawn), 0 if spawn is None else spawn.shape[1],
                    _ptr(ps), _ptr(log), _ptr(ticks), _ptr(status), _ptr(final)))
                if isinstance(pcg_seeds, np.random.SeedSequence):
                    pcg_seeds.spawn(N)                  # the children robots 0..N-1 drew from are now spawned
            else:
                ps = np.array(pcg_state, dtype=np.uint64, order="C")        # a copy: the library updates it in place
                if ps.shape != (N, PCG64_WORDS):
                    raise ValueError(f"pcg_state must be [N][6] = [{N}][6] (see pcg64_record), got {ps.shape}")
                arm()
                self._ck(self.lib.mpcb_held_closed_loop_pcg64_host(*common, _ptr(ps), _ptr(log), _ptr(ticks),
                                                                   _ptr(status), _ptr(final)))
            out = dict(log=log, ticks=ticks, status=status, final=final, **tr)
            if ps is not None:
                out["pcg_state"] = ps
            return out
        if seeds is not None:
            keys, key_len = seed_keys(seeds, N)
            rs = np.empty((N, 625), np.uint32) if return_rng_state else None
            arm()
            self._ck(self.lib.mpcb_held_closed_loop_seeded_host(self.h, C.byref(params), N, _ptr(ini), _ptr(tg), _ptr(og),
                                                                _ptr(thr), _ptr(sl), ev, n_ev, float(radius_u_turn),
                                                                _ptr(keys), key_len, _ptr(rs), _ptr(log), _ptr(ticks),
                                                                _ptr(status), _ptr(final)))
            out = dict(log=log, ticks=ticks, status=status, final=final, **tr)
            if return_rng_state:
                out["rng_state"] = rs
            return out
        if rng_state is None:
            arm()
            self._ck(self.lib.mpcb_held_closed_loop_events_host(self.h, C.byref(params), N, _ptr(ini), _ptr(tg), _ptr(og),
                                                                _ptr(thr), _ptr(sl), ev, n_ev, float(radius_u_turn),
                                                                _ptr(log), _ptr(ticks), _ptr(status), _ptr(final)))
            return dict(log=log, ticks=ticks, status=status, final=final, **tr)
        rs = np.array(rng_state, dtype=np.uint32, order="C")         # a copy: the library updates it in place
        if rs.shape != (N, 625):
            raise ValueError(f"rng_state must be [N][625] = [{N}][625] (key[624] + pos per robot), got {rs.shape}")
        arm()
        self._ck(self.lib.mpcb_held_closed_loop_actual_host(self.h, C.byref(params), N, _ptr(ini), _ptr(tg), _ptr(og),
                                                            _ptr(thr), _ptr(sl), ev, n_ev, float(radius_u_turn),
                                                            _ptr(rs), _ptr(log), _ptr(ticks), _ptr(status), _ptr(final)))
        return dict(log=log, ticks=ticks, status=status, final=final, rng_state=rs, **tr)

    def seed_generators_device(self, N, keys, key_len, out):
        """mpcb_rng_seed_device: the [N][625] records (key[624] + pos) of RandomState(keys[n]) (key_len == 0, keys[N]
        uint32) or RandomState(keys[n, :]) (keys[N][key_len] uint32), written to ``out``.  Raw device addresses (e.g.
        torch.Tensor.data_ptr()); enqueues on self.stream, does not synchronise."""
        vp = lambda x: C.c_void_p(int(x)) if x else None
        self._ck(self.lib.mpcb_rng_seed_device(self.h, int(N), vp(keys), int(key_len), vp(out)))

    def held_closed_loop_device_actual(self, params: "LoopParams", N, init, target, origin, first_threshold, slow_steps,
                                       rng_state, out_log, out_ticks, out_status, out_final=None, events=None,
                                       radius_u_turn=0.0, trace=None):
        """mpcb_held_closed_loop_actual_device: the actual run of ``held_closed_loop`` on raw device addresses (init
        [N][5], target / origin [N][2] float64, first_threshold [N] float64 or 0, slow_steps [N] int32 or 0, rng_state
        [N][625] uint32 updated in place, out_log [N][max_ticks][5], out_ticks / out_status [N] int32, out_final [N][6]
        or 0); ``events`` is a host script as for ``held_closed_loop``.  Rows of out_log after a robot's last tick are
        not written: fill it (with NaN, as the host entry does) beforehand.  ``trace``: (pred, control, cost) device
        addresses as for ``set_loop_trace`` (0 = not wanted), rows after a robot's last tick not written either.
        Enqueues on self.stream, does not synchronise."""
        vp = lambda x: C.c_void_p(int(x)) if x else None
        ev, n_ev = _event_script(events)
        if trace is not None:
            self.set_loop_trace(*trace)
        self._ck(self.lib.mpcb_held_closed_loop_actual_device(self.h, C.byref(params), int(N), vp(init), vp(target),
                                                              vp(origin), vp(first_threshold), vp(slow_steps), ev, n_ev,
                                                              float(radius_u_turn), vp(rng_state), vp(out_log),
                                                              vp(out_ticks), vp(out_status), vp(out_final)))

    def seed_pcg64_device(self, N, entropy, entropy_len, entropy_stride, spawn, spawn_len, out):
        """mpcb_pcg64_seed_device: the [N][6] uint64 records of default_rng(SeedSequence(entropy words, spawn-key
        words)) written to ``out`` -- entropy [entropy_len] shared (stride 0) or [N][entropy_len] (stride entropy_len),
        spawn [N][spawn_len] or 0 (uint32 words, see ``pcg64_seed_words``).  Raw device addresses; enqueues on
        self.stream, does not synchronise."""
        vp = lambda x: C.c_void_p(int(x)) if x else None
        self._ck(self.lib.mpcb_pcg64_seed_device(self.h, int(N), vp(entropy), int(entropy_len), int(entropy_stride),
                                                 vp(spawn), int(spawn_len), vp(out)))

    def held_closed_loop_device_pcg64(self, params: "LoopParams", N, init, target, origin, first_threshold, slow_steps,
                                      pcg_state, out_log, out_ticks, out_status, out_final=None, events=None,
                                      radius_u_turn=0.0, trace=None):
        """mpcb_held_closed_loop_pcg64_device: ``held_closed_loop_device_actual`` with per-robot Generator(PCG64)
        records, pcg_state [N][6] uint64 updated in place (raw device addresses), ``trace`` likewise.  Enqueues on
        self.stream, does not synchronise."""
        vp = lambda x: C.c_void_p(int(x)) if x else None
        ev, n_ev = _event_script(events)
        if trace is not None:
            self.set_loop_trace(*trace)
        self._ck(self.lib.mpcb_held_closed_loop_pcg64_device(self.h, C.byref(params), int(N), vp(init), vp(target),
                                                             vp(origin), vp(first_threshold), vp(slow_steps), ev, n_ev,
                                                             float(radius_u_turn), vp(pcg_state), vp(out_log),
                                                             vp(out_ticks), vp(out_status), vp(out_final)))

    def held_ctrl_init_device(self, params: "LoopParams", N, init, target, origin, first_threshold, slow_steps, ctrl):
        """mpcb_held_ctrl_init_device: sets up the [N] ``HeldCtrl`` records at ``ctrl`` as the closed loop sets up a robot
        -- init [N][5] x, y, phi, v, beta, target / origin [N][2] float64, first_threshold [N] float64 or 0 (= +inf),
        slow_steps [N] int32 or 0.  Raw device addresses (e.g. torch.Tensor.data_ptr()); enqueues on self.stream, does
        not synchronise."""
        vp = lambda x: C.c_void_p(int(x)) if x else None
        self._ck(self.lib.mpcb_held_ctrl_init_device(self.h, C.byref(params), int(N), vp(init), vp(target), vp(origin),
                                                     vp(first_threshold), vp(slow_steps), vp(ctrl)))

    def held_ctrl_step_device(self, params: "LoopParams", N, ctrl, measured=0, events=0, n_ev=0, radius_u_turn=0.0,
                              proposal=0, running=0):
        """mpcb_held_ctrl_step_device: one step of the online controller on the [N] ``HeldCtrl`` records at ``ctrl``
        (set up by ``held_ctrl_init_device`` with the same ``params``).  A robot holding a proposal commits measured[n]
        (the [N][5] applied x, y, phi, v, beta; 0 = the proposal unchanged) and then its events [N][n_ev]
        (``LoopEvent`` rows, ``tick`` ignored, kind 0 = empty slot); a running robot then writes its next proposal to
        proposal [N][5] (NaN rows for the others), and ``running`` (a device int32, zeroed by the caller) receives the
        number of robots holding one.  Raw device addresses; enqueues on self.stream, does not synchronise.
        Run the plant between two steps on ``torch.cuda.ExternalStream(solver.stream)``: then the stream orders the
        plant after the step that made the proposal and before the step that commits it, and no step needs a
        synchronisation (reading ``running`` is the only one)."""
        vp = lambda x: C.c_void_p(int(x)) if x else None
        self._ck(self.lib.mpcb_held_ctrl_step_device(self.h, C.byref(params), int(N), vp(ctrl), vp(measured), vp(events),
                                                     int(n_ev), float(radius_u_turn), vp(proposal), vp(running)))

    def full_closed_loop(self, cost, H, init_state, target, origin, first_threshold=None, eps=0.001, max_ticks=256,
                         trace=False):
        """Closed loop of the FULL-tree scripts for a batch of robots (mpcb_full_closed_loop_host): one batched
        FULL solve per tick with the carried threshold; stops per robot on target / after two repeated
        positions / at max_ticks. Returns dict(log[N,max_ticks,5], ticks[N], status[N]); ``trace=True`` adds pred,
        control and cost as ``held_closed_loop`` does (a stall tick repeats the last accepted trajectory)."""
        ini = _arr(init_state, np.float64, (-1, 3))
        N = ini.shape[0]
        tg = _arr(np.broadcast_to(np.asarray(target, np.float64).reshape(-1, 2), (N, 2)), np.float64)
        og = _arr(np.broadcast_to(np.asarray(origin, np.float64).reshape(-1, 2), (N, 2)), np.float64)
        thr = None if first_threshold is None else _arr(np.broadcast_to(np.asarray(first_threshold, np.float64), (N,)), np.float64)
        log = np.empty((N, max_ticks, 5))
        ticks = np.empty(N, np.int32)
        status = np.empty(N, np.int32)
        tr = self._host_trace(N, int(max_ticks), H) if trace else {}
        self._ck(self.lib.mpcb_full_closed_loop_host(self.h, cost, H, N, _ptr(ini), _ptr(tg), _ptr(og), _ptr(thr),
                                                     float(eps), int(max_ticks), _ptr(log), _ptr(ticks), _ptr(status)))
        return dict(log=log, ticks=ticks, status=status, **tr)

    def full_closed_loop_device(self, cost, H, N, init_state, target, origin, first_threshold, eps, max_ticks, out_log,
                                out_ticks, out_status, trace=None):
        """mpcb_full_closed_loop_device: ``full_closed_loop`` on raw device addresses (e.g. torch.Tensor.data_ptr()):
        init_state [N][3], target / origin [N][2], first_threshold [N] float64 or 0 (= +inf), out_log
        [N][max_ticks][5] float64, out_ticks / out_status [N] int32.  The inputs are only read.  Rows of out_log after
        a robot's last tick are not written: fill it (with NaN, as the host entry does) beforehand.  ``trace``:
        (pred, control, cost) device addresses as for ``set_loop_trace`` (0 = not wanted), rows after a robot's last
        tick not written either.  The whole run is one graph launch on self.stream; does not synchronise."""
        vp = lambda x: C.c_void_p(int(x)) if x else None
        if trace is not None:
            self.set_loop_trace(*trace)
        self._ck(self.lib.mpcb_full_closed_loop_device(self.h, int(cost), int(H), int(N), vp(init_state), vp(target),
                                                       vp(origin), vp(first_threshold), float(eps), int(max_ticks),
                                                       vp(out_log), vp(out_ticks), vp(out_status)))

    def dump_leaves(self, mode, cost, H, state, target, origin, flags=0, algo=ALGO_LEAFWALK, leaf_begin=0, count=None):
        st = _arr(state, np.float64).ravel()[:3].copy()
        tg = _arr(target, np.float64).ravel()[:2].copy()
        og = _arr(origin, np.float64).ravel()[:2].copy()
        if count is None:
            count = (self.S if mode == MODE_HELD else self.S ** H) - leaf_begin
        xy = np.empty((count, 2), np.float32)
        cs = np.empty(count, np.float64)
        self._ck(self.lib.mpcb_dump_leaves_host(self.h, mode, cost, H, algo, st.ctypes.data_as(_dp),
                                                tg.ctypes.data_as(_dp), og.ctypes.data_as(_dp), int(flags),
                                                int(leaf_begin), int(count), xy.ctypes.data_as(_fp),
                                                cs.ctypes.data_as(_dp)))
        return xy, cs


def nccl_unique_id() -> bytes:
    """128-byte NCCL id (rank 0 creates it, the caller distributes it)."""
    buf = C.create_string_buffer(128)
    rc = load().mpcb_nccl_unique_id(buf)
    if rc != 0:
        raise MpcbError(rc, "ncclGetUniqueId failed (is libnccl.so.2 loadable?)")
    return buf.raw


class NcclComm:
    """Native NCCL communicator bound to a Solver's device (mpcb_nccl_comm_create)."""

    def __init__(self, solver: "Solver", nranks: int, rank: int, unique_id: bytes):
        self.solver = solver
        self.comm = C.c_void_p()
        rc = solver.lib.mpcb_nccl_comm_create(solver.h, nranks, rank, C.c_char_p(unique_id), C.byref(self.comm))
        if rc != 0:
            raise MpcbError(rc, "ncclCommInitRank failed")

    def allreduce_min(self, cost_ptr: int, index_ptr: int):
        """Lexicographic (cost, index) min over ranks, in place on 1-element device buffers."""
        rc = self.solver.lib.mpcb_allreduce_min(self.solver.h, self.comm, C.c_void_p(cost_ptr), C.c_void_p(index_ptr))
        if rc != 0:
            raise MpcbError(rc, "mpcb_allreduce_min failed")

    def close(self):
        if self.comm:
            self.solver.lib.mpcb_nccl_comm_destroy(self.comm)
            self.comm = None


_default = {}


def default_solver(device: int = 0) -> Solver:
    """Process-wide solver per device used by the reference-API modules."""
    s = _default.get(device)
    if s is None:
        s = _default[device] = Solver(device)
    return s
