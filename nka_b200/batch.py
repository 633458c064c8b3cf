"""Batched accelerators: `nbatch` independent NKA instances of one length in one handle.

Each member has its own subspace, list, Gram factor, vtol decisions, relax and restart, and gives bit for
bit what a single `NKA` handle in the capacity shape (INTEGRATION.md section 6) gives when fed that
member's calls.  One batched update is a fixed number of kernel launches whatever `nbatch` is.
Device-only and single-GPU: rows of f are CUDA float64 tensor rows (INTEGRATION.md section 7).
"""
from __future__ import annotations

import ctypes as C
import weakref

import numpy as np

from . import _lib
from .nka import NKAError, _is_torch

MAX_BATCH = 65535


class _Batch:
    """What BatchNKA and InterleavedBatchNKA share: the life cycle, masks, vtol and the queries, through the
    C functions <_prefix>_*."""
    _prefix = "nka_batch"
    _max_batch = MAX_BATCH
    _name = "batched accelerator"

    def __init__(self, nbatch: int | None = None, vlen: int | None = None, mvec: int | None = None,
                 vtol: float = 0.01, device: int = -1, stream: int | None = None):
        self._h = None
        self._lib = _lib.load()
        if nbatch is not None:
            self.init(nbatch, vlen, mvec, vtol=vtol, device=device, stream=stream)

    def _c(self, name: str):
        return getattr(self._lib, "%s_%s" % (self._prefix, name))

    # -- life cycle -------------------------------------------------------
    def init(self, nbatch: int, vlen: int, mvec: int, vtol: float = 0.01, device: int = -1,
             stream: int | None = None):
        """Re-initialising frees the previous storage.  Bad arguments raise ValueError before any CUDA call."""
        if nbatch is None or not 1 <= nbatch <= self._max_batch:
            raise ValueError("nbatch must be in 1..%d" % self._max_batch)
        if vlen is None or vlen < 1:
            raise ValueError("vlen must be >= 1")
        if mvec is None or mvec <= 0:
            raise ValueError("mvec must be > 0")
        if mvec > _lib.MAX_MVEC:
            raise ValueError("mvec > %d is not supported by this build" % _lib.MAX_MVEC)
        if not vtol > 0.0:
            raise ValueError("vtol must be > 0")
        self.delete()
        self._h = self._c("init")(nbatch, vlen, mvec, vtol, device, stream)
        if not self._h:
            raise NKAError("%s_init returned NULL" % self._prefix)
        self.nbatch, self.vlen, self.mvec = nbatch, vlen, mvec
        return self

    def delete(self):
        if self._h:
            self._c("delete")(self._h)
            self._h = None

    def __del__(self):
        try:
            self.delete()
        except Exception:
            pass

    def _handle(self):
        if not self._h:
            raise NKAError("%s is not initialised" % self._name)
        return self._h

    def _uncaptured(self, call: str, why: str):
        h = self._handle()
        if self._c("stream_capturing")(h) != 0:
            raise NKAError("%s cannot be captured in a CUDA graph: %s" % (call, why))
        return h

    def _mask(self, mask, what: str):
        return _mask_address(mask, self.nbatch, what)

    # -- masks and vtol ---------------------------------------------------
    def relax(self, mask=None) -> None:
        m = self._mask(mask, "mask")
        self._c("relax")(self._handle(), m)

    def restart(self, mask=None) -> None:
        m = self._mask(mask, "mask")
        self._c("restart")(self._handle(), m)

    def set_vec_tol(self, vtol: float) -> None:
        if not vtol > 0.0:
            raise ValueError("vtol must be > 0")
        self._c("set_vec_tol")(self._handle(), vtol)

    # -- queries ----------------------------------------------------------
    def num_vec(self) -> np.ndarray:
        out = np.zeros(self.nbatch, dtype=np.int32)
        self._c("num_vec")(self._uncaptured("num_vec", "it copies the device state to the host and synchronises"),
                           out.ctypes.data_as(C.POINTER(C.c_int)))
        return out

    def defined(self) -> bool:
        return bool(self._h) and bool(self._c("defined")(
            self._uncaptured("defined", "it copies the device state to the host and synchronises")))

    def state(self, b: int) -> dict:
        """Member b's state, with the keys and layout of NKA.state()."""
        if not 0 <= b < self.nbatch:
            raise ValueError("member index out of range")
        v = _lib.StateView()
        self._c("get_state")(self._uncaptured("state", "it copies the device state to the host and synchronises"),
                             b, C.byref(v))
        return _state_dict(v)

    def set_stream(self, stream: int | None):
        """The stream every later call is queued on; set the capture stream here before a capture begins."""
        self._c("set_stream")(self._uncaptured("set_stream", "it synchronises the handle's stream"), stream)

    def synchronize(self):
        self._c("synchronize")(self._uncaptured("synchronize", "it synchronises the handle's stream"))

    def stream_capturing(self) -> int:
        return self._c("stream_capturing")(self._handle())

    def launch_count(self) -> int:
        return self._c("launch_count")(self._handle())


class BatchNKA(_Batch):
    """`nbatch` accelerators sharing vlen, mvec and vtol, updated together."""

    def __init__(self, *args, **kwargs):
        self._loops = weakref.WeakSet()          # its device-side loops and queues
        super().__init__(*args, **kwargs)

    def delete(self):
        for loop in list(self._loops):
            loop.destroy()
        super().delete()

    def _rows(self, T, name: str, nrows: int | None = None, what: str = "nbatch") -> int:
        """The row stride of T, a CUDA float64 tensor [nrows, vlen] with unit column stride; nrows, named
        `what` in messages, is nbatch unless given.  Only a tensor of nbatch rows has its device checked here:
        fixed_point_queue checks its problem rows' devices itself, after slot_problem's."""
        if what == "nbatch":
            nrows = self.nbatch
        if not _is_torch(T):
            raise ValueError("%s must be a CUDA float64 tensor of shape [%s, vlen]" % (name, what))
        import torch
        if T.dtype != torch.float64 or T.dim() != 2 or tuple(T.shape) != (nrows, self.vlen):
            raise ValueError("%s must be a CUDA float64 tensor of shape [%s, vlen] = [%s, %d]"
                             % (name, what, what if nrows is None else nrows, self.vlen))
        if T.stride(1) != 1 and self.vlen > 1:
            raise ValueError("%s must have unit column stride (%s.stride(1) == 1)" % (name, name))
        ld = T.stride(0)
        if ld < self.vlen:
            if nrows > 1:
                raise ValueError("%s's row stride must be >= vlen" % name)
            ld = self.vlen                      # one row: its stride is never used to address anything
        if what == "nbatch" and not T.is_cuda:
            raise ValueError("%s must be a CUDA tensor: the batched accelerator is device-only" % name)
        return ld

    # -- the hot path -----------------------------------------------------
    def accel_update(self, F, active=None) -> None:
        """F: CUDA float64 tensor [nbatch, vlen] with unit column stride; row b is member b's f and is
        overwritten with its accelerated correction.  active: optional length-nbatch CUDA bool / uint8
        tensor; an inactive member's row and state are left exactly as they are.  Capturable."""
        ldf = self._rows(F, "F")
        a = self._mask(active, "active")
        self._lib.nka_batch_accel_update(self._handle(), F.data_ptr(), ldf, a)

    # -- device-side fixed-point loops --------------------------------------
    def fixed_point_loop(self, residual, X, F, atol=0.0, rtol=1e-8, maxit=100, dtol: float = 0.0,
                         scale=None, restart_growth: float = 0.0) -> "FixedPointLoop":
        """A solve of x_b = G(x_b) for every member that runs to its end in one graph launch
        (INTEGRATION.md section 8).  residual: a zero-argument callable writing F = G(X) - X in place with
        torch ops; it is run once to warm up, then captured.  X, F: CUDA float64 tensors [nbatch, vlen]
        with unit column stride.  With r = ||F_b|| (or ||scale_b * F_b||), a member stops when r is not
        finite (NONFINITE), when r < max(atol_b, rtol_b * r0_b) (CONVERGED, r0_b = its r at the launch's
        first check), when dtol > 0 and r > dtol * r0_b (DIVERGED), or after maxit_b steps (MAXIT).
        atol, rtol: a number >= 0 or a contiguous CUDA float64 tensor of nbatch entries; maxit: an int >= 0
        or a contiguous CUDA int32 tensor of nbatch entries (the loop's history then has max(maxit) + 1
        rows); dtol: 0 (off) or >= 1; scale: None or a CUDA float64 tensor [nbatch, vlen] with unit column
        stride, read after the residual in every iteration, so the residual may rewrite it
        (INTEGRATION.md section 9a).  restart_growth: 0 (off) or a finite number > 0; when check k >= 1
        leaves a member running with r_k > restart_growth * r_{k-1}, its accelerator is restarted before
        that iteration's update (INTEGRATION.md section 9b)."""
        return self._fixed_point("loop", residual, X, F, atol, rtol, maxit, dtol, scale, restart_growth,
                                 lambda: (self.nbatch, "nbatch", ()),
                                 lambda stop: FixedPointLoop(self, None, X, F, stop.maxit))

    def fixed_point_queue(self, residual, X, F, slot_problem, X0, Xout=None, atol=0.0, rtol=1e-8,
                          maxit=100, dtol: float = 0.0, scale=None, restart_growth: float = 0.0) -> "FixedPointQueue":
        """Solve nproblems = X0.shape[0] problems x_p = G_p(x_p) on the members as slots, in one graph launch
        (INTEGRATION.md section 9).  When a slot's problem stops, the launch writes its final iterate to
        Xout[p], loads the next problem's X0 row into the slot and restarts the slot's accelerator.
        residual: a zero-argument callable writing F = G(X) - X for every row with torch ops, reading
        slot_problem (the problem of each row, -1 for an idle row, whose F is ignored) to find each row's
        parameters; it is run once to warm up, then captured.  X, F: CUDA float64 [nbatch, vlen], the slots'
        rows.  slot_problem: contiguous CUDA int32 [nbatch], set here to the launch's first assignment
        (slot b solves problem b) and kept by the queue.  X0, Xout: CUDA float64 [nproblems, vlen] with unit
        column stride; Xout=None solves in place (Xout is X0).  The stopping rule is fixed_point_loop's,
        with tensor atol, rtol and maxit holding one entry per problem (nproblems), found through
        slot_problem; scale is per slot, [nbatch, vlen], like F.  restart_growth is fixed_point_loop's,
        applied to each problem's own norms (INTEGRATION.md section 9b)."""
        if Xout is None:
            Xout = X0
        nproblems = X0.shape[0] if _is_torch(X0) and X0.dim() == 2 else None

        def problems():
            sp_bad = "slot_problem must be a contiguous CUDA int32 tensor of length nbatch = %d" % self.nbatch
            if not _is_torch(slot_problem):
                raise ValueError(sp_bad)
            import torch
            if slot_problem.dtype != torch.int32 or slot_problem.dim() != 1 or slot_problem.numel() != self.nbatch \
                    or (self.nbatch > 1 and slot_problem.stride(0) != 1):
                raise ValueError(sp_bad)
            if nproblems is not None and not 1 <= nproblems <= 2**31 - 1:
                raise ValueError("X0 must hold 1 to 2**31 - 1 problems (rows)")
            ldx0 = self._rows(X0, "X0", nproblems, "nproblems")
            ldxout = self._rows(Xout, "Xout", nproblems, "nproblems")
            for T, name in ((slot_problem, "slot_problem"), (X0, "X0"), (Xout, "Xout")):
                if not T.is_cuda:
                    raise ValueError("%s must be a CUDA tensor: the batched accelerator is device-only" % name)
            return nproblems, "nproblems", (slot_problem.data_ptr(), X0.data_ptr(), ldx0, Xout.data_ptr(), ldxout,
                                            nproblems)

        def make(stop):
            # the launch's first assignment, set before the residual's warm-up reads it
            import torch
            ids = torch.arange(self.nbatch, dtype=torch.int32, device=slot_problem.device)
            slot_problem.copy_(torch.where(ids < nproblems, ids, torch.full_like(ids, -1)))
            return FixedPointQueue(self, None, X, F, slot_problem, X0, Xout, nproblems)

        return self._fixed_point("queue", residual, X, F, atol, rtol, maxit, dtol, scale, restart_growth, problems, make)

    def _fixed_point(self, kind: str, residual, X, F, atol, rtol, maxit, dtol, scale, restart_growth, problems, make):
        """What fixed_point_loop (kind "loop") and fixed_point_queue ("queue") share.  problems(): the solve's
        own argument checks, after the stopping rule's; it returns the entries a tensor atol, rtol or maxit
        holds, their name ("nbatch" or "nproblems") and the arguments nka_batch_<kind>_create_restart takes
        between ldf and the stop test.  make(stop): the solve, before the residual is captured into it."""
        _check_stopping(atol, rtol, maxit, dtol)
        _check_restart_growth(restart_growth)
        count, what, args = problems()
        _check_lengths(count, what, atol, rtol, maxit)
        ldscale = self._rows(scale, "scale") if scale is not None else 0
        ldx = self._rows(X, "X")
        ldf = self._rows(F, "F")
        h = self._uncaptured("fixed_point_" + kind, "it captures the residual and synchronises")
        stop = _stop_test(atol, rtol, maxit, dtol, scale, ldscale)
        solve = make(stop)
        solve._graph = _capture(residual, F.device)
        solve._stop = (atol, rtol, maxit, scale)
        solve._h = self._c(kind + "_create_restart")(h, solve._graph.raw_cuda_graph(), X.data_ptr(), ldx, F.data_ptr(),
                                                     ldf, *args, C.byref(stop), float(restart_growth))
        if not solve._h:
            raise NKAError("nka_batch_%s_create returned NULL: CUDA refused the residual graph or the driver "
                           "has no conditional graph nodes (the reason is printed on stderr)" % kind)
        self._loops.add(solve)
        return solve


def _mask_address(mask, nbatch: int, what: str):
    """The device address of a length-nbatch CUDA bool / uint8 tensor, or None for every member."""
    if mask is None:
        return None
    if not _is_torch(mask):
        raise ValueError("%s must be a CUDA bool or uint8 tensor of length nbatch" % what)
    import torch
    if mask.dtype not in (torch.bool, torch.uint8) or not mask.is_cuda or mask.dim() != 1 \
            or mask.numel() != nbatch or (nbatch > 1 and mask.stride(0) != 1):
        raise ValueError("%s must be a contiguous CUDA bool or uint8 tensor of length nbatch" % what)
    return mask.data_ptr()


def _state_dict(v: _lib.StateView) -> dict:
    """An nka_state_view as the dict NKA.state() returns."""
    n = v.mvec + 1
    return {
        "subspace": v.subspace, "pending": v.pending, "first": v.first, "last": v.last,
        "free": v.free_slot, "next": list(v.next[:n]), "prev": list(v.prev[:n]),
        "chained": list(v.chained[:n]), "ndrop_last": v.ndrop_last, "evicted_last": v.evicted_last,
        "relaxed_last": v.relaxed_last, "error": v.error, "vtol": v.vtol, "min_margin": v.min_margin,
        "s_last": v.s_last, "c": np.array(v.c[:n]), "s": np.array(v.s[:n]),
        "h": np.array(v.h[: n * n]).reshape(n, n), "ncalls": v.ncalls,
    }


def _check_stopping(atol, rtol, maxit, dtol):
    """Numbers, or tensors of the right kind (their length is _check_lengths', their entries _stop_test's)."""
    for v, name in ((atol, "atol"), (rtol, "rtol")):
        if _is_torch(v):
            import torch
            if v.dtype != torch.float64 or v.dim() != 1 or not v.is_cuda or (v.numel() > 1 and v.stride(0) != 1):
                raise ValueError("%s must be a number >= 0 or a contiguous 1-D CUDA float64 tensor" % name)
        elif isinstance(v, bool) or not isinstance(v, (int, float)) or not v >= 0.0:
            raise ValueError("%s must be a number >= 0" % name)
    if _is_torch(maxit):
        import torch
        if maxit.dtype != torch.int32 or maxit.dim() != 1 or not maxit.is_cuda or (maxit.numel() > 1 and maxit.stride(0) != 1):
            raise ValueError("maxit must be an integer >= 0 or a contiguous 1-D CUDA int32 tensor")
    elif isinstance(maxit, bool) or not isinstance(maxit, (int, np.integer)) or maxit < 0 or maxit > 2**31 - 2:
        raise ValueError("maxit must be an integer >= 0")
    if isinstance(dtol, bool) or not isinstance(dtol, (int, float)) or not (dtol == 0.0 or dtol >= 1.0):
        raise ValueError("dtol must be 0 (off) or a number >= 1")


def _check_restart_growth(restart_growth):
    if isinstance(restart_growth, bool) or not isinstance(restart_growth, (int, float, np.integer, np.floating)) \
            or not 0.0 <= restart_growth < float("inf"):
        raise ValueError("restart_growth must be 0 (off) or a finite number > 0")


def _check_lengths(count: int, what: str, *values):
    for v, name in zip(values, ("atol", "rtol", "maxit")):
        if _is_torch(v) and v.numel() != count:
            raise ValueError("%s must hold one entry per %s: %d, not %d"
                             % (name, "member" if what == "nbatch" else "problem", count, v.numel()))


def _stop_test(atol, rtol, maxit, dtol, scale, ldscale) -> _lib.StopTest:
    """The nka_stop_test of validated arguments.  Tensor entries are checked here (this synchronises): a
    tolerance entry must be >= 0 (not NaN), a maxit entry in 0..2**31 - 2, whose maximum bounds the loop."""
    stop = _lib.StopTest()
    for v, name in ((atol, "atol"), (rtol, "rtol")):
        if _is_torch(v):
            if not bool((v >= 0.0).all()):
                raise ValueError("%s entries must be >= 0 (and not NaN)" % name)
            setattr(stop, name + "_dev", v.data_ptr())
        else:
            setattr(stop, name, float(v))
    if _is_torch(maxit):
        lo, hi = int(maxit.min()), int(maxit.max())
        if lo < 0 or hi > 2**31 - 2:
            raise ValueError("maxit entries must be integers in 0..2**31 - 2")
        stop.maxit, stop.maxit_dev = hi, maxit.data_ptr()
    else:
        stop.maxit = int(maxit)
    stop.dtol = float(dtol)
    if scale is not None:
        stop.scale_dev, stop.ldscale = scale.data_ptr(), ldscale
    return stop


def _capture(residual, device):
    """residual() run once on a side stream to warm up, then captured into a kept torch CUDA graph."""
    import torch
    side = torch.cuda.Stream(device=device)
    side.wait_stream(torch.cuda.current_stream(device))
    with torch.cuda.stream(side):
        residual()
    torch.cuda.current_stream(device).wait_stream(side)
    graph = torch.cuda.CUDAGraph(keep_graph=True)
    with torch.cuda.graph(graph):
        residual()
    torch.cuda.synchronize(device)
    return graph


class _FixedPoint:
    """What FixedPointLoop and FixedPointQueue share: a device-side solve over a BatchNKA through the C
    functions nka_batch_<_kind>_*.  Keeps the captured residual graph (and its memory pool), X, F, the stop
    test's tensors and the batch alive."""
    _kind = "loop"

    def __init__(self, batch: BatchNKA, graph, X, F):
        self._h = None
        self._stop = None
        self._batch, self._graph, self._X, self._F = batch, graph, X, F
        self._lib = batch._lib

    def _count(self) -> int:
        """Entries of results() and restarts(): one per member (loop) or problem (queue)."""
        return self._batch.nbatch

    def _handle(self, call: str, why: str):
        if not self._h:
            raise NKAError("fixed-point %s is destroyed" % self._kind)
        self._batch._uncaptured(call, why)
        return self._h

    def _c(self, name: str):
        return getattr(self._lib, "nka_batch_%s_%s" % (self._kind, name))

    def run(self) -> None:
        """One graph launch on the batch's stream: the whole solve (a queue's: every problem from problem 0 and
        the current X0 rows to its end, results in Xout).  Returns at once."""
        self._c("launch")(self._handle("run", "a graph with conditional nodes cannot become a child of another graph"))

    def results(self):
        """(steps, status, norm) per member (loop) or problem (queue) as numpy arrays; status is one of RUNNING,
        CONVERGED, MAXIT, NONFINITE, DIVERGED.  Synchronises."""
        h = self._handle("results", "it copies the %s's results to the host and synchronises" % self._kind)
        n = self._count()
        it = np.zeros(n, dtype=np.int32)
        st = np.zeros(n, dtype=np.int32)
        norm = np.zeros(n, dtype=np.float64)
        self._c("results")(h, it.ctypes.data_as(C.POINTER(C.c_int)), st.ctypes.data_as(C.POINTER(C.c_int)),
                           norm.ctypes.data_as(C.POINTER(C.c_double)))
        return it, st, norm

    def restarts(self) -> np.ndarray:
        """Restarts the residual-growth rule made per member (loop) or problem (queue; the restart of a slot
        taking a problem is not counted) in the last launch (int32; zeros when restart_growth is 0).
        Synchronises."""
        h = self._handle("restarts", "it copies the %s's restart counts to the host and synchronises" % self._kind)
        out = np.zeros(self._count(), dtype=np.int32)
        self._c("restarts")(h, out.ctypes.data_as(C.POINTER(C.c_int)))
        return out

    def destroy(self) -> None:
        if self._h:
            self._c("destroy")(self._h)
            self._h = None
        self._batch._loops.discard(self)

    def __del__(self):
        try:
            self.destroy()
        except Exception:
            pass


class FixedPointLoop(_FixedPoint):
    """A device-side fixed-point loop over a BatchNKA (BatchNKA.fixed_point_loop)."""

    def __init__(self, batch: BatchNKA, graph, X, F, maxit: int):
        super().__init__(batch, graph, X, F)
        self.maxit = maxit

    def history(self) -> np.ndarray:
        """[(maxit+1), nbatch]: row k holds each member's norm at check k, NaN where it made none.  Synchronises."""
        h = self._handle("history", "it copies the loop's history to the host and synchronises")
        out = np.zeros((self.maxit + 1, self._batch.nbatch), dtype=np.float64)
        self._lib.nka_batch_loop_history(h, out.ctypes.data_as(C.POINTER(C.c_double)))
        return out


class FixedPointQueue(_FixedPoint):
    """A device-side work queue over a BatchNKA (BatchNKA.fixed_point_queue); also keeps slot_problem, X0
    and Xout alive."""
    _kind = "queue"

    def __init__(self, batch: BatchNKA, graph, X, F, slot_problem, X0, Xout, nproblems: int):
        super().__init__(batch, graph, X, F)
        self._slot_problem, self.X0, self.Xout = slot_problem, X0, Xout
        self.nproblems = nproblems

    def _count(self) -> int:
        return self.nproblems


RUNNING, CONVERGED, MAXIT, NONFINITE, DIVERGED = 0, 1, 2, 3, 4
