"""Python host layer: same names, argument meaning and error behaviour as the reference's
``Space2`` / ``Field2`` / ``HholtzAdi`` / ``Poisson`` / ``Navier2D`` (file:line cited per class),
calling the C ABI only.  numpy arrays cross the boundary; everything else stays on the GPU."""
from __future__ import annotations

import ctypes as C
import os

import numpy as np

from ._lib import B2Error, check, lib

# BaseKind order of src/field.rs:173-177
CHEBYSHEV, CHEB_DIRICHLET, CHEB_NEUMANN, CHEB_DIRICHLET_NEUMANN, FOURIER_R2C, FOURIER_C2C = range(6)
PHYSICAL, SPECTRAL, ORTHO = 0, 1, 2


def chebyshev(n):
    """src/bases.rs:11-19 (funspace ``chebyshev``)."""
    return (CHEBYSHEV, n)


def cheb_dirichlet(n):
    return (CHEB_DIRICHLET, n)


def cheb_neumann(n):
    return (CHEB_NEUMANN, n)


def cheb_dirichlet_neumann(n):
    return (CHEB_DIRICHLET_NEUMANN, n)


def fourier_r2c(n):
    return (FOURIER_R2C, n)


def fourier_c2c(n):
    """bases.rs:15: complex physical values, n modes in FFT order.  Not on the Navier2D path: dense-matrix transform, n <= 1024."""
    return (FOURIER_C2C, n)


def _dp(a):
    return a.ctypes.data_as(C.POINTER(C.c_double))


class Context:
    """One per GPU / rank (replaces funspace ``initialize()`` -> ``Universe``, src/mpi/mod.rs:5,12)."""

    def __init__(self, device=0, rank=0, nranks=1, heap_bytes=0):
        self._h = C.c_void_p()
        check(lib().b2_ctx_create(device, rank, nranks, heap_bytes, C.byref(self._h)))
        self.device, self.rank, self.nranks = device, rank, nranks

    def close(self):
        """Release the context (streams, events, workspaces, symmetric heap, IPC mappings).  Every object created on
        it must be gone first; contexts are not destroyed implicitly."""
        if self._h:
            check(lib().b2_ctx_destroy(self._h))
            self._h = None

    @classmethod
    def distributed(cls, device, heap_bytes):
        """One context per rank of an initialised ``torch.distributed`` group (one process per GPU).
        The ranks exchange the CUDA-IPC handle of their symmetric heap so that every pencil transpose
        is a peer store inside the producing kernel (replaces funspace ``Decomp2d::transpose_*`` /
        MPI_Alltoallv, src/field_mpi.rs:456-477)."""
        import torch.distributed as dist

        rank, world = dist.get_rank(), dist.get_world_size()
        ctx = cls(device, rank, world, heap_bytes)
        if world > 1:
            h = C.create_string_buffer(64)
            check(lib().b2_ctx_heap_handle(ctx._h, h))
            handles = [None] * world
            dist.all_gather_object(handles, bytes(h.raw))
            check(lib().b2_ctx_attach_peers(ctx._h, b"".join(handles)))
            dist.barrier()
        return ctx

    def all_reduce_sum(self, x):
        if self.nranks == 1:
            return x
        import torch
        import torch.distributed as dist

        scalar = np.ndim(x) == 0
        t = torch.tensor(np.atleast_1d(np.asarray(x, dtype=np.float64)), dtype=torch.float64)
        if dist.get_backend() == "nccl":
            t = t.cuda(self.device)
        dist.all_reduce(t)
        return float(t.item()) if scalar else t.cpu().numpy()

    def all_gather_rows(self, a):
        """Concatenate the ranks' row slabs (gather(local) == global)."""
        if self.nranks == 1:
            return a
        import torch.distributed as dist

        parts = [None] * self.nranks
        dist.all_gather_object(parts, a)
        return np.concatenate([p for p in parts if p.shape[0] > 0], axis=0)

    def barrier(self):
        check(lib().b2_ctx_barrier(self._h))

    def sync(self):
        check(lib().b2_ctx_sync(self._h))

    def timer_start(self):
        check(lib().b2_ctx_timer_start(self._h))

    def timer_stop(self):
        ms = C.c_double()
        check(lib().b2_ctx_timer_stop(self._h, C.byref(ms)))
        return ms.value

    def launch_count(self):
        n = C.c_longlong()
        check(lib().b2_ctx_launch_count(self._h, C.byref(n)))
        return n.value

    def opprof(self, on):
        """Per-op cycle counters of the lane kernel: {op name: (cycles, calls)} since the last call."""
        buf = (C.c_ulonglong * 64)()
        check(lib().b2_ctx_opprof(self._h, int(on), buf))
        names = {1: "load", 2: "store", 3: "band", 4: "deriv", 5: "fdma", 6: "dct", 7: "rfft", 8: "fdiff", 9: "scalevec",
                 10: "zerotail", 11: "lanemask", 12: "zeroelem", 13: "scale", 15: "bandc",
                 16: "fdma.fwd_reduce", 17: "fdma.scan1", 18: "fdma.fwd_apply", 19: "fdma.compose", 20: "fdma.scan2", 21: "fdma.solve",
                 22: "dct.pre", 23: "dct.fft", 24: "dct.post", 25: "st.fill", 26: "st.wait", 27: "ld.direct_first", 28: "ld.direct_later", 29: "ld.combine", 30: "ld.plain", 31: "ld.stencil"}
        return {names[c]: (buf[c], buf[32 + c]) for c in names if buf[32 + c]}

    def profile(self, on):
        """Switch GEMM timing on/off; returns the GEMM milliseconds accumulated since the last call."""
        ms = C.c_double()
        check(lib().b2_ctx_profile(self._h, int(on), C.byref(ms)))
        return ms.value


_default_ctx = None


def default_context():
    global _default_ctx
    if _default_ctx is None:
        _default_ctx = Context(0)
    return _default_ctx


class Space2:
    """funspace ``Space2::new(&base0, &base1)`` (src/field.rs:81-90)."""

    def __init__(self, base0, base1, ctx=None):
        self.ctx = ctx or default_context()
        self.bases = (base0, base1)
        self._h = C.c_void_p()
        check(lib().b2_space2_create(self.ctx._h, base0[0], base0[1], base1[0], base1[1], C.byref(self._h)))

    def close(self):
        if getattr(self, "_h", None):
            _release(lib().b2_space_destroy, self._h)
            self._h = None

    __del__ = close

    def shape(self, kind):
        r, c, cx = C.c_int(), C.c_int(), C.c_int()
        check(lib().b2_space_shape(self._h, kind, C.byref(r), C.byref(c), C.byref(cx)))
        return (r.value, c.value), bool(cx.value)

    def shape_physical(self):
        return self.shape(PHYSICAL)[0]

    def shape_spectral(self):
        return self.shape(SPECTRAL)[0]

    def base_kind(self, axis):
        return self.bases[axis][0]

    def coords(self):
        out = []
        for ax in (0, 1):
            x = np.zeros(self.bases[ax][1])
            check(lib().b2_space_coords(self._h, ax, _dp(x)))
            out.append(x)
        return out

    LAYOUT_KEYS = ("E", "LN", "TPL", "fast", "CHW", "nsc", "NT", "smem")

    def lane_layout(self, orient):
        """Diagnostic (no reference counterpart): the lane-kernel layout this space's passes run with, fixed when the space
        was created.  orient 0: lanes along axis 1, orient 1: lanes along axis 0."""
        out = (C.c_int * 8)()
        check(lib().b2_space_lane_layout(self._h, orient, out))
        return dict(zip(self.LAYOUT_KEYS, out))


def _release(fn, handle):
    """Destroy a native object from close()/__del__: never raises (interpreter shutdown, already-destroyed context)."""
    try:
        fn(handle)
    except Exception:  # noqa: BLE001
        pass


def _host_dtype(space, kind):
    return np.complex128 if space.shape(kind)[1] else np.float64


class DeviceArray:
    """A device-resident ``Array2`` in one of the three shapes of a space."""

    def __init__(self, space, kind, handle=None, owner=True):
        self.space, self.kind = space, kind
        self._owner = owner
        if handle is None:
            self._h = C.c_void_p()
            check(lib().b2_array_create(space._h, kind, C.byref(self._h)))
        else:
            self._h = handle

    def close(self):
        if getattr(self, "_h", None) and self._owner:
            _release(lib().b2_array_destroy, self._h)
        self._h = None

    __del__ = close

    def local_rows(self):
        """(first row, number of rows) of this rank's slab (axis 0 split; whole array with one rank)."""
        r0, cnt = C.c_int(), C.c_int()
        check(lib().b2_array_local_rows(self._h, C.byref(r0), C.byref(cnt)))
        return r0.value, cnt.value

    def local_shape(self):
        shape, _ = self.space.shape(self.kind)
        return (self.local_rows()[1], shape[1])

    def set(self, a):
        shape = self.local_shape()
        a = np.ascontiguousarray(a, dtype=_host_dtype(self.space, self.kind))
        if a.shape != tuple(shape):
            raise B2Error(f"shape mismatch: got {a.shape}, expected {tuple(shape)}")  # reference: panic
        if a.size:
            check(lib().b2_array_set_host(self._h, a.ctypes.data_as(C.c_void_p), a.nbytes))
        return self

    def get(self):
        out = np.empty(self.local_shape(), dtype=_host_dtype(self.space, self.kind))
        if out.size:
            check(lib().b2_array_get_host(self._h, out.ctypes.data_as(C.c_void_p), out.nbytes))
        return out

    def axpy(self, alpha, x):
        check(lib().b2_array_axpy(self._h, alpha, x._h))
        return self

    def norm(self):
        """L2 norm of the global array (functions.rs:24-35): local sum of squares, all-reduced over the ranks."""
        v = C.c_double()
        check(lib().b2_array_norm2(self._h, C.byref(v)))   # collective with several ranks (summed on the device)
        return v.value


class Field2:
    """``FieldBase`` for N = 2 (src/field.rs:59-129): ``v``, ``vhat``, ``x``, ``dx`` and
    ``forward / backward / to_ortho / from_ortho / gradient``."""

    def __init__(self, space, handle=None):
        self.space = space
        self._owner = handle is None
        if handle is None:
            self._h = C.c_void_p()
            check(lib().b2_field_create(space._h, C.byref(self._h)))
        else:
            self._h = handle
        self.x = space.coords()
        self.dx = [self._get_dx(x, space.base_kind(i) in (FOURIER_R2C, FOURIER_C2C)) for i, x in enumerate(self.x)]

    def close(self):
        if getattr(self, "_h", None) and self._owner:
            _release(lib().b2_field_destroy, self._h)
        self._h = None

    __del__ = close

    @staticmethod
    def _get_dx(x, periodic):  # src/field.rs:135-163
        if periodic:
            return np.full(len(x), x[2] - x[1])
        mid = 0.5 * (x[1:] + x[:-1])
        return np.concatenate((mid, [x[-1]])) - np.concatenate(([x[0]], mid))

    def scale(self, scale):  # src/field.rs:93-100
        for i, sc in enumerate(scale):
            self.x[i] = self.x[i] * sc
            self.dx[i] = self.dx[i] * sc

    def average_axis(self, axis):
        """``FieldBase::average_axis`` (src/field/average.rs:26-35; slabs: src/field_mpi/average.rs:15-61): dx-weighted mean of
        ``v`` along ``axis``, reduced on the device; with several ranks the partial sums (axis 0) / row parts (axis 1) are combined
        like the reference's ``all_gather_sum`` / gather.  Returns the global 1-D array on every rank."""
        if axis not in (0, 1):
            raise B2Error("average_axis: axis 0 or 1")
        arr = C.c_void_p()
        check(lib().b2_field_array(self._h, 0, C.byref(arr)))
        lo = self.local_slice(PHYSICAL)
        w0 = np.ascontiguousarray((self.dx[0] / abs(self.x[0][-1] - self.x[0][0]))[lo])
        w1 = np.ascontiguousarray(self.dx[1] / abs(self.x[1][-1] - self.x[1][0]))
        if len(w0) == 0:
            w0 = np.zeros(1)   # a rank without rows still takes part in the collective below
        ctx = self.space.ctx
        if axis == 0:
            out = np.zeros(len(w1))
            check(lib().b2_array_weighted_sum(arr, _dp(w0), _dp(w1), 1, _dp(out)))
            return ctx.all_reduce_sum(out)
        out = np.zeros(max(1, lo.stop - lo.start))
        check(lib().b2_array_weighted_sum(arr, _dp(w0), _dp(w1), 2, _dp(out)))
        return ctx.all_gather_rows(out[: lo.stop - lo.start])

    def average(self):
        """``FieldBase::average`` (src/field/average.rs:53-59): volume-weighted mean of ``v``."""
        arr = C.c_void_p()
        check(lib().b2_field_array(self._h, 0, C.byref(arr)))
        lo = self.local_slice(PHYSICAL)
        w0 = np.ascontiguousarray((self.dx[0] / abs(self.x[0][-1] - self.x[0][0]))[lo])
        w1 = np.ascontiguousarray(self.dx[1] / abs(self.x[1][-1] - self.x[1][0]))
        if len(w0) == 0:
            w0 = np.zeros(1)
        out = np.zeros(1)
        check(lib().b2_array_weighted_sum(arr, _dp(w0), _dp(w1), 0, _dp(out)))
        return float(self.space.ctx.all_reduce_sum(out)[0])

    def local_rows(self, kind):
        """(first row, count) of this rank's slab of ``v`` (PHYSICAL) or ``vhat`` (SPECTRAL): axis 0 is
        split in contiguous blocks (y-pencil of src/field_mpi.rs:71-88); one rank owns everything."""
        r0, cnt = C.c_int(), C.c_int()
        check(lib().b2_field_local_rows(self._h, kind, C.byref(r0), C.byref(cnt)))
        return r0.value, cnt.value

    def local_slice(self, kind):
        r0, cnt = self.local_rows(kind)
        return slice(r0, r0 + cnt)

    # ---- rank bookkeeping and host-side gather / scatter of the slabs (src/field_mpi.rs:309-321, 363-453) ----
    # Host conveniences for set-up, output and tests: they move whole arrays through torch.distributed object collectives and are
    # not part of the timestep (the pencil exchanges of the hot path are peer stores inside the kernels).
    def nrank(self):
        return self.space.ctx.rank

    def nprocs(self):
        return self.space.ctx.nranks

    def get_coords_local(self, axis):
        """Coordinates of this rank's part of the physical array along ``axis`` (src/field_mpi.rs:128-131): axis 0 is split."""
        return self.x[axis][self.local_slice(PHYSICAL)] if axis == 0 else self.x[axis]

    def _gather(self, local, root):
        ctx = self.space.ctx
        if ctx.nranks == 1:
            return local
        import torch.distributed as dist

        if root is None:
            return ctx.all_gather_rows(local)
        parts = [None] * ctx.nranks if ctx.rank == root else None
        dist.gather_object(local, parts, dst=root)
        return np.concatenate([p for p in parts if p.shape[0] > 0], axis=0) if ctx.rank == root else None

    def _scatter(self, glob, kind, root):
        ctx = self.space.ctx
        if ctx.nranks == 1:
            return np.asarray(glob)
        import torch.distributed as dist

        bounds = [None] * ctx.nranks
        dist.all_gather_object(bounds, self.local_rows(kind))
        parts = None
        if ctx.rank == root:
            shape, _ = self.space.shape(kind)
            glob = np.asarray(glob)
            if glob.shape != tuple(shape):
                raise B2Error(f"shape mismatch: got {glob.shape}, expected {tuple(shape)}")   # reference: panic
            parts = [np.ascontiguousarray(glob[r0:r0 + cnt]) for r0, cnt in bounds]
        out = [None]
        dist.scatter_object_list(out, parts, src=root)
        return out[0]

    def gather_physical_root(self, root=0):
        """The global physical array on ``root`` (None elsewhere), src/field_mpi.rs:391-399."""
        return self._gather(self.v, root)

    def gather_spectral_root(self, root=0):
        """The global spectral array on ``root`` (None elsewhere), src/field_mpi.rs:371-380."""
        return self._gather(self.vhat, root)

    def all_gather_physical(self):
        """The global physical array on every rank, src/field_mpi.rs:439-444."""
        return self._gather(self.v, None)

    def all_gather_spectral(self):
        """The global spectral array on every rank, src/field_mpi.rs:447-453."""
        return self._gather(self.vhat, None)

    def scatter_physical_root(self, v_global=None, root=0):
        """Distribute ``root``'s global physical array over the ranks' slabs of ``v``, src/field_mpi.rs:410-419."""
        self.v = self._scatter(v_global, PHYSICAL, root)

    def scatter_spectral_root(self, vhat_global=None, root=0):
        """Distribute ``root``'s global spectral array over the ranks' slabs of ``vhat``, src/field_mpi.rs:430-436."""
        self.vhat = self._scatter(vhat_global, SPECTRAL, root)

    # host views of the device-resident data (this rank's rows)
    @property
    def v(self):
        out = np.empty((self.local_rows(PHYSICAL)[1], self.space.shape_physical()[1]), dtype=_host_dtype(self.space, PHYSICAL))
        if out.size:
            check(lib().b2_field_get_v_host(self._h, out.ctypes.data_as(C.c_void_p), out.nbytes))
        return out

    @v.setter
    def v(self, a):
        a = np.ascontiguousarray(a, dtype=_host_dtype(self.space, PHYSICAL))   # complex only on a FourierC2c axis 0
        if a.shape != (self.local_rows(PHYSICAL)[1], self.space.shape_physical()[1]):
            raise B2Error(f"shape mismatch: got {a.shape}")
        if a.size:
            check(lib().b2_field_set_v_host(self._h, a.ctypes.data_as(C.c_void_p), a.nbytes))

    @property
    def vhat(self):
        shape, cx = self.space.shape(SPECTRAL)
        out = np.empty((self.local_rows(SPECTRAL)[1], shape[1]), dtype=np.complex128 if cx else np.float64)
        if out.size:
            check(lib().b2_field_get_vhat_host(self._h, out.ctypes.data_as(C.c_void_p), out.nbytes))
        return out

    def vhat_into(self, out):
        """Download ``vhat`` into a caller-owned C-contiguous array (e.g. a view of pinned host memory) without
        allocating: the device-to-host copy then runs at PCIe speed instead of through a pageable bounce."""
        shape, cx = self.space.shape(SPECTRAL)
        want = (self.local_rows(SPECTRAL)[1], shape[1])
        if out.shape != want or out.dtype != (np.complex128 if cx else np.float64) or not out.flags.c_contiguous:
            raise B2Error(f"vhat_into: need a C-contiguous {want} array of {'complex128' if cx else 'float64'}")
        if out.size:
            check(lib().b2_field_get_vhat_host(self._h, out.ctypes.data_as(C.c_void_p), out.nbytes))
        return out

    @vhat.setter
    def vhat(self, a):
        shape, cx = self.space.shape(SPECTRAL)
        a = np.ascontiguousarray(a, dtype=np.complex128 if cx else np.float64)
        if a.shape != (self.local_rows(SPECTRAL)[1], shape[1]):
            raise B2Error(f"shape mismatch: got {a.shape}, expected {(self.local_rows(SPECTRAL)[1], shape[1])}")
        if a.size:
            check(lib().b2_field_set_vhat_host(self._h, a.ctypes.data_as(C.c_void_p), a.nbytes))

    def forward(self):
        check(lib().b2_forward(self._h))

    def backward(self):
        check(lib().b2_backward(self._h))

    def dealias(self):
        """``dealias(&mut field)`` (src/navier_stokes/functions.rs:72-82)."""
        check(lib().b2_field_dealias(self._h))

    def to_ortho(self, out=None):
        if out is None:
            out = DeviceArray(self.space, ORTHO)
        check(lib().b2_to_ortho(self._h, out._h))
        return out

    def from_ortho(self, arr):
        check(lib().b2_from_ortho(self._h, arr._h))

    def gradient(self, deriv, scale=None, out=None):
        if out is None:
            out = DeviceArray(self.space, ORTHO)
        sc = None
        if scale is not None:
            sc = (C.c_double * 2)(float(scale[0]), float(scale[1]))
        check(lib().b2_gradient(self._h, int(deriv[0]), int(deriv[1]), sc, out._h))
        return out


class _Solver:
    def solve(self, inp, out=None, axis=0):
        """``Solve::solve(&input, &mut output, axis)`` (src/solver.rs:59-82); ``axis`` is ignored
        as in the reference's field solvers (src/solver/hholtz_adi.rs:120)."""
        if isinstance(inp, np.ndarray):
            inp = DeviceArray(self.field.space, ORTHO).set(inp)
        if out is None:
            out = DeviceArray(self.field.space, SPECTRAL)
        check(lib().b2_solve(self._h, inp._h, out._h))
        return out

    solve_par = solve

    def close(self):
        if getattr(self, "_h", None):
            _release(lib().b2_solver_destroy, self._h)
        self._h = None

    __del__ = close


class HholtzAdi(_Solver):
    """``HholtzAdi::new(&field, c)`` (src/solver/hholtz_adi.rs:48-76)."""

    def __init__(self, field, c):
        self.field = field
        self._h = C.c_void_p()
        check(lib().b2_hholtz_adi_create(field._h, float(c[0]), float(c[1]), C.byref(self._h)))


class Hholtz(_Solver):
    """``Hholtz::new(&field, c)`` (src/solver/hholtz.rs:66-101): ``(I - c D2) vhat = A f`` through the eigendecomposition
    of axis 0 (``FdmaTensor`` with alpha = 1) instead of the ADI factorisation."""

    def __init__(self, field, c):
        self.field = field
        self._h = C.c_void_p()
        kind0, n0 = field.space.bases[0]
        if kind0 in (CHEB_DIRICHLET, CHEB_NEUMANN):
            lam, fwd, bwd = hholtz_eig(kind0, n0, c[0])
            check(lib().b2_hholtz_create(field._h, float(c[0]), float(c[1]), _dp(lam), _dp(fwd), _dp(bwd), C.byref(self._h)))
        else:
            check(lib().b2_hholtz_create(field._h, float(c[0]), float(c[1]), None, None, None, C.byref(self._h)))


def hholtz_eig(kind0, n0, c0, parity_split=None):
    """Eigendecomposition of ``C0^-1 (-c0 B0)`` for ``Hholtz`` (src/solver/hholtz.rs:79-81 + fdma_tensor.rs:117-129): the
    Poisson routine with the sign of the Laplacian flipped (its eigenvalues are then >= 0, so the singularity shift of
    ``Poisson::new`` never triggers -- ``Hholtz`` has none)."""
    return poisson_eig(kind0, n0, -float(c0), parity_split)


def _eig_sorted(x):
    """src/solver/utils.rs:67-100: LAPACK dgeev, real parts, eigenvalues sorted descending."""
    ev, evec = np.linalg.eig(x)
    ev, evec = ev.real, evec.real
    perm = np.argsort(ev, kind="stable")[::-1]
    return ev[perm], evec[:, perm]


def poisson_eig(kind0, n0, c0, parity_split=None):
    if os.environ.get("B2_EIG_CACHE"):   # optional on-disk cache of the host LAPACK setup (minutes at n = 8193)
        d = os.environ["B2_EIG_CACHE"]
        f = os.path.join(d, f"eig_k{kind0}_n{n0}_c{float(c0)!r}_p{parity_split}.npz")
        if os.path.exists(f):
            z = np.load(f)
            return z["lam"], z["fwd"], z["bwd"]
        lam, fwd, bwd = _poisson_eig(kind0, n0, c0, parity_split)
        os.makedirs(d, exist_ok=True)
        tmp = f"{f}.{os.getpid()}.tmp.npz"   # several ranks may fill the cache at once: write aside, then rename
        np.savez(tmp, lam=lam, fwd=fwd, bwd=bwd)
        os.replace(tmp, f)
        return lam, fwd, bwd
    return _poisson_eig(kind0, n0, c0, parity_split)


def _poisson_eig(kind0, n0, c0, parity_split=None):
    """Host-side setup of ``FdmaTensor::from_matrix`` (src/solver/fdma_tensor.rs:117-129) + the
    singularity rule of ``Poisson::new`` (src/solver/poisson.rs:84-86):  X = C0^-1 A0 = Q L Q^-1,
    returns (lam, fwd = Q^-1 C0^-1, bwd = Q).  A0 and C0 only couple indices of equal parity, so
    for large n the two parity blocks are diagonalised separately (4x less LAPACK work; the solve
    x = Q (..) Q^-1 C0^-1 rhs does not depend on how eigenvectors are scaled or grouped)."""
    m = n0 - 2
    a0 = np.zeros((m, m))
    cm = np.zeros((m, m))
    check(lib().b2_host_poisson_matrices(kind0, n0, float(c0), _dp(a0), _dp(cm)))
    if parity_split is None:
        parity_split = m >= 16
    if not parity_split:
        cinv = np.linalg.inv(cm)
        lam, q = _eig_sorted(cinv @ a0)
        fwd = np.linalg.inv(q) @ cinv
    else:
        lam = np.zeros(m)
        q = np.zeros((m, m))
        fwd_p = np.zeros((m, m))
        for par in (0, 1):
            idx = np.arange(par, m, 2)
            cinv = np.linalg.inv(cm[np.ix_(idx, idx)])
            l_p, q_p = _eig_sorted(cinv @ a0[np.ix_(idx, idx)])
            lam[idx] = l_p  # temporary slot; permuted below
            q[np.ix_(idx, idx)] = q_p
            fwd_p[np.ix_(idx, idx)] = np.linalg.inv(q_p) @ cinv
        perm = np.argsort(lam, kind="stable")[::-1]
        lam, q, fwd = lam[perm], q[:, perm], fwd_p[perm, :]
    if abs(lam[0]) < 1e-10:
        lam = lam - 1e-10
    return np.ascontiguousarray(lam), np.ascontiguousarray(fwd), np.ascontiguousarray(q)


class Poisson(_Solver):
    """``Poisson::new(&field, c)`` (src/solver/poisson.rs:54-94).  ``eig``: (lam, fwd, bwd) of axis 0 when the caller already
    has the host eigendecomposition (as ``Navier2D(pois_eig=...)``)."""

    def __init__(self, field, c, eig=None):
        self.field = field
        self._h = C.c_void_p()
        kind0, n0 = field.space.bases[0]
        if kind0 in (CHEB_DIRICHLET, CHEB_NEUMANN):
            lam, fwd, bwd = eig if eig is not None else poisson_eig(kind0, n0, c[0])
            lam, fwd, bwd = (np.ascontiguousarray(a, dtype=np.float64) for a in (lam, fwd, bwd))
            check(lib().b2_poisson_create(field._h, float(c[0]), float(c[1]), _dp(lam), _dp(fwd), _dp(bwd), C.byref(self._h)))
        else:
            check(lib().b2_poisson_create(field._h, float(c[0]), float(c[1]), None, None, None, C.byref(self._h)))


class _NavSpace:
    """Space view of a field owned by the native Navier2D object."""

    def __init__(self, nav, which):
        self._nav, self._which = nav, which


class Navier2D:
    """``Navier2D`` (src/navier_stokes/navier.rs:49-466).  ``new_confined`` / ``new_periodic`` build
    the same six fields, three ``HholtzAdi`` and one ``Poisson`` solver; ``update()`` advances one
    step on the GPU."""

    FIELDS = {"temp": 0, "velx": 1, "vely": 2, "pres": 3, "pseu": 4, "tempbc": 5}

    def __init__(self, nx, ny, ra, pr, dt, aspect, bc="rbc", periodic=False, ctx=None, pois_eig=None, init_random=True):
        """``pois_eig``: optional (lam, fwd, bwd) of ``poisson_eig`` (the host LAPACK setup of the confined Poisson
        solver) when the caller already has it.  ``init_random``: the reference constructors end with
        ``init_random(0.1)`` (navier.rs:305,425); pass False to start from zero fields."""
        self.ctx = ctx or default_context()
        self.nx, self.ny, self.ra, self.pr, self.dt, self.aspect = nx, ny, ra, pr, dt, aspect
        self.periodic = periodic
        self.scale = [aspect, 1.0]
        self._h = C.c_void_p()
        if periodic:
            args = (None, None, None)
        else:
            lam, fwd, bwd = pois_eig if pois_eig is not None else poisson_eig(CHEB_NEUMANN, nx, 1.0 / aspect ** 2)
            args = (_dp(lam), _dp(fwd), _dp(bwd))
        check(lib().b2_navier2d_create(self.ctx._h, nx, ny, ra, pr, dt, aspect, bc.encode(), int(periodic), *args, C.byref(self._h)))
        bx = (lambda k: fourier_r2c(nx)) if periodic else (lambda k: (k, nx))
        self.bc = bc
        kinds = {"temp": (bx(CHEB_DIRICHLET if periodic else CHEB_NEUMANN), cheb_dirichlet(ny) if bc == "rbc" else cheb_dirichlet_neumann(ny)),
                 "velx": (bx(CHEB_DIRICHLET), cheb_dirichlet(ny)), "vely": (bx(CHEB_DIRICHLET), cheb_dirichlet(ny)),
                 "pres": (bx(CHEBYSHEV), chebyshev(ny)), "pseu": (bx(CHEB_NEUMANN), cheb_neumann(ny)),
                 "tempbc": (bx(CHEBYSHEV), chebyshev(ny))}
        self.nranks = self.ctx.nranks
        for name, idx in self.FIELDS.items():
            fh = C.c_void_p()
            check(lib().b2_navier_field(self._h, idx, C.byref(fh)))
            sp = _BorrowedSpace(self.ctx, kinds[name], fh)
            f = Field2(sp, handle=fh)
            if name in ("velx", "vely", "temp", "pres"):
                f.scale(self.scale)
            setattr(self, name, f)
        if init_random:
            self.init_random(0.1)

    def close(self):
        """Free every device array, solver and space of this solver."""
        if getattr(self, "_h", None):
            for k in ("_field", "_field2", "_temp_twin", "_diag_a", "_diag_b", "_vel_twin", "_div_a", "_div_b"):
                if getattr(self, k, None) is not None:
                    setattr(self, k, None)
            _release(lib().b2_navier_destroy, self._h)
        self._h = None

    __del__ = close

    @classmethod
    def new_confined(cls, nx, ny, ra, pr, dt, aspect, bc="rbc", ctx=None, **kw):
        """navier.rs:215-308."""
        return cls(nx, ny, ra, pr, dt, aspect, bc, periodic=False, ctx=ctx, **kw)

    @classmethod
    def new_periodic(cls, nx, ny, ra, pr, dt, aspect, bc="rbc", ctx=None, **kw):
        """navier.rs:336-428."""
        return cls(nx, ny, ra, pr, dt, aspect, bc, periodic=True, ctx=ctx, **kw)

    # initial conditions: navier.rs:156-182, functions.rs:85-140
    def _unit(self, f):
        x, y = f.x
        return (x - x[0]) / (x[-1] - x[0]), (y - y[0]) / (y[-1] - y[0])

    def set_velocity(self, amp, m, n):
        x, y = self._unit(self.velx)
        self.velx.v = (amp * np.outer(np.sin(np.pi * m * x), np.cos(np.pi * n * y)))[self.velx.local_slice(PHYSICAL)]
        self.velx.forward()
        x, y = self._unit(self.vely)
        self.vely.v = (-amp * np.outer(np.cos(np.pi * m * x), np.sin(np.pi * n * y)))[self.vely.local_slice(PHYSICAL)]
        self.vely.forward()

    def set_temperature(self, amp, m, n):
        x, y = self._unit(self.temp)
        self.temp.v = (-amp * np.outer(np.cos(np.pi * m * x), np.sin(np.pi * n * y)))[self.temp.local_slice(PHYSICAL)]
        self.temp.forward()

    def init_random(self, amp, seeds=(1, 2, 3)):
        """U(-amp, amp) physical fields, then forward (navier.rs:171-182).  With several ranks every rank
        draws the same global field and keeps its rows (the reference draws on rank 0 and scatters,
        src/navier_stokes_mpi/functions.rs:269-286)."""
        for f, s in zip((self.temp, self.velx, self.vely), seeds):
            full = np.random.default_rng(s).uniform(-amp, amp, size=f.space.shape_physical())
            f.v = full[f.local_slice(PHYSICAL)]
            f.forward()

    # Integrate (src/lib.rs:167-178)
    def update(self, nsteps=1):
        check(lib().b2_navier_update(self._h, int(nsteps)))

    def get_time(self):
        t = C.c_double()
        check(lib().b2_navier_get_time(self._h, C.byref(t)))
        return t.value

    def get_dt(self):
        return self.dt

    def div_norm(self):
        v = C.c_double()
        check(lib().b2_navier_div_norm(self._h, C.byref(v)))   # same value on every rank (all_gather_sum of navier_eq.rs:51,64)
        return v.value

    def div(self):
        """``Navier2D::div`` (src/navier_stokes/navier_eq.rs:19-24): d(velx)/dx + d(vely)/dy in the orthonormal space, computed
        on the device (two gradients on a twin of the velocity space, summed); returns the global array on every rank."""
        if getattr(self, "_vel_twin", None) is None:
            self._vel_twin = Field2(Space2(*self.velx.space.bases, ctx=self.ctx))
            self._div_a = DeviceArray(self._vel_twin.space, ORTHO)
            self._div_b = DeviceArray(self._vel_twin.space, ORTHO)
        tw = self._vel_twin
        check(lib().b2_array_copy(self._borrow(tw, 1)._h, self._borrow(self.velx, 1)._h))
        tw.gradient([1, 0], self.scale, out=self._div_a)
        check(lib().b2_array_copy(self._borrow(tw, 1)._h, self._borrow(self.vely, 1)._h))
        tw.gradient([0, 1], self.scale, out=self._div_b)
        self._div_a.axpy(1.0, self._div_b)
        return self.ctx.all_gather_rows(self._div_a.get())

    def reset_time(self):
        """navier.rs:185-187."""
        self.set_time(0.0)

    def exit(self):
        """navier.rs:482-489: break when |div| is NaN."""
        return bool(np.isnan(self.div_norm()))

    # diagnostics (SURVEY 8f item 1; src/navier_stokes/functions.rs:146-233): everything runs on the device through the C ABI --
    # transforms, projections, derivatives, the pointwise products and the dx-weighted means of src/field/average.rs
    # (b2_array_weighted_sum over this rank's rows); with several ranks the partial sums are added across the ranks like
    # `all_gather_sum` in src/field_mpi/average.rs:15-61.  Only scalars (and one row profile for Nu) reach the host.
    def _borrow(self, f, which):
        h = C.c_void_p()
        check(lib().b2_field_array(f._h, which, C.byref(h)))
        return DeviceArray(f.space, PHYSICAL if which == 0 else SPECTRAL, handle=h, owner=False)

    def _diag_field(self):
        if getattr(self, "_field", None) is None:
            bx = fourier_r2c(self.nx) if self.periodic else chebyshev(self.nx)
            self._field = Field2(Space2(bx, chebyshev(self.ny), ctx=self.ctx))
            self._field2 = Field2(Space2(bx, chebyshev(self.ny), ctx=self.ctx))
            # the solver's own fields are borrowed handles without a standalone space: projections go through a twin
            self._temp_twin = Field2(Space2(*self.temp.space.bases, ctx=self.ctx))
            self._diag_a = DeviceArray(self._temp_twin.space, ORTHO)
            self._diag_b = DeviceArray(self._field.space, ORTHO)
            height = self.scale[1] * 2.0   # functions.rs:12-21
            self.nu = float(np.sqrt(self.pr / (self.ra / height ** 3.0)))
            self.ka = float(np.sqrt(1.0 / ((self.ra / height ** 3.0) * self.pr)))
            f = self._field
            lo = f.local_slice(PHYSICAL)
            self._w0 = np.ascontiguousarray((f.dx[0] / abs(f.x[0][-1] - f.x[0][0]))[lo])   # src/field/average.rs:26-35: dx / length
            self._w1 = np.ascontiguousarray(f.dx[1] / abs(f.x[1][-1] - f.x[1][0]))
        return self._field

    def _wsum(self, arr, mode):
        """this rank's part of average(v) (mode 0) or average_axis(v, 0) (mode 1), then summed over the ranks"""
        out = np.zeros(len(self._w1) if mode == 1 else 1)
        check(lib().b2_array_weighted_sum(arr._h, _dp(self._w0), _dp(self._w1), mode, _dp(out)))
        out = self.ctx.all_reduce_sum(out)
        return out if mode == 1 else float(out[0])

    def _temp_ortho_into(self, f):
        """f.vhat = to_ortho(temp) + to_ortho(tempbc)  (tempbc lives in the orthonormal space already)"""
        check(lib().b2_array_copy(self._borrow(self._temp_twin, 1)._h, self._borrow(self.temp, 1)._h))
        self._temp_twin.to_ortho(out=self._diag_a)
        fv = self._borrow(f, 1)
        check(lib().b2_array_copy(fv._h, self._diag_a._h))
        fv.axpy(1.0, self._borrow(self.tempbc, 1))

    def eval_nu(self):
        """Nusselt number from the heat flux at the plates (functions.rs:146-168)."""
        f = self._diag_field()
        self._temp_ortho_into(f)
        f.gradient([0, 1], [1.0, -self.scale[1] / 2.0], out=self._diag_b)   # d/dy * (-2 / scale_y)
        check(lib().b2_array_copy(self._borrow(f, 1)._h, self._diag_b._h))
        f.backward()
        x_avg = self._wsum(self._borrow(f, 0), 1)
        return float((x_avg[-1] + x_avg[0]) / 2.0)

    def eval_nuvol(self):
        """Volumetric Nusselt number (functions.rs:175-207)."""
        f = self._diag_field()
        g = self._field2
        self._temp_ortho_into(g)
        check(lib().b2_array_copy(self._borrow(f, 1)._h, self._borrow(g, 1)._h))
        g.backward()                                                           # T in physical space
        self.vely.backward()
        f.gradient([0, 1], [1.0, -self.scale[1]], out=self._diag_b)            # -dT/dy / scale_y
        check(lib().b2_array_copy(self._borrow(f, 1)._h, self._diag_b._h))
        f.backward()
        fv = self._borrow(f, 0)
        check(lib().b2_array_combine(fv._h, self._borrow(g, 0)._h, self._borrow(self.vely, 0)._h, 2, 1.0 / self.ka))   # + uy T / ka
        return self._wsum(fv, 0) * 2.0 * self.scale[1]

    def eval_re(self):
        """Reynolds number from the kinetic energy (functions.rs:215-233)."""
        f = self._diag_field()
        self.velx.backward()
        self.vely.backward()
        fv = self._borrow(f, 0)
        check(lib().b2_array_combine(fv._h, self._borrow(self.velx, 0)._h, self._borrow(self.vely, 0)._h, 1, 2.0 * self.scale[1] / self.nu))
        return self._wsum(fv, 0)

    def callback_from_filename(self, flow_name, info_name, suppress_io=False, write_flow_intervall=None):
        """``Navier2D::callback_from_filename`` (src/navier_stokes/navier_io.rs:84-147): write the flow field (always, or when
        the time is within dt of a multiple of ``write_flow_intervall``), then print ``time |div| Nu Nuv Re`` and append
        ``time nu nuv re`` to ``info_name`` unless ``suppress_io``.  The running statistics of the reference (``statistics.h5``)
        are out of scope (SURVEY 2 row 28).  Snapshots use the dataset names of the reference's HDF5 files (snapshot.py)."""
        t, dt = self.get_time(), self.get_dt()
        if flow_name:
            d = os.path.dirname(flow_name)
            if d and self.ctx.rank == 0:
                os.makedirs(d, exist_ok=True)
            if write_flow_intervall is None or (t + dt / 2.0) % write_flow_intervall < dt:
                self.write_unwrap(flow_name)
        if suppress_io:
            return None
        div, nu, nuv, re = self.div_norm(), self.eval_nu(), self.eval_nuvol(), self.eval_re()
        if self.ctx.rank == 0:
            print(f"time = {t:4.2f}      |div| = {div:4.2e}     Nu = {nu:5.3e}     Nuv = {nuv:5.3e}    Re = {re:5.3e}")
            if info_name:
                d = os.path.dirname(info_name)
                if d:
                    os.makedirs(d, exist_ok=True)
                with open(info_name, "a") as fh:
                    fh.write(f"{t} {nu} {nuv} {re}\n")
        return div, nu, nuv, re

    io_dir = None            # set to a directory (the reference uses "data") to make callback() write flow files and info.txt there
    write_intervall = None   # navier.rs: Option<f64>, forwarded to callback_from_filename by callback()

    def callback(self, info_name=None):
        """``Integrate::callback`` (navier.rs:476-480).  With ``io_dir`` set it is the reference's callback: flow field to
        ``<io_dir>/flow{time:0>8.2}.h5`` (``.npz`` when h5py is not installed) and one line to ``<io_dir>/info.txt``; by default (``io_dir`` None) it only prints the
        diagnostics line (and appends to ``info_name`` when given) so that library users do not get files they did not ask for."""
        if self.io_dir is not None:
            from . import snapshot as sn

            flow = os.path.join(self.io_dir, f"flow{self.get_time():0>8.2f}{sn.default_ext()}")   # .npz container without h5py
            return self.callback_from_filename(flow, os.path.join(self.io_dir, "info.txt"), False, self.write_intervall)
        return self.callback_from_filename(None, info_name, False, None)

    def set_mode(self, fused):
        check(lib().b2_navier_set_mode(self._h, int(fused)))

    def launches_per_step(self):
        k = C.c_longlong()
        check(lib().b2_navier_launch_count(self._h, C.byref(k)))
        return k.value

    def info(self):
        """Schedule facts: parity-block GEMMs on/off, padded sizes, Poisson block sizes, parallel branches."""
        v = (C.c_longlong * 8)()
        check(lib().b2_navier_info(self._h, v))
        keys = ("parity_blocks", "P0", "P1", "m0", "ce", "co", "branches", "launches_per_step")
        return dict(zip(keys, (int(x) for x in v)))

    # snapshot / restart (src/navier_stokes/navier_io.rs:21-62; MPI: gathered to / scattered from rank 0, src/field_mpi/io.rs)
    def write(self, filename):
        """``Navier2D::write``: backward() the four state fields, then ``ux, uy, temp, pres, tempbc`` groups and the scalars.
        With several ranks the arrays are gathered and rank 0 writes (src/navier_stokes_mpi/navier_io.rs)."""
        from . import snapshot as sn

        data = {}
        fields = list(sn.FIELD_GROUPS) + [("tempbc", "tempbc")]
        for attr, group in fields:
            f = getattr(self, attr)
            if attr != "tempbc":
                f.backward()
            v = self.ctx.all_gather_rows(f.v) if self.nranks > 1 else f.v
            vhat = self.ctx.all_gather_rows(f.vhat) if self.nranks > 1 else f.vhat
            data.update(sn.field_datasets(group, f.x[0], f.x[1], v, vhat))
        data["time"] = self.get_time()
        nu = np.sqrt(self.pr / (self.ra / 8.0)); ka = np.sqrt(1.0 / ((self.ra / 8.0) * self.pr))   # functions.rs:12-21, height 2
        data.update({"ra": self.ra, "pr": self.pr, "nu": nu, "ka": ka})
        if self.ctx.rank == 0:
            sn.save_datasets(filename, data)
        if self.nranks > 1:
            self.ctx.barrier()

    def read(self, filename):
        """``Navier2D::read``: ``vhat`` of ux, uy, temp, pres (interpolated spectrally when the snapshot has another
        resolution, src/field/io.rs:151-176), ``backward()``, and ``time``."""
        from . import snapshot as sn

        data = sn.load_datasets(filename)
        for attr, group in sn.FIELD_GROUPS:
            f = getattr(self, attr)
            shape, cx = f.space.shape(SPECTRAL)
            vh = sn.read_vhat(data, group, shape, cx, f.space.bases[0][0] == FOURIER_R2C)
            f.vhat = vh[f.local_slice(SPECTRAL)]
            f.backward()
        self.set_time(float(data["time"]))

    def write_unwrap(self, filename):
        try:
            self.write(filename)
        except Exception as e:  # noqa: BLE001 - navier_io.rs:57-62 prints and carries on
            print(f"Error while writing file {filename!r}. Error: {e}")

    def read_unwrap(self, filename):
        try:
            self.read(filename)
            print(f"Reading file {filename!r} was successfull.")
        except Exception as e:  # noqa: BLE001
            print(f"Error while reading file {filename!r}. Error: {e}")

    def set_time(self, t):
        check(lib().b2_navier_set_time(self._h, float(t)))

    def state(self):
        """This rank's slabs of the four spectral state arrays."""
        return {k: getattr(self, k).vhat for k in ("temp", "velx", "vely", "pres")}

    def gather_state(self):
        """Global state arrays on every rank (gather_spectral of src/field_mpi.rs:363-376)."""
        return {k: self.ctx.all_gather_rows(v) for k, v in self.state().items()}


class _BorrowedSpace(Space2):
    """Space2 facade for fields owned by a native Navier2D (no second native space is created;
    shapes and coordinates are computed from the base kinds)."""

    def __init__(self, ctx, bases, field_handle):
        self.ctx, self.bases, self._h = ctx, bases, None

    def _len(self, ax, kind):
        k, n = self.bases[ax]
        if kind == PHYSICAL:
            return n
        if k == FOURIER_R2C:
            return n // 2 + 1
        if kind == ORTHO or k == CHEBYSHEV:
            return n
        return n - 2

    def shape(self, kind):
        return (self._len(0, kind), self._len(1, kind)), (self.bases[0][0] == FOURIER_R2C and kind != PHYSICAL)

    def coords(self):
        out = []
        for k, n in self.bases:
            out.append(2 * np.pi * np.arange(n) / n if k == FOURIER_R2C else -np.cos(np.pi * np.arange(n) / (n - 1)))
        return out


MAX_TIMESTEP = 10_000_000


def integrate(pde, max_time, save_intervall=None):
    """``integrate`` loop (src/lib.rs:187-219): update, callback at save intervals, stop at
    ``max_time`` or when ``exit()`` reports a NaN divergence."""
    eps_dt = pde.get_dt() * 1e-4
    timestep = 0
    while True:
        pde.update()
        timestep += 1
        t = pde.get_time()
        if save_intervall is not None:   # lib.rs:197-199: both sides of the save time
            r = t % save_intervall
            if r < pde.get_dt() / 2.0 or r > save_intervall - pde.get_dt() / 2.0:
                pde.callback()
        if t + eps_dt >= max_time:
            break
        if timestep >= MAX_TIMESTEP:   # lib.rs:23,209-212
            break
        if pde.exit():
            break
