"""Device-backed stand-ins for the `spl.linalg.stencil` containers the reference's hot path is
written against (SURVEY.md Appendix C), plus the Kronecker-sum operator that replaces the
assembled 2-D `StencilMatrix` (section 8a, a3).

* `StencilVectorSpace`, `StencilVector`: same constructor, attributes and operators as the
  spl classes the reference uses (`.space .starts .ends .pads .npts`, `[]` with GLOBAL
  indices, `.copy() .dot() .toarray()`, `+ - *`, `.update_ghost_regions()`), storage is a
  torch fp64 CUDA tensor.  Axis 1 is the slowest axis; under a slab partition (dist.py) the
  tensor carries `p1` ghost planes below/above the owned planes.
* `StencilMatrix`: 1-D banded matrix `[i, k]`, k in [-p, p] (host NumPy, uploaded once) or
  full 2-D stencil `[i1, i2, k1, k2]`.
* `KronSumMatrix`: A = sum_a M (x) .. (x) K_a (x) .. (x) M, or a single Kronecker product.

Every arithmetic operation launches a kernel of libpoms_b200.so; nothing here computes on
the CPU and nothing falls back.
"""
import numpy as np
import torch

from . import _lib
from . import bsplines as bs
from . import profiling

FORM_SINGLE, FORM_SUM = 0, 1
EPI_STORE, EPI_RESID, EPI_JACOBI, EPI_DINV, EPI_AXPY = 0, 1, 2, 3, 4


def _stream():
    return torch.cuda.current_stream().cuda_stream


class DeviceContext:
    """Per-device workspace (reduction scratch) and a pool of device scalars."""

    _cache = {}

    def __init__(self, device):
        L = _lib.lib()
        self.device = device
        self.ws = torch.zeros(int(L.poms_workspace_bytes()), dtype=torch.uint8, device=device)
        self.scal = torch.zeros(64, dtype=torch.float64, device=device)
        self.one = torch.ones(1, dtype=torch.float64, device=device)

    @classmethod
    def get(cls, device):
        device = torch.device(device)
        if device.type != "cuda":
            raise _lib.PomsError("poms_b200 runs on CUDA devices only (got %s); there is no "
                                 "CPU path" % device)
        if device.index is None:
            device = torch.device("cuda", torch.cuda.current_device())
        if device not in cls._cache:
            cls._cache[device] = cls(device)
        return cls._cache[device]

    def sptr(self, i):
        return self.scal.data_ptr() + 8 * i

    @property
    def ws_ptr(self):
        return self.ws.data_ptr()


class SubComm:
    """The few mpi4py communicator methods the reference calls on `cart.subcomm[i]`
    (sources/kron_product.py:156,224; pyccel/pyccel_functions.py:98,158): Allgatherv of host
    arrays along one axis of the process grid.  Axis 1 = the slab group, other axes = one rank."""

    def __init__(self, slab=None):
        self.slab = slab if (slab is not None and slab.size > 1) else None

    def Get_size(self):
        return self.slab.size if self.slab is not None else 1

    def Get_rank(self):
        return self.slab.rank if self.slab is not None else 0

    size = property(Get_size)
    rank = property(Get_rank)

    def py2f(self):
        return 0

    def Allgatherv(self, sendbuf, recvbuf):
        """recvbuf: array, or [array, counts, displs(, type)] like mpi4py."""
        send = np.ascontiguousarray(sendbuf, dtype=np.float64).reshape(-1)
        if isinstance(recvbuf, (list, tuple)):
            recv, counts, displs = recvbuf[0], recvbuf[1], recvbuf[2]
        else:
            recv, counts, displs = recvbuf, None, None
        if self.slab is None:
            recv.reshape(-1)[:send.size] = send
            return
        import torch.distributed as dist
        G = self.slab.size
        dev = self.slab.device if self.slab.device is not None else "cpu"
        n = torch.tensor([send.size], dtype=torch.int64, device=dev)
        ns = [torch.zeros_like(n) for _ in range(G)]
        dist.all_gather(ns, n, group=self.slab.group)
        ns = [int(v.item()) for v in ns]
        mx = max(ns)
        pad = torch.zeros(mx, dtype=torch.float64, device=dev)
        pad[:send.size] = torch.as_tensor(send, device=dev)
        parts = [torch.empty_like(pad) for _ in range(G)]
        dist.all_gather(parts, pad, group=self.slab.group)
        flat = recv.reshape(-1)
        off = 0
        for r in range(G):
            o = int(displs[r]) if displs is not None else off
            c = int(counts[r]) if counts is not None else ns[r]
            flat[o:o + c] = parts[r][:c].cpu().numpy()
            off += ns[r]


class _PaddedData:
    """`StencilVector._data` of spl: the local array padded by `pads` ghost entries on every side of
    every axis (sources/utils.py:99, pyccel/kron_product.py:53,81-87 index it directly).  The device
    storage has ghost planes along axis 1 only (slab partition) and none inside a plane, so this is a
    host-side window: reads gather the padded array (in-plane ghosts of a non-periodic space are
    zero), writes scatter the owned entries (and the axis-1 ghost planes that exist) back."""

    def __init__(self, vec):
        self._v = vec

    @property
    def shape(self):
        V = self._v.space
        return tuple(n + 2 * p for n, p in zip(V.local_shape, V.pads))

    def _gather(self):
        v = self._v
        V = v.space
        out = np.zeros(self.shape)
        own = tuple(slice(p, p + n) for n, p in zip(V.local_shape, V.pads))
        out[own] = v.data.cpu().numpy()
        p0 = V.pads[0]
        rest = own[1:]
        if V.glo:
            out[(slice(p0 - V.glo, p0),) + rest] = v._log[:V.glo].cpu().numpy()
        if V.ghi:
            n0 = V.local_shape[0]
            out[(slice(p0 + n0, p0 + n0 + V.ghi),) + rest] = v._log[V.glo + n0:].cpu().numpy()
        return out

    def _scatter(self, arr):
        v = self._v
        V = v.space
        own = tuple(slice(p, p + n) for n, p in zip(V.local_shape, V.pads))
        v.data.copy_(torch.as_tensor(np.ascontiguousarray(arr[own]), device=V.device))
        p0, n0 = V.pads[0], V.local_shape[0]
        rest = own[1:]
        if V.glo:
            v._log[:V.glo].copy_(torch.as_tensor(np.ascontiguousarray(
                arr[(slice(p0 - V.glo, p0),) + rest]), device=V.device))
        if V.ghi:
            v._log[V.glo + n0:].copy_(torch.as_tensor(np.ascontiguousarray(
                arr[(slice(p0 + n0, p0 + n0 + V.ghi),) + rest]), device=V.device))

    def __array__(self, dtype=None, copy=None):
        a = self._gather()
        return a if dtype is None else a.astype(dtype)

    def __getitem__(self, key):
        return self._gather()[key]

    def __setitem__(self, key, value):
        a = self._gather()
        a[key] = value
        self._scatter(a)

    def copy(self, order="C"):
        return np.array(self._gather(), order=order)

    @property
    def T(self):
        return self._gather().T


class Cart:
    """Minimal cartesian-decomposition record (spl.ddm.cart.Cart attribute names)."""

    def __init__(self, npts, pads, periods, reorder=False, comm=None, slab=None):
        self.npts = tuple(int(n) for n in npts)
        self.pads = tuple(int(p) for p in pads)
        self.periods = tuple(bool(b) for b in periods)
        self.ndim = len(self.npts)
        self.slab = slab
        rank, size = (slab.rank, slab.size) if slab is not None else (0, 1)
        self._rank, self._size = rank, size
        self.nprocs = [size] + [1] * (self.ndim - 1)
        self.coords = [rank] + [0] * (self.ndim - 1)
        if slab is not None:
            s1, e1 = slab.bounds(self.npts[0])
        else:
            s1, e1 = 0, self.npts[0] - 1
        self.starts = (s1,) + tuple(0 for _ in self.npts[1:])
        self.ends = (e1,) + tuple(n - 1 for n in self.npts[1:])
        # one sub-communicator per axis (spl: cart.subcomm[i]; used by the reference's per-line
        # Allgatherv, sources/kron_product.py:140-141,156,162): the slab group along axis 1, a
        # single-rank communicator along every other axis
        self.subcomm = [SubComm(slab if d == 0 else None) for d in range(self.ndim)]
        self.comm_cart = comm


class StencilVectorSpace:
    def __init__(self, *args, device=None, slab=None, **kw):
        if len(args) == 1 and isinstance(args[0], Cart):
            cart = args[0]
        else:
            npts, pads, periods = (list(args) + [None] * 3)[:3]
            npts = kw.get("npts", npts)
            pads = kw.get("pads", pads)
            periods = kw.get("periods", periods) or [False] * len(npts)
            cart = Cart(npts, pads, periods, slab=slab)
        if any(cart.periods):
            raise NotImplementedError("periodic spaces are not on the POMS hot path")
        self._cart = cart
        self.npts = cart.npts
        self.pads = cart.pads
        self.periods = cart.periods
        self.starts = cart.starts
        self.ends = cart.ends
        self.ndim = cart.ndim
        self.slab = cart.slab
        self.device = torch.device(device) if device is not None else torch.device("cuda")
        p1 = self.pads[0]
        self.glo = p1 if (self.slab is not None and self.slab.rank > 0) else 0
        self.ghi = p1 if (self.slab is not None and self.slab.rank < self.slab.size - 1) else 0
        self.local_shape = tuple(e - s + 1 for s, e in zip(self.starts, self.ends))
        # row pitch (doubles): even, so that every row starts 16-byte aligned (TMA global strides,
        # 128-bit loads).  The pad column, if any, is kept at zero by every kernel.
        n_last = self.local_shape[-1]
        self.ld = n_last + (n_last & 1) if self.ndim >= 2 else n_last
        self.pitched_shape = self.local_shape[:-1] + (self.ld,)

    @property
    def cart(self):
        return self._cart

    @property
    def dimension(self):
        return int(np.prod(self.npts))

    @property
    def local_size(self):
        """Owned DOFs."""
        return int(np.prod(self.local_shape))

    @property
    def flat_size(self):
        """Doubles in the owned storage range (includes the zero pad column)."""
        return int(np.prod(self.pitched_shape))

    def zeros(self):
        return StencilVector(self)

    def compatible(self, other):
        return (self.npts == other.npts and self.starts == other.starts
                and self.ends == other.ends and self.glo == other.glo and self.ghi == other.ghi)


class StencilVector:
    def __init__(self, V, _buf=None, zero=True, peer=False):
        """zero=False: storage is left uninitialised except for the pad column and the ghost
        planes (for vectors that a kernel overwrites completely; saves a full-size memset).
        peer=True (persistent work vectors of slab-partitioned spaces): storage from the slab's
        IPC-shared arena, so that halo exchanges are peer stores; COLLECTIVE (every rank must
        create its peer vectors in the same order)."""
        self._space = V
        shape = (V.glo + V.local_shape[0] + V.ghi,) + V.pitched_shape[1:]
        if _buf is None and peer and V.slab is not None and V.slab.size > 1:
            n_max = -(-V.npts[0] // V.slab.size) + 2 * V.pads[0]   # largest slab + both ghost blocks
            got = V.slab.alloc_planes(n_max, V.pitched_shape[1:])
            if got is not None:
                _buf = got[0][:shape[0]]                            # zero-initialised by the arena
                self._arena_key = got[1]
        if _buf is None:
            if zero:
                _buf = torch.zeros(shape, dtype=torch.float64, device=V.device)
            else:
                _buf = torch.empty(shape, dtype=torch.float64, device=V.device)
                if V.ld != V.local_shape[-1]:
                    _buf[..., V.local_shape[-1]:] = 0.0
                if V.glo:
                    _buf[:V.glo] = 0.0
                if V.ghi:
                    _buf[V.glo + V.local_shape[0]:] = 0.0
        assert tuple(_buf.shape) == shape and _buf.is_contiguous()
        self._buf = _buf
        self.flat = _buf[V.glo:V.glo + V.local_shape[0]]          # owned planes, pitched
        self.data = self.flat[..., :V.local_shape[-1]]             # logical (n1, .., n_last) view
        self._log = _buf[..., :V.local_shape[-1]]                  # same incl. the ghost planes

    # ---- spl-compatible surface ---------------------------------------------------------
    @property
    def space(self):
        return self._space

    @property
    def starts(self):
        return self._space.starts

    @property
    def ends(self):
        return self._space.ends

    @property
    def pads(self):
        return self._space.pads

    @property
    def shape(self):
        return (self._space.dimension,)

    def _local(self, key):
        if not isinstance(key, tuple):
            key = (key,)
        out = []
        for d, i in enumerate(key):
            off = self._space.starts[d] - (self._space.glo if d == 0 else 0)
            if isinstance(i, slice):
                a = None if i.start is None else i.start - off
                b = None if i.stop is None else i.stop - off
                out.append(slice(a, b, i.step))
            else:
                out.append(int(i) - off)
        return tuple(out)

    # Indexing uses GLOBAL indices like spl (axis 1 reaches into the ghost planes of a slab) and goes
    # through the logical view: the zero pad column of the pitched storage is never addressed, so
    # `x[:, :] = 1.` cannot corrupt the BLAS-1 kernels that run over it.  Deviation from spl: a full
    # slice covers the owned entries (+ axis-1 ghost planes), spl's also covers in-plane ghosts, which
    # this storage does not have (`_data` emulates them).
    def __getitem__(self, key):
        v = self._log[self._local(key)]
        return v.item() if v.ndim == 0 else v.cpu().numpy()

    def __setitem__(self, key, value):
        if isinstance(value, np.ndarray):
            value = torch.as_tensor(value, dtype=torch.float64, device=self._buf.device)
        self._log[self._local(key)] = value

    @property
    def _data(self):
        return _PaddedData(self)

    @_data.setter
    def _data(self, arr):
        _PaddedData(self)._scatter(np.asarray(arr, dtype=np.float64))

    def copy(self):
        w = StencilVector(self._space, _buf=torch.empty_like(self._buf))
        w._buf.copy_(self._buf)
        return w

    def toarray(self):
        """Global-size flat array with the owned entries filled in (spl semantics)."""
        V = self._space
        if V.slab is None:
            return self.data.reshape(-1).cpu().numpy()
        out = np.zeros(V.npts)
        out[V.starts[0]:V.ends[0] + 1] = self.data.cpu().numpy()
        return out.reshape(-1)

    def dot(self, other):
        """Sum over owned entries (+ all-reduce over slabs); returns a Python float."""
        ctx = DeviceContext.get(self._buf.device)
        dot_into(self, other, ctx.sptr(0), ctx)
        v = ctx.scal[0:1]
        if self._space.slab is not None:
            v = self._space.slab.allreduce_sum(v.clone())
        return float(v.item())

    def update_ghost_regions(self, direction=None):
        if self._space.slab is not None:
            self._space.slab.exchange(self)

    def _axpby(self, a, b, y):
        z = StencilVector(self._space, zero=False)
        L = _lib.lib()
        _lib.check(L.poms_axpby(z.ptr, float(a), self.ptr, float(b),
                                 y.ptr if y is not None else None, self.n_owned, _stream()),
                   "poms_axpby")
        return z

    def __mul__(self, a):
        return self._axpby(a, 0.0, None)

    __rmul__ = __mul__

    def __add__(self, v):
        return self._axpby(1.0, 1.0, v)

    def __sub__(self, v):
        return self._axpby(1.0, -1.0, v)

    def __neg__(self):
        return self._axpby(-1.0, 0.0, None)

    # ---- device helpers ------------------------------------------------------------------
    @property
    def ptr(self):
        """Device pointer of the first OWNED entry."""
        return self.flat.data_ptr()

    @property
    def n_owned(self):
        """Length of the contiguous owned storage range (BLAS-1 kernels run over it)."""
        return self._space.flat_size

    @property
    def ld(self):
        return self._space.ld

    @property
    def pld(self):
        s = self._space.pitched_shape
        return s[-1] * s[-2]

    def zero_(self):
        self._buf.zero_()
        return self

    def copy_(self, other):
        self._buf.copy_(other._buf)
        return self

    @classmethod
    def from_array(cls, V, arr):
        """Upload a GLOBAL (n1, ..., nd) array; each slab keeps its owned planes
        (`array_to_vect_stencil`, /root/reference/sources/utils.py:92-101)."""
        v = cls(V)
        arr = np.asarray(arr, dtype=np.float64).reshape(V.npts)
        loc = arr[V.starts[0]:V.ends[0] + 1]
        v.data.copy_(torch.as_tensor(np.ascontiguousarray(loc), device=V.device))
        return v


def dot_into(x, y, out_ptr, ctx=None):
    """*out = x.y over owned entries (local part), asynchronous."""
    ctx = ctx or DeviceContext.get(x._buf.device)
    _lib.check(_lib.lib().poms_dot(x.ptr, y.ptr, x.n_owned, out_ptr, ctx.ws_ptr, _stream()),
               "poms_dot")


# ==========================================================================================
# matrices
# ==========================================================================================
class StencilMatrix:
    """spl-style stencil matrix on the host (setup object), uploaded on first use.
    1-D: `_data[i, k+p]` = A[i, i+k]; 2-D: `_data[i1, i2, k1+p1, k2+p2]`."""

    def __init__(self, V, W=None):
        W = W or V
        assert V.npts == W.npts and V.pads == W.pads
        if V.ndim not in (1, 2, 3):
            raise NotImplementedError("StencilMatrix: 1-D bands or full 2-D / 3-D stencils")
        self._domain, self._codomain = V, W
        self.ndim = V.ndim
        self.starts = tuple(0 for _ in V.npts)
        self.ends = tuple(n - 1 for n in V.npts)
        self.pads = V.pads
        self._data = np.zeros(tuple(V.npts) + tuple(2 * p + 1 for p in V.pads))
        self._dev = None
        self._slab_dev = {}

    @property
    def domain(self):
        return self._domain

    @property
    def codomain(self):
        return self._codomain

    @property
    def shape(self):
        n = int(np.prod(self._domain.npts))
        return (n, n)

    def _index(self, key):
        assert isinstance(key, tuple) and len(key) == 2 * self.ndim
        out = list(key[:self.ndim])
        for k, p in zip(key[self.ndim:], self.pads):
            if isinstance(k, slice):
                a = None if k.start is None else k.start + p
                b = None if k.stop is None else k.stop + p
                out.append(slice(a, b, k.step))
            else:
                out.append(k + p)
        return tuple(out)

    def __getitem__(self, key):
        return self._data[self._index(key)]

    def __setitem__(self, key, value):
        self._data[self._index(key)] = value
        self._dev = None
        self._slab_dev = {}

    def remove_spurious_entries(self):
        for d, (n, p) in enumerate(zip(self._domain.npts, self.pads)):
            i = np.arange(n)[:, None]
            k = np.arange(-p, p + 1)[None, :]
            bad = (i + k < 0) | (i + k >= n)
            shape = [1] * (2 * self.ndim)
            shape[d], shape[self.ndim + d] = bad.shape
            self._data[np.broadcast_to(bad.reshape(shape), self._data.shape)] = 0.0
        self._dev = None
        self._slab_dev = {}

    # host-side views used by setup code and tests
    def tocoo(self):
        from scipy.sparse import coo_matrix
        npts = self._domain.npts
        grids = np.meshgrid(*[np.arange(n) for n in npts], indexing="ij")
        rows, cols, vals = [], [], []
        for ks in np.ndindex(*[2 * p + 1 for p in self.pads]):
            js = [g + k - p for g, k, p in zip(grids, ks, self.pads)]
            ok = np.ones(grids[0].shape, dtype=bool)
            for j, n in zip(js, npts):
                ok &= (j >= 0) & (j < n)
            v = self._data[(Ellipsis,) + ks]
            ok &= v != 0.0
            rows.append(np.ravel_multi_index([g[ok] for g in grids], npts))
            cols.append(np.ravel_multi_index([j[ok] for j in js], npts))
            vals.append(v[ok])
        n = int(np.prod(npts))
        return coo_matrix((np.concatenate(vals), (np.concatenate(rows), np.concatenate(cols))),
                          shape=(n, n))

    def tocsr(self):
        return self.tocoo().tocsr()

    def toarray(self):
        return self.tocoo().toarray()

    def band(self, P=None):
        assert self.ndim == 1
        return bs.pad_band(self._data, self.pads[0] if P is None else P)

    def device_data(self, device):
        if self._dev is None or self._dev.device != torch.device(device):
            self._dev = torch.as_tensor(np.ascontiguousarray(self._data), device=device)
        return self._dev

    # ---- operator interface shared with KronSumMatrix (2-D full stencil only) -------------
    def _rows_for(self, V):
        """Device stencil rows of the planes a slab owns."""
        key = (V.starts[0], V.ends[0], str(V.device))
        if key not in self._slab_dev:
            loc = np.ascontiguousarray(self._data[V.starts[0]:V.ends[0] + 1])
            self._slab_dev[key] = torch.as_tensor(loc, device=V.device)
        return self._slab_dev[key]

    def apply(self, x, y, epi=EPI_STORE, b=None, omega=0.0, dot_ptr=None):
        assert self.ndim in (2, 3)
        V = x.space
        if V.slab is not None:
            V.slab.exchange(x)
        ctx = DeviceContext.get(V.device)
        S = self._rows_for(V)
        if self.ndim == 3:
            # full 3-D stencil ((2p+1)^3 coefficients per row): EXTENSION of the reference's 2-D type
            n1, n2, n3 = V.local_shape
            nbytes = 8 * S.numel() + 16 * V.local_size
            with profiling.region("stencil_matvec_3d", nbytes):
                _lib.check(_lib.lib().poms_stencil_matvec_3d(
                    x.ptr, y.ptr, b.ptr if b is not None else None, S.data_ptr(), n1, n2, n3, x.ld, x.pld,
                    V.glo, V.ghi, self.pads[0], self.pads[1], self.pads[2], epi, float(omega), dot_ptr,
                    ctx.ws_ptr, _stream()), "poms_stencil_matvec_3d")
            return
        n1, n2 = V.local_shape
        _lib.check(_lib.lib().poms_stencil_matvec_2d(
            x.ptr, y.ptr, b.ptr if b is not None else None, S.data_ptr(), n1, n2, x.ld,
            V.glo, V.ghi, self.pads[0], self.pads[1], epi, float(omega), dot_ptr, ctx.ws_ptr,
            _stream()), "poms_stencil_matvec_2d")

    def dot(self, v):
        if self.ndim not in (2, 3):
            raise NotImplementedError("StencilMatrix.dot: 2-D / 3-D stencils (1-D factors are applied "
                                      "through kron_dot / KronSumMatrix)")
        out = StencilVector(v.space)
        self.apply(v, out)
        return out

    def diagonal_vector(self, V):
        d = StencilVector(V)
        centre = (slice(V.starts[0], V.ends[0] + 1),) + (slice(None),) * (self.ndim - 1) + tuple(self.pads)
        loc = np.ascontiguousarray(self._data[centre])
        d.flat.fill_(1.0)          # pad column: 0/1 keeps the pad at zero
        d.data.copy_(torch.as_tensor(loc, device=V.device))
        return d

    def jacobi_first(self, x, b, omega, dot_ptr):
        V = b.space
        ctx = DeviceContext.get(V.device)
        if not hasattr(self, "_diag") or self._diag[0] is not V:
            self._diag = (V, self.diagonal_vector(V))
        _lib.check(_lib.lib().poms_diag_scale(x.ptr, b.ptr, self._diag[1].ptr, b.n_owned,
                                               float(omega), dot_ptr, ctx.ws_ptr, _stream()),
                   "poms_diag_scale")


def reaction_robin(c, robin, ndim):
    """Checked (c, robin) of `KronSumMatrix.poisson`: c as a float, robin as None or a list of ndim
    (alpha_lo, alpha_hi) float pairs.  Raises ValueError for a negative or non-finite value, a wrong
    number of pairs, and for c = 0 without a positive alpha (the operator would be singular: constants
    are in its kernel)."""
    try:
        c = float(c)
    except (TypeError, ValueError):
        raise ValueError("c must be a number (got %r)" % (c,)) from None
    if not np.isfinite(c) or c < 0.0:
        raise ValueError("c must be finite and >= 0 (got %r)" % c)
    if robin is not None:
        try:
            pairs = [tuple(float(v) for v in ab) for ab in robin]
        except (TypeError, ValueError):
            raise ValueError("robin must be None or %d pairs (alpha_lo, alpha_hi) of numbers" % ndim) from None
        if len(pairs) != ndim or any(len(ab) != 2 for ab in pairs):
            raise ValueError("robin must have one pair (alpha_lo, alpha_hi) per axis (%d)" % ndim)
        for a, ab in enumerate(pairs):
            if not all(np.isfinite(v) and v >= 0.0 for v in ab):
                raise ValueError("robin coefficients must be finite and >= 0 (axis %d: %r)" % (a, ab))
        robin = pairs
    if c == 0.0 and (robin is None or not any(v > 0.0 for ab in robin for v in ab)):
        raise ValueError("c = 0 needs a Robin coefficient alpha > 0 on at least one face: -Lap u with "
                         "du/dn = 0 everywhere is singular (constants are in its kernel)")
    return c, robin


def convection_beta(beta, ndim):
    """Checked velocity of `KronSumMatrix.poisson`: None, or a list of ndim finite floats (ValueError)."""
    if beta is None:
        return None
    try:
        vals = [float(v) for v in beta]
    except (TypeError, ValueError):
        raise ValueError("beta must be None or %d numbers (one velocity component per axis)" % ndim) from None
    if len(vals) != ndim:
        raise ValueError("beta must have one component per axis (%d), got %d" % (ndim, len(vals)))
    if not all(np.isfinite(v) for v in vals):
        raise ValueError("beta must be finite (got %r)" % (vals,))
    return vals


def _gen_eig_min(Sb, Mb, lower):
    """Smallest generalised eigenvalue of S x = l M x for a symmetric band S (possibly indefinite) and the
    SPD mass band M (host), given a lower bound `lower` of it.  n <= 1500: dense LAPACK; above: shift-invert
    Lanczos (sparse LU of S - s M) at a shift s below `lower`, the same size split as `mg._gen_eig_max`."""
    n = Sb.shape[0]
    if n <= 1500:
        from scipy.linalg import eigh
        return float(eigh(bs.band_to_dense(Sb), bs.band_to_dense(Mb), eigvals_only=True,
                          subset_by_index=[0, 0])[0])
    import scipy.sparse as sp
    from scipy.sparse.linalg import eigsh

    def csc(band):
        p = (band.shape[1] - 1) // 2
        diags = [band[max(0, -k):n - max(0, k), k + p] for k in range(-p, p + 1)]
        return sp.diags(diags, list(range(-p, p + 1)), shape=(n, n), format="csc")
    v0 = np.cos(np.arange(n) * 0.7) + 1.5          # deterministic start vector
    return float(eigsh(csc(Sb), k=1, M=csc(Mb), sigma=lower - 1.0, which="LM", v0=v0,
                       return_eigenvectors=False)[0])


def symmetric_part_lmin(Ks, Ms, c, beta, lengths):
    """lambda_min(A_s, M (x) .. (x) M) of the operator with the bands Ks (K_a + R_a, without c M and
    without the advection), Ms and the axis lengths L_a: A_s = sum_a S_a (x) M_others + c M (x) .. (x) M
    with S_a = K_a + R_a + (beta_a / 2)(E_hi - E_lo), because G_a + G_a^T = E_hi - E_lo.  All factors are
    symmetric and share M, so the value is c + sum_a lambda_min(S_a, M_a): d 1-D problems.

    Lower bound of a 1-D value (the shift of the sparse path): Galerkin eigenvalues are bounded below by
    the continuous ones, and u(x0)^2 <= e |u'|^2 + (1/e + 1/L) |u|^2 with e = 2 / |beta| gives
    lambda_min(S_a, M_a) >= -(beta^2 / 4 + |beta| / (2 L))."""
    lam = c
    for a, (K, M) in enumerate(zip(Ks, Ms)):
        S = np.array(K, dtype=np.float64)
        b = beta[a] if beta is not None else 0.0
        p = (S.shape[1] - 1) // 2
        S[0, p] -= 0.5 * b
        S[-1, p] += 0.5 * b
        la = _gen_eig_min(S, M, -(0.25 * b * b + 0.5 * abs(b) / lengths[a]))
        # K_a + R_a is positive semi-definite: a rounding-level negative value of a pure Neumann axis is 0
        lam += max(la, 0.0) if b == 0.0 else la
    return lam


class KronSumMatrix:
    """Kronecker-structured operator on a d-dim tensor-product space (d = 2, 3).

    form == FORM_SUM:   A = sum_a  M_1 (x) .. K_a .. (x) M_d   (bands Ms[a], Ks[a]); the last
                        K must already contain K + c M for the weak form -Lap u + c u (`poisson`).
    form == FORM_SINGLE: A = A_1 (x) .. (x) A_d                 (bands Ms[a]).
    Narrower bands are zero-padded to the common half-bandwidth P = max(pads).
    """

    def __init__(self, Ms, Ks=None, form=None):
        Ms = [np.asarray(m._data if isinstance(m, StencilMatrix) else m, dtype=np.float64)
              for m in Ms]
        self.ndim = len(Ms)
        if self.ndim not in (2, 3):
            raise NotImplementedError("KronSumMatrix: 2-D or 3-D")
        if Ks is None:
            form = FORM_SINGLE
        else:
            form = FORM_SUM if form is None else form
            Ks = [np.asarray(k._data if isinstance(k, StencilMatrix) else k, dtype=np.float64)
                  for k in Ks]
        self.form = form
        self.npts = tuple(m.shape[0] for m in Ms)
        self.pads = tuple((m.shape[1] - 1) // 2 for m in Ms)
        self.P = max(self.pads)
        if not 1 <= self.P <= 5:
            raise ValueError("half-bandwidth must be 1..5")
        self.Ms = [bs.pad_band(m, self.P) for m in Ms]
        self.Ks = [bs.pad_band(k, self.P) for k in Ks] if Ks is not None else None
        n = int(np.prod(self.npts))
        self.shape = (n, n)
        self._dev = {}

    @classmethod
    def poisson(cls, p, knots, c=1.0, robin=None, beta=None):
        """-Lap(u) + beta . grad(u) + c u with du/dn + alpha u = 0 on the boundary (the weak form's natural
        condition) on the tensor-product space with the given per-axis knot vectors.  The defaults (c = 1,
        no Robin term, no convection) are the operator `assembly_2d` builds (/root/reference/sources/
        matrix_assembler.py:82-179), K(x)M + M(x)(K+M) [2-D] / K(x)M(x)M + M(x)K(x)M + M(x)M(x)(K+M) [3-D].

        robin: None, or one pair (alpha_lo, alpha_hi) per axis: alpha int_F u v ds on the faces
        x_a = T_a[p] and x_a = T_a[n_a].  On an open knot vector only the first (last) basis function
        is non-zero there, with value 1, so the face term is (alpha e e^T) (x) M_others: one diagonal
        entry of K_a.  c M(x)..(x)M goes into the last K as K + c M.  Both keep the Kronecker-sum
        form and change no interior row.  c >= 0, alpha >= 0, and c > 0 or some alpha > 0 (otherwise
        the operator is singular): ValueError.

        beta: None, or one constant velocity component per axis: int (beta . grad u) v = sum_a beta_a
        G_a (x) M_others with the 1-D advection band G_a (`bsplines.assemble_1d_advection`), added into
        K_a.  The operator is then not symmetric; its symmetric part must be positive definite (checked
        from d 1-D eigenproblems, `symmetric_part_lmin`), otherwise ValueError: an inflow face
        (beta . n < 0) needs enough of alpha or c."""
        from . import setup_device as sd
        c, robin = reaction_robin(c, robin, len(knots))
        beta = convection_beta(beta, len(knots))
        asm = sd.assemble_1d_bands if sd.enabled() else bs.assemble_1d_bands
        MK = [asm(p, T) for T in knots]
        Ms = [m for m, k in MK]
        Ks = [k for m, k in MK]
        if robin is not None:
            for a, (lo, hi) in enumerate(robin):
                Ks[a] = Ks[a].copy()
                Ks[a][0, p] += lo
                Ks[a][-1, p] += hi
        if beta is not None:
            lengths = [float(T[-1] - T[0]) for T in knots]
            lam = symmetric_part_lmin(Ks, Ms, c, beta, lengths)
            if not lam > 0.0:
                raise ValueError(
                    "the symmetric part of -Lap u + beta.grad u + c u with these Robin terms is not positive "
                    "definite (lambda_min = %.3e): an inflow face (beta . n < 0) needs alpha + c large enough "
                    "(e.g. alpha >= |beta_a| / 2 there)" % lam)
            adv = sd.assemble_1d_advection if sd.enabled() else bs.assemble_1d_advection
            for a, b in enumerate(beta):
                if b != 0.0:
                    Ks[a] = Ks[a] + b * adv(p, knots[a])
        Ks[-1] = Ks[-1] + c * Ms[-1]
        A = cls(Ms, Ks)
        A.mass_bands = Ms
        return A

    def _toeplitz(self):
        """Interior (Toeplitz) rows of the axis-1 and axis-2 bands: host arrays handed to the 3-D
        TMA kernel, which then takes those coefficients from the kernel-parameter constant bank.
        Rows [lo, hi) of BOTH bands of an axis are bit-identical to the middle row (uniform knots:
        all rows except the first/last 2p)."""
        if getattr(self, "_toep", None) is None:
            W = 2 * self.P + 1
            coef = np.zeros((self.ndim, 2, W))
            rng = np.zeros(2 * self.ndim, dtype=np.int32)
            for a in range(self.ndim):
                m = self.Ms[a]
                k = self.Ks[a] if self.Ks is not None else np.zeros_like(m)
                n = m.shape[0]
                mid = n // 2
                same = np.all(m == m[mid], axis=1) & np.all(k == k[mid], axis=1)
                lo = mid
                while lo > 0 and same[lo - 1]:
                    lo -= 1
                hi = mid + 1
                while hi < n and same[hi]:
                    hi += 1
                coef[a, 0], coef[a, 1] = m[mid], k[mid]
                rng[2 * a], rng[2 * a + 1] = lo, hi
            self._toep = (np.ascontiguousarray(coef), rng)
        return self._toep

    def _bands(self, V):
        """Device band pointers for the rows a space owns (axis-1 rows are the slab's)."""
        key = (V.starts[0], V.ends[0], str(V.device))
        if key not in self._dev:
            def up(bands):
                out = []
                for a, b_ in enumerate(bands):
                    loc = b_[V.starts[0]:V.ends[0] + 1] if a == 0 else b_
                    out.append(torch.as_tensor(np.ascontiguousarray(loc), device=V.device))
                return out
            m = up(self.Ms)
            k = up(self.Ks) if self.Ks is not None else [None] * self.ndim
            self._dev[key] = (m, k)
        return self._dev[key]

    def apply(self, x, y, epi=EPI_STORE, b=None, omega=0.0, dot_ptr=None, dot_with=None):
        """y = epilogue(A x) in one fused pass; optional fused reduction into *dot_ptr.
        dot_with (3-D, EPI_AXPY): request *dot_ptr = y . dot_with instead of the epilogue's own
        reduction; returns True when the kernel did it (False: the caller computes the dot)."""
        V = x.space
        self._fused_dot = False
        assert V.npts == self.npts, (V.npts, self.npts)
        ctx = DeviceContext.get(V.device)
        m, k = self._bands(V)
        kp = [t.data_ptr() if t is not None else None for t in k]
        L = _lib.lib()
        bp = b.ptr if b is not None else None
        # algorithmic bytes: read x, write y (+ read b for the fused residual/Jacobi epilogues)
        nbytes = (16 if (epi == EPI_STORE or bp is None) else 24) * V.local_size
        slab = V.slab
        n1 = V.local_shape[0]
        P = self.P
        if (slab is not None and slab.size > 1 and self.ndim == 3 and dot_ptr is None
                and n1 >= 4 * P and slab.overlap):
            # Slab-partitioned 3-D pass without a fused reduction: the halo exchange runs on the
            # communication stream WHILE the planes that need no ghost data are computed; the P
            # planes next to each neighbour follow once the ghosts have arrived.
            lo = P if slab.rank > 0 else 0
            hi = P if slab.rank < slab.size - 1 else 0
            ev = slab.exchange_async(x)
            inner = nbytes * (n1 - lo - hi) // n1
            with profiling.region("kron_matvec_3d", inner):
                self._launch(L, V, x, y, bp, m, kp, epi, omega, None, ctx, lo, n1 - hi)
            torch.cuda.current_stream().wait_event(ev)
            with profiling.region("kron_matvec_3d_edge", nbytes - inner, launches=(lo > 0) + (hi > 0)):
                if lo:
                    self._launch(L, V, x, y, bp, m, kp, epi, omega, None, ctx, 0, lo)
                if hi:
                    self._launch(L, V, x, y, bp, m, kp, epi, omega, None, ctx, n1 - hi, n1)
            return
        if slab is not None:
            slab.exchange(x)
        with profiling.region("kron_matvec_%dd" % self.ndim, nbytes + (8 * V.local_size if dot_with is not None else 0)):
            self._launch(L, V, x, y, bp, m, kp, epi, omega, dot_ptr, ctx, dot_with=dot_with)
        return self._fused_dot

    def _launch(self, L, V, x, y, bp, m, kp, epi, omega, dot_ptr, ctx, z0=0, z1=None, dot_with=None):
        """One kernel launch for the output planes [z0, z1) of the slab (default: all of them).  A
        sub-range is the same kernel on shifted pointers: the planes outside it are ghost planes of
        the sub-problem (glo + z0 below, ghi + n1 - z1 above)."""
        if self.ndim == 2:
            n1, n2 = V.local_shape
            assert z0 == 0 and z1 is None
            coef, rng = self._toeplitz()
            rng = rng.copy()
            # axis-1 rows are the slab's: shift the global interior range to local row numbers
            rng[0] = max(0, int(rng[0]) - V.starts[0])
            rng[1] = max(int(rng[0]), min(n1, int(rng[1]) - V.starts[0]))
            _lib.check(L.poms_kron_matvec_2d_ex(
                x.ptr, y.ptr, bp, n1, n2, x.ld, V.glo, V.ghi, self.P, self.form,
                m[0].data_ptr(), kp[0], m[1].data_ptr(), kp[1], epi, float(omega), dot_ptr,
                ctx.ws_ptr, _stream(), coef.ctypes.data, rng.ctypes.data), "poms_kron_matvec_2d")
        else:
            n1, n2, n3 = V.local_shape
            z1 = n1 if z1 is None else z1
            coef, rng = self._toeplitz()
            rng = rng.copy()
            # axis-1 rows are the slab's: shift the global interior range to local row numbers
            rng[0] = max(0, int(rng[0]) - V.starts[0] - z0)
            rng[1] = max(int(rng[0]), min(z1 - z0, int(rng[1]) - V.starts[0] - z0))
            W = 2 * self.P + 1
            off = 8 * z0 * x.pld                        # bytes from plane 0 to plane z0
            import ctypes
            fused = ctypes.c_int(0)
            _lib.check(L.poms_kron_matvec_3d_dotv(
                x.ptr + off, y.ptr + off, bp + off if bp is not None else None, z1 - z0, n2, n3,
                x.ld, x.pld, V.glo + z0, V.ghi + n1 - z1, self.P, self.form,
                m[0].data_ptr() + 8 * z0 * W, kp[0] + 8 * z0 * W if kp[0] is not None else None,
                m[1].data_ptr(), kp[1], m[2].data_ptr(), kp[2], epi,
                float(omega), dot_ptr, ctx.ws_ptr, _stream(), coef.ctypes.data, rng.ctypes.data,
                dot_with.ptr + off if dot_with is not None else None, ctypes.byref(fused)),
                "poms_kron_matvec_3d_dotv")
            self._fused_dot = bool(fused.value)

    def dot(self, v):
        out = StencilVector(v.space, zero=False)
        self.apply(v, out)
        return out

    def jacobi_first(self, x, b, omega, dot_ptr):
        """x = omega * b / diag(A) (+ *dot_ptr = x.x): jacobi() and the first damped-Jacobi
        sweep from a zero guess."""
        V = b.space
        ctx = DeviceContext.get(V.device)
        m, k = self._bands(V)
        kp = [t.data_ptr() if t is not None else None for t in k]
        L = _lib.lib()
        if self.ndim == 2:
            n1, n2 = V.local_shape
            _lib.check(L.poms_jacobi_first_2d(
                x.ptr, b.ptr, n1, n2, b.ld, self.P, self.form, m[0].data_ptr(), kp[0],
                m[1].data_ptr(), kp[1], float(omega), dot_ptr, ctx.ws_ptr, _stream()),
                "poms_jacobi_first_2d")
        else:
            n1, n2, n3 = V.local_shape
            _lib.check(L.poms_jacobi_first_3d(
                x.ptr, b.ptr, n1, n2, n3, b.ld, b.pld, self.P, self.form, m[0].data_ptr(), kp[0],
                m[1].data_ptr(), kp[1], m[2].data_ptr(), kp[2], float(omega), dot_ptr,
                ctx.ws_ptr, _stream()), "poms_jacobi_first_3d")

    # host-side helpers (setup / tests)
    def diagonal_host(self):
        P = self.P
        d = 0.0
        if self.form == FORM_SINGLE:
            d = np.ones(())
            for m in self.Ms:
                d = np.multiply.outer(d, m[:, P])
            return d
        for a in range(self.ndim):
            t = np.ones(())
            for c in range(self.ndim):
                t = np.multiply.outer(t, (self.Ks[c] if c == a else self.Ms[c])[:, P])
            d = d + t
        return d

    def __getitem__(self, key):
        """A[i1, i2(, i3), k1, k2(, k3)] (e.g. the diagonal A[i1,i2,0,0] read by
        /root/reference/sources/solvers.py:158,213)."""
        idx, off = key[:self.ndim], key[self.ndim:]
        P = self.P
        if self.form == FORM_SINGLE:
            return float(np.prod([m[i, k + P] for m, i, k in zip(self.Ms, idx, off)]))
        tot = 0.0
        for a in range(self.ndim):
            t = 1.0
            for c in range(self.ndim):
                t *= (self.Ks[c] if c == a else self.Ms[c])[idx[c], off[c] + P]
            tot += t
        return tot

    def to_stencil_array(self):
        """Full (n1, .., nd, 2P+1, .., 2P+1) stencil of the operator (host, tests)."""
        d = self.ndim

        def outer(bands):
            t = np.ones(())
            for a, bnd in enumerate(bands):
                shp = [1] * (2 * d)
                shp[a], shp[d + a] = bnd.shape
                t = t * bnd.reshape(shp)
            return t
        if self.form == FORM_SINGLE:
            return outer(self.Ms)
        tot = 0.0
        for a in range(d):
            tot = tot + outer([self.Ks[c] if c == a else self.Ms[c] for c in range(d)])
        return tot
