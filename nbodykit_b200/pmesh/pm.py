"""
`pmesh.pm` surface used by the FFTPower path (SURVEY.md §8b), backed by libnbk_b200.so.

  ParticleMesh(BoxSize, Nmesh, dtype, comm)   base/mesh.py:50
     .paint(pos, mass=, resampler=, transform=, hold=, out=)   source/mesh/catalog.py:287-296
     .decompose(pos, smoothing) -> Layout(.recvlength, .exchange)           :271-284
     .affine.shift(0.5), .create(type=, value=), .reshape(Nmesh=), .x/.k/.w coordinate lists
  RealField / ComplexField: device-resident fields with r2c/c2r, apply, slabs, csum/cmean ...

Decomposition (P = comm.size GPUs): the real field is split in x slabs [x_start, x_start+x_n);
the complex field that r2c leaves behind is split in y slabs and stored transposed,
[y_n][Nx][Nzc] (`ComplexField.transposed`), exactly one NCCL all-to-all per transform.
With P == 1 the complex field is the plain [Nx][Ny][Nzc] array.
"""
import ctypes
import math

import numpy
import torch

from .. import _lib
from .._lib import F4, F8, check, darr, iarr, lib, stage
from . import window as _window

_TORCH_REAL = {"f4": torch.float32, "f8": torch.float64}
_TORCH_CPLX = {"f4": torch.complex64, "f8": torch.complex128}
_CODE = {"f4": F4, "f8": F8}


def _real_typestr(dtype):
    """'f4'/'f8' for any real or complex dtype spec"""
    dt = numpy.dtype(dtype)
    if dt.kind == "c":
        return "f4" if dt.itemsize == 8 else "f8"
    if dt.kind == "f" and dt.itemsize in (4, 8):
        return "f%d" % dt.itemsize
    raise TypeError("unsupported mesh dtype %s" % str(dtype))


def _stream():
    return ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)


def _ptr(t):
    return ctypes.c_void_p(t.data_ptr() if t is not None else None)


def _is_pow2(n):
    return n > 0 and (n & (n - 1)) == 0


def current_device():
    if not torch.cuda.is_available():
        raise _lib.NbkError("nbodykit_b200 needs a CUDA device (sm_100a); there is no CPU fallback")
    return torch.device("cuda", torch.cuda.current_device())


def as_device_tensor(a, dtype=None, device=None):
    """numpy array / torch tensor / scalar column -> contiguous device tensor (no copy if already there)"""
    device = device or current_device()
    if isinstance(a, torch.Tensor):
        t = a
    else:
        a = numpy.ascontiguousarray(a)
        t = torch.from_numpy(a)
    if dtype is not None and t.dtype != dtype:
        t = t.to(dtype)
    return t.to(device, non_blocking=True).contiguous()


class Affine(object):
    """pm.affine: grid = pos * scale + translate; .shift(s) adds s cells (catalog.py:292)"""

    def __init__(self, ndim, scale, translate=0.0, period=None):
        self.ndim = ndim
        self.scale = scale
        self.translate = translate
        self.period = period

    def shift(self, amount):
        return Affine(self.ndim, self.scale, self.translate + amount, self.period)


class Layout(object):
    """result of pm.decompose: which local particles go to which rank (ghosts duplicated)"""

    def __init__(self, comm, indices, sendcounts, recvcounts):
        self.comm = comm
        self.indices = indices            # device int64: local particle index per send slot, grouped by dest
        self.sendcounts = sendcounts      # python ints, len P
        self.recvcounts = recvcounts
        self.sendlength = int(sum(sendcounts))
        self.recvlength = int(sum(recvcounts))

    def exchange(self, data):
        """route a per-particle column (n, ...) -> (recvlength, ...).  Returns a new device tensor."""
        t = as_device_tensor(data) if not isinstance(data, torch.Tensor) else data
        if self.comm.size == 1 and self.indices is None:
            return t
        send = t.index_select(0, self.indices)
        if self.comm.size == 1:
            return send
        out = torch.empty((self.recvlength,) + tuple(t.shape[1:]), dtype=t.dtype, device=t.device)
        self.comm.all_to_all_single(out, send, list(self.recvcounts), list(self.sendcounts))
        return out


_PEER_STAGE_CACHE = {}


_COPY_STREAMS = {}


def _copy_streams(device):
    """two side streams per device for the NVLink copies of the pipelined slab exchange"""
    key = str(device)
    if key not in _COPY_STREAMS:
        _COPY_STREAMS[key] = [torch.cuda.Stream(device=device) for _ in range(2)]
    return _COPY_STREAMS[key]


def _push_chunks(x_n):
    """parts the slab exchange of r2c is pipelined in (NBK_FFT_PUSH_CHUNKS, default 4; 1 = y pass, then all copies)"""
    import os
    try:
        n = int(os.environ.get("NBK_FFT_PUSH_CHUNKS", "4"))
    except ValueError:
        n = 4
    return max(1, min(n, int(x_n)))


def _transpose_mode():
    """how the slab transpose of a distributed FFT crosses NVLink: 'push' (line pass into send blocks + one strided bulk
    copy per peer, default) or 'stores' (the line pass stores every 128..256-byte run straight into the peer's field);
    NBK_FFT_TRANSPOSE_MODE selects"""
    import os
    m = os.environ.get("NBK_FFT_TRANSPOSE_MODE", "push")
    return m if m in ("push", "stores") else "push"


class SlabLayout(object):
    """device-side routing plan (nbk_route_count): compact list of the particles with REMOTE destination slabs
    (index | bitmask << 32).  Local particles are never moved -- `route()` returns only what arrives from other
    ranks; `exchange()` keeps the pmesh contract (local + received in one array)."""

    def __init__(self, pm, n, ghosts, sendcounts, recvcounts):
        self.pm = pm
        self.comm = pm.comm
        self.n = n
        self.ghosts = ghosts
        self.sendcounts = sendcounts
        self.recvcounts = recvcounts
        self.sendlength = int(sum(sendcounts))
        self.recvlength = n + int(sum(recvcounts))     # pmesh semantics: what this rank will paint

    def route(self, pos, mass=None, want_index=False):
        """(received positions, received masses | None): copies for remote slabs travel in one all-to-all per column.
        want_index=True additionally returns the source row of every SENT row (for `gather_back`)."""
        P = self.comm.size
        dev = pos.device
        nsend, nrecv = int(sum(self.sendcounts)), int(sum(self.recvcounts))
        spos = torch.empty((nsend, 3), dtype=pos.dtype, device=dev)
        smass = torch.empty(nsend, dtype=mass.dtype, device=dev) if mass is not None else None
        sidx = torch.empty(nsend, dtype=torch.int64, device=dev) if want_index else None
        if nsend:
            off = torch.tensor([0] + list(numpy.cumsum(self.sendcounts)[:-1]), dtype=torch.int64, device=dev)
            cur = torch.zeros(P, dtype=torch.int64, device=dev)
            with stage("route_scatter"):
                check(lib().nbk_route_scatter(_ptr(pos), F4 if pos.dtype == torch.float32 else F8, _ptr(mass),
                                              (F4 if mass.dtype == torch.float32 else F8) if mass is not None else F8,
                                              _ptr(self.ghosts), int(self.ghosts.shape[0]), P, _ptr(off), _ptr(cur), _ptr(spos),
                                              _ptr(smass), _ptr(sidx), _stream()), "nbk_route_scatter")
        rpos = torch.empty((nrecv, 3), dtype=pos.dtype, device=dev)
        with stage("route_alltoall"):
            self.comm.all_to_all_single(rpos, spos, list(self.recvcounts), list(self.sendcounts))
            rmass = None
            if mass is not None:
                rmass = torch.empty(nrecv, dtype=mass.dtype, device=dev)
                self.comm.all_to_all_single(rmass, smass, list(self.recvcounts), list(self.sendcounts))
        if want_index:
            return rpos, rmass, sidx
        return rpos, rmass

    def gather_back(self, values, sidx, out, mode="sum"):
        """reverse of `route` for per-row results: `values[k]` was computed by the destination for the k-th row it
        received; they travel back and are combined into out[source row]: ADDED with mode='sum' (pmesh
        `layout.gather(mode='sum')`), or the minimum kept with mode='min' (`layout.gather(mode=numpy.fmin)`)"""
        if mode not in ("sum", "min"):
            raise ValueError("gather_back: mode must be 'sum' or 'min', not %r" % (mode,))
        nsend = int(sum(self.sendcounts))
        back = torch.empty(nsend, dtype=values.dtype, device=values.device)
        self.comm.all_to_all_single(back, values.contiguous(), list(self.sendcounts), list(self.recvcounts))
        if nsend:
            if mode == "sum":
                out.index_add_(0, sidx, back.to(out.dtype))
            else:
                out.index_reduce_(0, sidx, back.to(out.dtype), "amin")
        return out

    def exchange(self, data):
        t = as_device_tensor(data) if not isinstance(data, torch.Tensor) else data
        P = self.comm.size
        parts, counts = [], []
        gidx, gmask = self.ghosts & 0xffffffff, self.ghosts >> 32
        for r in range(P):
            idx = gidx[((gmask >> r) & 1) != 0]
            parts.append(t.index_select(0, idx))
            counts.append(int(idx.numel()))
        send = torch.cat(parts) if parts else t[:0]
        recv = torch.empty((int(sum(self.recvcounts)),) + tuple(t.shape[1:]), dtype=t.dtype, device=t.device)
        self.comm.all_to_all_single(recv, send, list(self.recvcounts), counts)
        return torch.cat([t, recv])


class ParticleMesh(object):
    def __init__(self, BoxSize, Nmesh, dtype="f4", comm=None, np=None, plan_method=None, resampler="cic"):
        from .. import CurrentMPIComm
        self.comm = comm if comm is not None else CurrentMPIComm.get()
        Nm = numpy.array(Nmesh)
        ndim = 3 if Nm.ndim == 0 else len(Nm)
        if ndim != 3:
            raise NotImplementedError("only 3-D meshes are supported by the B200 FFTPower path")
        self.Nmesh = numpy.empty(3, dtype="i8")
        self.Nmesh[:] = Nmesh
        self.BoxSize = numpy.empty(3, dtype="f8")
        self.BoxSize[:] = BoxSize
        self.ndim = 3
        self._dtype_in = numpy.dtype(dtype)
        # complex dtype ('c8'/'c16', pmesh then transforms c2c and keeps all N^3 modes: fftpower.py:572,
        # convpower/catalog.py:151-176).  The configuration-space fields of this path are real-valued: they are
        # STORED as real arrays, and the full spectrum is the Hermitian completion of the r2c result
        # (nbk_hermitian_expand) -- identical values, a third of the memory traffic of a c2c transform.
        self.cplx = self._dtype_in.kind == "c"
        if self.cplx and self.comm.size > 1:
            raise NotImplementedError(
                "complex-typed meshes (dtype='c8'/'c16') are single-GPU here; on several GPUs use dtype='f4'/'f8' "
                "(ConvolvedFFTPower reproduces the full-mesh result from the compressed field on any number of GPUs)")
        self.dtype = self._dtype_in if self.cplx else numpy.dtype(_real_typestr(dtype))
        self.typestr = _real_typestr(dtype)
        self.resampler = _window.FindResampler(resampler)
        self.affine = Affine(3, self.Nmesh / self.BoxSize, 0.0, self.Nmesh.copy())

        P = self.comm.size
        self.np = [P]
        Nx, Ny, Nz = [int(v) for v in self.Nmesh]
        if P > 1 and (Nx % P or Ny % P):
            raise ValueError("Nmesh[0] and Nmesh[1] must be divisible by the number of GPUs (%d)" % P)
        self.x_n = Nx // P
        self.x_start = self.comm.rank * self.x_n
        self.y_n = Ny // P
        self.y_start = self.comm.rank * self.y_n
        self.Nzc = Nz if self.cplx else Nz // 2 + 1      # stored length of the last axis of a ComplexField
        self.transposed = P > 1
        # power-of-two meshes use the transform of fft.cu (NVLink peer transpose when P > 1); any other side goes
        # through the mixed-radix transform of fft_mixed.cu (sides 2^a 3^b 5^c 7^d, every side even; others raise)
        self.mixed_fft = not all(_is_pow2(n) for n in (Nx, Ny, Nz))
        self._nmesh_c = iarr(self.Nmesh)
        self._box_c = darr(self.BoxSize)
        self._coords = {}

    # ---- shapes
    @property
    def real_shape(self):
        return (self.x_n, int(self.Nmesh[1]), int(self.Nmesh[2]))

    @property
    def complex_shape(self):
        if self.transposed:
            return (self.y_n, int(self.Nmesh[0]), self.Nzc)
        return (int(self.Nmesh[0]), int(self.Nmesh[1]), self.Nzc)

    def reshape(self, Nmesh=None, BoxSize=None, dtype=None):
        if Nmesh is None:
            Nmesh = self.Nmesh
        if BoxSize is None:
            BoxSize = self.BoxSize
        if dtype is None:
            dtype = self.dtype
        Nm = numpy.empty(3, dtype="i8")
        Nm[:] = Nmesh
        if (Nm == self.Nmesh).all() and numpy.allclose(BoxSize, self.BoxSize) and numpy.dtype(dtype) == numpy.dtype(self.dtype):
            return self
        return ParticleMesh(BoxSize=BoxSize, Nmesh=Nm, dtype=dtype, comm=self.comm)

    def create(self, type=None, base=None, value=None, mode=None):
        type = _typestr_to_type(type if type is not None else mode)
        f = type(self)
        if value is not None:
            f[...] = value
        return f

    # ---- coordinates (host numpy, float32 by default: SURVEY B.5 / A12)
    def create_coords(self, field_type, return_indices=False, dtype="f4"):
        """three broadcastable host arrays for this rank's part of a real / complex field"""
        ct = numpy.dtype(dtype).type
        N = [int(v) for v in self.Nmesh]
        out, ind = [], []
        if field_type in ("real", RealField):
            ranges = [numpy.arange(self.x_start, self.x_start + self.x_n), numpy.arange(N[1]), numpy.arange(N[2])]
            for d in range(3):
                i = ranges[d].copy()
                i[i >= (N[d] + 1) // 2] -= N[d]      # wrapped to [-L/2, L/2) (SURVEY A9)
                x = i.astype(ct) * ct(self.BoxSize[d] / N[d])
                shape = [1, 1, 1]; shape[d] = len(x)
                out.append(x.reshape(shape)); ind.append(ranges[d].reshape(shape))
        else:
            if self.transposed:
                # stored [y_n][Nx][Nzc]: the iteration axis 0 is y -- coordinate arrays follow STORAGE order
                ranges = [numpy.arange(N[0]), numpy.arange(self.y_start, self.y_start + self.y_n), numpy.arange(self.Nzc)]
                shapes = [(1, N[0], 1), (self.y_n, 1, 1), (1, 1, self.Nzc)]
            else:
                ranges = [numpy.arange(N[0]), numpy.arange(N[1]), numpy.arange(self.Nzc)]
                shapes = [(N[0], 1, 1), (1, N[1], 1), (1, 1, self.Nzc)]
            for d in range(3):
                j = ranges[d].copy()
                j[j >= (N[d] + 1) // 2] -= N[d]
                k = j.astype(ct) * ct(2 * numpy.pi / self.BoxSize[d])
                out.append(k.reshape(shapes[d])); ind.append(ranges[d].reshape(shapes[d]))
        return (out, ind) if return_indices else out

    @property
    def x(self):
        return self.create_coords("real")

    @property
    def k(self):
        return self.create_coords("complex")

    # ---- particle routing (source/mesh/catalog.py:271-284)
    def decompose(self, pos, smoothing=None, transform=None):
        """destination slab(s) of every particle: every rank whose x planes lie within `smoothing`
        cells of the particle (ghosts duplicated, periodic)."""
        P = self.comm.size
        if smoothing is None:
            smoothing = 0.5 * self.resampler.support
        if P == 1:
            n = int(pos.shape[0])
            return Layout(self.comm, None, [n], [n])
        pos = pos if isinstance(pos, torch.Tensor) else torch.as_tensor(numpy.asarray(pos))
        if pos.is_cuda:
            return self._decompose_device(pos, float(smoothing))
        Nx = int(self.Nmesh[0])
        gx = pos[:, 0].to(torch.float64) * float(self.Nmesh[0] / self.BoxSize[0])
        lo = torch.floor(gx - smoothing).to(torch.int64)
        hi = torch.floor(gx + smoothing).to(torch.int64)
        # slabs touched by cells lo..hi (at most 2 when smoothing < x_n, the only supported case)
        if 2 * smoothing + 1 > self.x_n:
            raise ValueError("x slab of %d planes is thinner than the window reach" % self.x_n)
        r_lo = torch.remainder(lo, Nx) // self.x_n
        r_hi = torch.remainder(hi, Nx) // self.x_n
        idx = torch.arange(pos.shape[0], device=pos.device, dtype=torch.int64)
        dup = r_hi != r_lo
        dest = torch.cat([r_lo, r_hi[dup]])
        src = torch.cat([idx, idx[dup]])
        order = torch.argsort(dest, stable=True)
        counts = torch.bincount(dest, minlength=P).cpu().tolist()
        recv = self.comm.alltoall(counts)
        return Layout(self.comm, src[order], counts, recv)

    # ---- NVLink peer-memory staging for the slab transpose (P > 1)
    def _peer_stage(self):
        """(local staging tensor viewed as this rank's transposed complex field, ctypes array of the P peer
        pointers, symmetric-memory handle) -- allocated collectively at the first distributed transform.  None when
        symmetric memory is unavailable: the transform then goes through pack + NCCL all-to-all + unpack."""
        if hasattr(self, "_stage"):
            return self._stage
        self._stage = None
        import os
        if self.comm.size == 1 or os.environ.get("NBK_FFT_TRANSPOSE", "peer") != "peer":
            return None
        # one staging buffer per (communicator, field shape, precision): FFTPower builds a fresh ParticleMesh per
        # call, and a symmetric-memory rendezvous costs tens of milliseconds
        key = (id(self.comm), tuple(self.complex_shape), self.typestr)
        if key in _PEER_STAGE_CACHE:
            self._stage = _PEER_STAGE_CACHE[key]
            return self._stage
        try:
            import torch.distributed as dist
            import torch.distributed._symmetric_memory as symm_mem
            dev = current_device()
            nreal = 2 * int(numpy.prod(self.complex_shape))
            buf = symm_mem.empty(nreal, dtype=_TORCH_REAL[self.typestr], device=dev)
            group = getattr(self.comm, "group", None) or dist.group.WORLD
            hdl = symm_mem.rendezvous(buf, group.group_name)
            ptrs = (ctypes.c_void_p * self.comm.size)(*[int(p) for p in hdl.buffer_ptrs])
            view = torch.view_as_complex(buf.view(-1, 2)).view(self.complex_shape)
            ok = torch.ones(1, device=dev)
            self.comm.allreduce_tensor(ok)                     # every rank got here
            self._stage = (view, ptrs, hdl)
            _PEER_STAGE_CACHE[key] = self._stage
        except Exception as e:   # noqa: BLE001  (any failure -> NCCL path, still on the GPU)
            import logging
            logging.getLogger("ParticleMesh").warning("peer-memory transpose unavailable (%s); using NCCL all-to-all", e)
            self._stage = None
            _PEER_STAGE_CACHE[key] = None
        return self._stage

    def _decompose_device(self, pos, smoothing):
        """routing plan for device-resident positions: one kernel pass, one tiny all-to-all of the counts"""
        P = self.comm.size
        n = int(pos.shape[0])
        if pos.dtype not in (torch.float32, torch.float64):
            pos = pos.to(torch.float64)
        pos = pos.contiguous()
        ghosts = torch.empty(max(n, 1), dtype=torch.int64, device=pos.device)    # capacity; only the entries written are read
        counts = torch.zeros(P + 1, dtype=torch.int64, device=pos.device)
        with stage("route_count"):
            check(lib().nbk_route_count(_ptr(pos), F4 if pos.dtype == torch.float32 else F8, n, smoothing, self._box_c,
                                        self._nmesh_c, P, self.comm.rank, _ptr(counts), _ptr(ghosts), _stream()),
                  "nbk_route_count")
        c = [int(v) for v in counts.cpu().tolist()]
        sendcounts, nlist = c[:P], c[P]
        recvcounts = self.comm.alltoall_ints(sendcounts)
        return SlabLayout(self, n, ghosts[:nlist], sendcounts, recvcounts)

    # ---- paint (source/mesh/catalog.py:287,295-296)
    def paint(self, pos, mass=1.0, resampler=None, transform=None, hold=False, gradient=None, layout=None, out=None,
              method=None):
        if gradient is not None:
            raise NotImplementedError("gradient painting is not part of the FFTPower path")
        if out is None:
            out = RealField(self)
            hold = False
        if not isinstance(out, RealField):
            raise TypeError("paint: `out` must be a RealField")
        res = self.resampler if resampler is None else _window.FindResampler(resampler)
        if res.code is None:
            raise NotImplementedError("no CUDA scatter kernel for window '%s'" % res.name)
        shift = 0.0
        if transform is not None:
            shift = float(numpy.atleast_1d(transform.translate - self.affine.translate).ravel()[0])
        if layout is not None:
            pos = layout.exchange(pos)
            if not numpy.isscalar(mass):
                mass = layout.exchange(mass)
        dev = out.value.device
        p = as_device_tensor(pos, device=dev)
        if p.dtype not in (torch.float32, torch.float64):
            p = p.to(torch.float64)
        if p.ndim != 2 or p.shape[1] != 3:
            raise ValueError("paint: position must have shape (n, 3)")
        m = None
        scale_after = None
        if numpy.isscalar(mass):
            if float(mass) != 1.0:
                scale_after = float(mass)
        else:
            m = as_device_tensor(mass, device=dev)
            if m.dtype not in (torch.float32, torch.float64):
                m = m.to(torch.float64)
            if m.shape[0] != p.shape[0]:
                raise ValueError("paint: mass and position length mismatch")
        if scale_after is not None:
            if not hold:
                out[...] = 0
            target = RealField(self)
            self._scatter(p, m, res, shift, target, None, method, clear=True)
            out.axpy(target, scale_after)
        else:
            # hold=False: the tiled path zeroes the mesh inside its bucketing pass, the direct path after a fill
            self._scatter(p, m, res, shift, out, None, method, clear=not hold)
        return out

    def paint_interlaced(self, pos, mass, resampler, out1, out2, method=None, hold=True):
        """both meshes of the interlaced branch (catalog.py:289-296) in one pass over the particles"""
        res = _window.FindResampler(resampler)
        if res.code is None:
            raise NotImplementedError("no CUDA scatter kernel for window '%s'" % res.name)
        dev = out1.value.device
        p = as_device_tensor(pos, device=dev)
        if p.dtype not in (torch.float32, torch.float64):
            p = p.to(torch.float64)
        m = None
        if mass is not None and not numpy.isscalar(mass):
            m = as_device_tensor(mass, device=dev)
            if m.dtype not in (torch.float32, torch.float64):
                m = m.to(torch.float64)
        self._scatter(p, m, res, 0.0, out1, out2, method, clear=not hold)

    # below this many particles per mesh cell the per-tile overhead of the tiled path outweighs its gain
    TILED_MIN_OCCUPANCY = 0.02

    def _scatter(self, p, m, res, shift, out1, out2, method=None, clear=False):
        """dispatch to the tile-sorted shared-memory path or to the direct REDG path.
        method: None (choose), 'tiled', 'direct'.  clear: zero the mesh(es) first (hold=False)"""
        L = lib()
        n = int(p.shape[0])
        pcode = F4 if p.dtype == torch.float32 else F8
        mcode = (F4 if m.dtype == torch.float32 else F8) if m is not None else F8
        code = _CODE[self.typestr]
        ok = bool(L.nbk_paint_tiled_supported(self._nmesh_c, self.x_n, res.code)) and shift in (0.0, 0.5)
        if method == 'tiled' and not ok:
            raise ValueError("the tiled paint path needs mesh sides that are multiples of 16 (>= 32)")
        if method is None:
            cells = float(self.x_n) * float(self.Nmesh[1]) * float(self.Nmesh[2])
            method = 'tiled' if (ok and n >= self.TILED_MIN_OCCUPANCY * cells and n >= 100000) else 'direct'
        if method == 'tiled':
            nbytes = int(L.nbk_paint_tiled_workspace(n, pcode, mcode if m is not None else 0, self._nmesh_c, self.x_n))
            work = torch.empty(nbytes, dtype=torch.uint8, device=p.device)
            with stage("paint"):
                check(L.nbk_paint_tiled(_ptr(p), pcode, n, _ptr(m), mcode, res.code, float(shift), self._box_c,
                                        self._nmesh_c, self.x_start, self.x_n, _ptr(out1.value),
                                        _ptr(out2.value) if out2 is not None else None, code, _ptr(work), nbytes,
                                        1 if clear else 0, _stream()), "nbk_paint_tiled")
            return
        if clear:
            out1[...] = 0
            if out2 is not None:
                out2[...] = 0
        with stage("paint"):
            if out2 is None:
                check(L.nbk_paint(_ptr(p), pcode, n, _ptr(m), mcode, res.code, float(shift), self._box_c, self._nmesh_c,
                                  self.x_start, self.x_n, _ptr(out1.value), code, _stream()), "nbk_paint")
            else:
                check(L.nbk_paint_interlaced(_ptr(p), pcode, n, _ptr(m), mcode, res.code, self._box_c, self._nmesh_c,
                                             self.x_start, self.x_n, _ptr(out1.value), _ptr(out2.value), code,
                                             _stream()), "nbk_paint_interlaced")

    def cell_index(self, pos, resampler="cic", shift=0.0):
        """wrapped leftmost stencil cell of every particle, (n,3) int32 device tensor"""
        res = _window.FindResampler(resampler)
        p = as_device_tensor(pos)
        out = torch.empty((p.shape[0], 3), dtype=torch.int32, device=p.device)
        check(lib().nbk_cell_index(_ptr(p), F4 if p.dtype == torch.float32 else F8, p.shape[0], res.code,
                                   float(shift), self._box_c, self._nmesh_c, _ptr(out), _stream()), "nbk_cell_index")
        return out


class _Slabs(object):
    """field.slabs: iterate over planes of the first stored axis; .x / .i / .optx give per-plane coords"""

    def __init__(self, field):
        self.field = field

    def __len__(self):
        return self.field.value.shape[0]

    def __iter__(self):
        for i in range(len(self)):
            yield self.field.value[i]

    def _coords(self, want_index):
        f = self.field
        kind = "real" if isinstance(f, RealField) else "complex"
        xs, ind = f.pm.create_coords(kind, return_indices=True)
        src = ind if want_index else xs
        ax0 = self._axis0()
        for i in range(len(self)):
            yield [src[d][i] if d == ax0 else src[d][0] for d in range(3)]

    def _axis0(self):
        """physical dimension that runs along the first STORED axis"""
        f = self.field
        return 1 if (isinstance(f, ComplexField) and f.pm.transposed) else 0

    @property
    def x(self):
        return self._coords(False)

    @property
    def optx(self):
        return self._coords(False)

    @property
    def i(self):
        return self._coords(True)


class Field(object):
    """base of RealField / ComplexField: a device tensor + its ParticleMesh"""

    def __init__(self, pm, value=None):
        self.pm = pm
        self.attrs = {}
        shape, tdt = self._layout(pm)
        if value is None:
            value = torch.empty(shape, dtype=tdt, device=current_device())
        self.value = value

    # -- pmesh-compatible members
    @property
    def Nmesh(self):
        return self.pm.Nmesh

    @property
    def BoxSize(self):
        return self.pm.BoxSize

    @property
    def shape(self):
        return tuple(self.value.shape)

    @property
    def cshape(self):
        N = [int(v) for v in self.pm.Nmesh]
        return tuple(N) if isinstance(self, RealField) else (N[0], N[1], self.pm.Nzc)

    @property
    def size(self):
        return self.value.numel()

    @property
    def csize(self):
        return int(numpy.prod(self.cshape))

    @property
    def slabs(self):
        return _Slabs(self)

    @property
    def x(self):
        return self.pm.create_coords("real" if isinstance(self, RealField) else "complex")

    def _flat_real(self):
        v = self.value
        return torch.view_as_real(v).reshape(-1) if v.is_complex() else v.reshape(-1)

    def __getitem__(self, idx):
        return self.value[idx]

    def __setitem__(self, idx, val):
        whole = idx is Ellipsis or (isinstance(idx, slice) and idx == slice(None))
        if whole and numpy.isscalar(val) and not isinstance(val, complex):
            flat = self._flat_real()
            if self.value.is_complex():
                # real scalar into a complex field: fill real part, zero imaginary
                if float(val) == 0.0:
                    check(lib().nbk_fill(_ptr(flat), _CODE[self.pm.typestr], flat.numel(), 0.0, _stream()), "nbk_fill")
                else:
                    self.value[...] = val
            else:
                check(lib().nbk_fill(_ptr(flat), _CODE[self.pm.typestr], flat.numel(), float(val), _stream()), "nbk_fill")
            return
        if isinstance(val, Field):
            val = val.value
        elif isinstance(val, numpy.ndarray):
            val = torch.from_numpy(val).to(self.value.device)
        self.value[idx] = val

    def __array__(self, dtype=None, copy=None):
        a = self.value.detach().cpu().numpy()
        return a.astype(dtype) if dtype is not None else a

    def numpy(self):
        return self.__array__()

    def copy(self):
        out = type(self)(self.pm, self.value.clone())
        out.attrs = dict(self.attrs)
        return out

    # -- in-place arithmetic on the whole field (kernels in csrc/core.cu)
    def scale(self, a):
        flat = self._flat_real()
        check(lib().nbk_scale(_ptr(flat), _CODE[self.pm.typestr], flat.numel(), float(a), _stream()), "nbk_scale")
        return self

    def axpy(self, other, a=1.0):
        """self += a * other"""
        flat = self._flat_real()
        o = other._flat_real()
        if o.numel() != flat.numel():
            raise ValueError("field shape mismatch")
        check(lib().nbk_axpy(_ptr(flat), _ptr(o), _CODE[self.pm.typestr], flat.numel(), float(a), _stream()), "nbk_axpy")
        return self

    def __imul__(self, a):
        if numpy.isscalar(a) and not isinstance(a, complex):
            return self.scale(a)
        self.value *= (a.value if isinstance(a, Field) else a)
        return self

    def __itruediv__(self, a):
        if numpy.isscalar(a) and not isinstance(a, complex):
            return self.scale(1.0 / a)
        self.value /= (a.value if isinstance(a, Field) else a)
        return self

    def __iadd__(self, a):
        if isinstance(a, Field):
            return self.axpy(a, 1.0)
        self.value += a
        return self

    def __isub__(self, a):
        if isinstance(a, Field):
            return self.axpy(a, -1.0)
        self.value -= a
        return self

    def csum(self):
        """collective sum of all elements (catalog.py:388)"""
        if self.value.is_complex():
            return complex(self.pm.comm.allreduce(complex(self.value.sum().item())))
        acc = torch.zeros(1, dtype=torch.float64, device=self.value.device)
        flat = self._flat_real()
        check(lib().nbk_sum(_ptr(flat), _CODE[self.pm.typestr], flat.numel(), _ptr(acc), _stream()), "nbk_sum")
        return float(self.pm.comm.allreduce(acc.item()))

    def cmean(self):
        return self.csum() / float(numpy.prod(self.cshape if isinstance(self, RealField) else self.pm.Nmesh))

    def cast(self, type=None, out=None):
        type = _typestr_to_type(type) if type is not None else self.__class__
        if isinstance(self, type):
            return self
        if issubclass(type, BaseComplexField):
            return self.r2c(out=None if out is self else out)
        return self.c2r(out=None if out is self else out)

    def apply(self, func, kind="wavenumber", out=None):
        """apply func(coords, value) plane by plane (contract: base/mesh.py:126-145).

        The reference's own window-compensation transfer functions run as one CUDA pass
        (nbk_compensate).  Any other Python callback is evaluated the way pmesh evaluates it -- as
        host NumPy code, one x-plane at a time -- because it *is* host code."""
        if out is Ellipsis or out is self:
            target = self
        elif out is None:
            target = self.copy()
        else:
            target = out
            target.value.copy_(self.value)
        name = getattr(func, "__name__", "")
        if isinstance(target, ComplexField) and kind == "circular" and name in _lib.COMP \
                and getattr(func, "__module__", "").startswith("nbodykit_b200"):
            target.compensate(name)
            return target
        if not target._apply_device(func, kind):
            target._apply_host(func, kind)
        return target

    def _coords_for(self, kind):
        """(coordinate arrays the callback gets for `kind`, physical dimension running along storage axis 0)"""
        pm = self.pm
        is_real = isinstance(self, RealField)
        coords, ind = pm.create_coords("real" if is_real else "complex", return_indices=True)
        N = [float(v) for v in pm.Nmesh]
        if kind == "index":
            use = ind
        elif kind == "relative" and is_real:
            use = coords
        elif kind == "circular" and not is_real:
            use = [(c.astype("f8") * (pm.BoxSize[d] / N[d])).astype(c.dtype) for d, c in enumerate(coords)]
        elif kind in ("wavenumber", "relative"):
            use = coords
        else:
            raise ValueError("unknown kind %s" % kind)
        return use, self.slabs._axis0()

    APPLY_PLANES = 16

    def _apply_device(self, func, kind):
        """func(coords, values) evaluated ON THE DEVICE: the callback gets torch tensors (a batch of planes of the field
        and broadcastable coordinate tensors), so callbacks written with arithmetic operators -- and the package's
        own MeshFilters (filters.py) -- never move the field out of HBM.  Returns False, leaving the field untouched,
        when the callback cannot work on device tensors (it calls NumPy functions): the host plane loop takes over."""
        use, ax0 = self._coords_for(kind)
        dev = self.value.device
        tc = [torch.from_numpy(numpy.ascontiguousarray(c)).to(dev) for c in use]
        n0 = int(self.value.shape[0])
        step = max(1, min(n0, self.APPLY_PLANES))

        def batch(i, values):
            cs = [c[i:i + step] if d == ax0 else c for d, c in enumerate(tc)]
            return func(cs, values)
        if n0 == 0:
            return True
        try:     # dry run on a copy of the first batch
            res = batch(0, self.value[0:step].clone())
            if not isinstance(res, torch.Tensor) or tuple(res.shape) != tuple(self.value[0:step].shape):
                return False
        except Exception:    # noqa: BLE001  (numpy-only callbacks raise TypeError / RuntimeError on device tensors)
            return False
        for i in range(0, n0, step):
            res = batch(i, self.value[i:i + step])
            self.value[i:i + step] = res.to(self.value.dtype)
        return True

    def resample(self, out):
        """the field on the mesh of `out` by Fourier-space resampling (pmesh `Field.resample`, base/mesh.py:317-327):
        common modes are copied, the others are zero; real fields go through r2c / c2r.  Single GPU."""
        pm, dst = self.pm, out.pm
        if pm.comm.size > 1 or pm.cplx or dst.cplx:
            raise NotImplementedError("Fourier-space resampling is implemented for one GPU and Hermitian-compressed meshes")
        src_c = self if isinstance(self, BaseComplexField) else self.r2c()
        dst_c = out if isinstance(out, BaseComplexField) else ComplexField(dst)
        val = src_c.value if pm.typestr == dst.typestr else src_c.value.to(dst_c.value.dtype)
        check(lib().nbk_resample_complex(_ptr(val), _ptr(dst_c.value), _CODE[dst.typestr], pm._nmesh_c, dst._nmesh_c, _stream()),
              "nbk_resample_complex")
        if isinstance(out, RealField):
            dst_c.c2r(out=out)
        out.attrs = dict(self.attrs)
        return out

    def _apply_host(self, func, kind):
        use, ax0 = self._coords_for(kind)
        for i in range(self.value.shape[0]):
            plane = self.value[i].cpu().numpy()
            cs = [c[i:i + 1] if d == ax0 else c for d, c in enumerate(use)]
            res = numpy.asarray(func(cs, plane[None, ...]))[0]
            self.value[i] = torch.from_numpy(numpy.ascontiguousarray(res.astype(plane.dtype))).to(self.value.device)


class RealField(Field):
    @staticmethod
    def _layout(pm):
        return pm.real_shape, _TORCH_REAL[pm.typestr]

    @property
    def dtype(self):
        return self.pm.dtype

    def preview(self, Nmesh=None, axes=None):
        """the field, optionally summed over the axes NOT listed in `axes`, as a numpy array on every rank (pmesh
        `Field.preview`; fftpower.py:432).  The reduction over dropped axes runs on the device; only the projected
        array crosses PCIe."""
        pm = self.pm
        if Nmesh is not None and any(numpy.ones(3, 'i8') * Nmesh != pm.Nmesh):
            raise NotImplementedError("preview at a different resolution is not implemented")
        if axes is None:
            axes = [0, 1, 2]
        axes = [axes] if numpy.isscalar(axes) else list(axes)
        drop = tuple(a for a in range(3) if a not in axes)
        local = self.value.sum(dim=drop, dtype=torch.float64) if drop else self.value
        local = local.cpu().numpy()
        if pm.comm.size > 1:
            if 0 in axes:                  # x is kept: concatenate the slabs
                local = numpy.concatenate(pm.comm.allgather(local), axis=0)
            else:                          # x is summed over: add the slabs
                local = pm.comm.allreduce(local)
        kept = [a for a in range(3) if a in axes]      # current axis order (ascending)
        if axes != kept:
            local = local.transpose([kept.index(a) for a in axes])
        return local

    def readout(self, pos, out=None, resampler=None, transform=None, gradient=None, layout=None):
        """values of the field at `pos` through the window (pmesh `RealField.readout`, used by
        algorithms/fftrecon.py:239-244): out[p] = sum_stencil W * field[cell].  Device tensors in -> device tensor
        out, numpy in -> numpy out.  With x slabs the partial sums of the owning ranks are exchanged and added."""
        pm = self.pm
        if gradient is not None:
            raise NotImplementedError("gradient readout is not part of the FFTPower path")
        res = pm.resampler if resampler is None else _window.FindResampler(resampler)
        if res.code is None:
            raise NotImplementedError("no CUDA readout kernel for window '%s'" % res.name)
        shift = 0.0
        if transform is not None:
            shift = float(numpy.atleast_1d(transform.translate - pm.affine.translate).ravel()[0])
        was_numpy = not isinstance(pos, torch.Tensor)
        p = as_device_tensor(pos, device=self.value.device)
        if p.dtype not in (torch.float32, torch.float64):
            p = p.to(torch.float64)
        if p.ndim != 2 or p.shape[1] != 3:
            raise ValueError("readout: position must have shape (n, 3)")
        p = p.contiguous()
        n = int(p.shape[0])
        o = out
        if o is None or not isinstance(o, torch.Tensor):
            o = torch.empty(n, dtype=_TORCH_REAL[pm.typestr], device=p.device)
        if o.dtype not in (torch.float32, torch.float64) or not o.is_contiguous() or o.shape[0] != n:
            raise ValueError("readout: `out` must be a contiguous float32/float64 array of length n")
        def gather(pp, oo):
            check(lib().nbk_readout(_ptr(self.value), _CODE[pm.typestr], _ptr(pp), F4 if pp.dtype == torch.float32 else F8,
                                    int(pp.shape[0]), res.code, shift, pm._box_c, pm._nmesh_c, pm.x_start, pm.x_n, _ptr(oo),
                                    F4 if oo.dtype == torch.float32 else F8, 0, _stream()), "nbk_readout")
        if pm.comm.size == 1:
            gather(p, o)
        else:
            # x slabs: every rank sums its own planes for its local rows and for the rows whose stencil reaches it
            # (the ghost list of decompose); the partial sums travel back and are added (layout.gather, mode='sum')
            lay = layout if isinstance(layout, SlabLayout) else pm.decompose(p, smoothing=0.5 * res.support + abs(shift))
            rpos, _, sidx = lay.route(p, None, want_index=True)
            acc = torch.empty(n, dtype=torch.float64, device=p.device)
            gather(p, acc)
            part = torch.empty(int(rpos.shape[0]), dtype=torch.float64, device=p.device)
            if rpos.shape[0]:
                gather(rpos.contiguous(), part)
            lay.gather_back(part, sidx, acc)
            o.copy_(acc.to(o.dtype))
        if out is not None and not isinstance(out, torch.Tensor):
            out[...] = o.cpu().numpy()
            return out
        return o.cpu().numpy() if was_numpy else o

    def r2c(self, out=None, scale=1.0):
        """forward FFT, normalised by 1/prod(N).  out=Ellipsis has no in-place meaning here (the
        transform is out of place); the real buffer stays valid.  `scale` (extension) multiplies the
        result inside the last FFT pass -- e.g. the 1/nbar of the 1+delta normalisation."""
        pm = self.pm
        if out is None or out is Ellipsis:
            out = ComplexField(pm)
        code = _CODE[pm.typestr]
        P = pm.comm.size
        Nx, Ny, Nz = [int(v) for v in pm.Nmesh]
        if pm.cplx:
            half = torch.empty((Nx, Ny, Nz // 2 + 1), dtype=out.value.dtype, device=out.value.device)
            with stage("r2c"):
                if pm.mixed_fft:
                    check(lib().nbk_r2c_mr(_ptr(self.value), _ptr(half), code, pm._nmesh_c, float(scale), _stream()),
                          "nbk_r2c_mr")
                else:
                    check(lib().nbk_r2c(_ptr(self.value), _ptr(half), code, pm._nmesh_c, float(scale), _stream()), "nbk_r2c")
                check(lib().nbk_hermitian_expand(_ptr(half), _ptr(out.value), code, pm._nmesh_c, _stream()),
                      "nbk_hermitian_expand")
        elif P == 1 and pm.mixed_fft:
            with stage("r2c"):
                check(lib().nbk_r2c_mr(_ptr(self.value), _ptr(out.value), code, pm._nmesh_c, float(scale), _stream()),
                      "nbk_r2c_mr")
        elif P == 1:
            with stage("r2c"):
                check(lib().nbk_r2c(_ptr(self.value), _ptr(out.value), code, pm._nmesh_c, float(scale), _stream()), "nbk_r2c")
        elif pm.mixed_fft:
            self._r2c_mixed_slabs(out, float(scale))
        else:
            Nzc = pm.Nzc
            work = torch.empty((pm.x_n, Ny, Nzc), dtype=out.value.dtype, device=out.value.device)
            st = pm._peer_stage()
            if st is not None:
                # z pass locally; y pass writes every output row straight into its owner's staging buffer over
                # NVLink (fused compute + transpose); barriers bracket the remote writes; x pass reads the staging
                # buffer and writes the result field
                view, ptrs, hdl = st
                from .._lib import lib as _L
                with stage("fft_z"):
                    check(_L().nbk_fft_z_forward(_ptr(self.value), _ptr(work), code, pm.x_n * Ny, Nz, _stream()), "fft_z_forward")
                if _transpose_mode() == "push":
                    # y pass into P contiguous send blocks, then one strided bulk copy per peer over NVLink
                    send = torch.empty((P, pm.y_n, pm.x_n, Nzc), dtype=out.value.dtype, device=out.value.device)
                    nchunk = _push_chunks(pm.x_n)
                    if nchunk <= 1:
                        with stage("fft_y_pack"):
                            check(_L().nbk_fft_lines_pack(_ptr(work), _ptr(send), code, Ny, Nzc, pm.x_n, P, 0, 1.0, _stream()),
                                  "fft_lines_pack")
                        hdl.barrier(channel=0)
                        with stage("fft_y_scatter"):
                            check(_L().nbk_slab_push(_ptr(send), ptrs, code, pm.y_n, pm.x_n, Nzc, pm.x_start, P, pm.comm.rank,
                                                     _stream()), "slab_push")
                    else:
                        # pipelined: the slab is transformed in `nchunk` parts of x planes; part c travels over NVLink on a
                        # copy stream (two of them, alternating: two copy engines) while part c + 1 is transformed
                        hdl.barrier(channel=0)          # every rank is past its previous x pass: the staging buffers are free
                        main = torch.cuda.current_stream()
                        copies = _copy_streams(out.value.device)
                        per = (pm.x_n + nchunk - 1) // nchunk
                        with stage("fft_y_scatter"):    # (the y pass of all parts + the exposed tail of the copies)
                            for c in range(nchunk):
                                o0 = c * per
                                oc = min(per, pm.x_n - o0)
                                if oc <= 0:
                                    break
                                check(_L().nbk_fft_lines_pack_range(_ptr(work), _ptr(send), code, Ny, Nzc, pm.x_n, o0, oc, P, 0, 1.0,
                                                                    _stream()), "fft_lines_pack_range")
                                ev = torch.cuda.Event()
                                ev.record(main)
                                cs = copies[c % len(copies)]
                                cs.wait_event(ev)
                                check(_L().nbk_slab_push_range(_ptr(send), ptrs, code, pm.y_n, pm.x_n, Nzc, pm.x_start, o0, oc, P,
                                                               pm.comm.rank, ctypes.c_void_p(cs.cuda_stream)), "slab_push_range")
                            for cs in copies:
                                main.wait_stream(cs)
                else:
                    hdl.barrier(channel=0)
                    with stage("fft_y_scatter"):
                        check(_L().nbk_fft_lines_scatter(_ptr(work), ptrs, code, Ny, Nzc, pm.x_n, pm.x_start, P, 0, 1.0,
                                                         _stream()), "fft_lines_scatter")
                hdl.barrier(channel=1)
                scale = float(scale) / (float(Nx) * Ny * Nz)
                with stage("fft_x"):
                    check(_L().nbk_fft_lines_oop(_ptr(view), _ptr(out.value), code, Nx, Nzc, Nzc, pm.y_n, Nx * Nzc, 0, scale,
                                                 _stream()), "fft_lines_oop(x)")
                out.attrs = dict(self.attrs)
                return out
            send = torch.empty_like(work)
            with stage("fft_zy"):
                check(lib().nbk_fft_zy_forward(_ptr(self.value), _ptr(work), code, pm.x_n, Ny, Nz, _stream()), "fft_zy_forward")
            with stage("fft_pack"):
                check(lib().nbk_transpose_pack(_ptr(work), _ptr(send), code, pm.x_n, Ny, Nzc, P, _stream()), "transpose_pack")
            recv = torch.view_as_real(work).view(-1)
            with stage("fft_alltoall"):
                pm.comm.all_to_all_single(recv, torch.view_as_real(send).view(-1))
            with stage("fft_unpack"):
                check(lib().nbk_transpose_unpack(_ptr(recv), _ptr(out.value), code, pm.y_n, Nx, Nzc, P, _stream()), "transpose_unpack")
            scale = float(scale) / (float(Nx) * Ny * Nz)
            with stage("fft_x"):
                check(lib().nbk_fft_lines(_ptr(out.value), code, Nx, Nzc, Nzc, pm.y_n, Nx * Nzc, 0, scale, _stream()), "fft_lines(x)")
        out.attrs = dict(self.attrs)
        return out

    def _r2c_mixed_slabs(self, out, scale):
        """P > 1, mixed-radix sizes: z and y passes on the x slab, pack + NCCL all-to-all + unpack into the transposed
        [y_n][Nx][Nzc] layout, x pass (the NVLink peer transpose serves power-of-two sizes only)"""
        pm = self.pm
        L, code, P = lib(), _CODE[pm.typestr], pm.comm.size
        Nx, Ny, Nz = [int(v) for v in pm.Nmesh]
        Nzc = pm.Nzc
        work = torch.empty((pm.x_n, Ny, Nzc), dtype=out.value.dtype, device=out.value.device)
        with stage("fft_zy"):
            check(L.nbk_fft_mr_z(_ptr(self.value), _ptr(work), code, pm.x_n * Ny, Nz, 0, 1.0, _stream()), "fft_mr_z")
            check(L.nbk_fft_mr_lines(_ptr(work), _ptr(work), code, Ny, Nzc, Nzc, pm.x_n, Ny * Nzc, 0, 1.0, _stream()),
                  "fft_mr_lines(y)")
        send = torch.empty_like(work)
        with stage("fft_pack"):
            check(L.nbk_transpose_pack(_ptr(work), _ptr(send), code, pm.x_n, Ny, Nzc, P, _stream()), "transpose_pack")
        recv = torch.view_as_real(work).view(-1)
        with stage("fft_alltoall"):
            pm.comm.all_to_all_single(recv, torch.view_as_real(send).view(-1))
        with stage("fft_unpack"):
            check(L.nbk_transpose_unpack(_ptr(recv), _ptr(out.value), code, pm.y_n, Nx, Nzc, P, _stream()), "transpose_unpack")
        with stage("fft_x"):
            check(L.nbk_fft_mr_lines(_ptr(out.value), _ptr(out.value), code, Nx, Nzc, Nzc, pm.y_n, Nx * Nzc, 0,
                                     scale / (float(Nx) * Ny * Nz), _stream()), "fft_mr_lines(x)")


class BaseComplexField(Field):
    pass


class ComplexField(BaseComplexField):
    @property
    def compressed(self):
        """Hermitian-compressed last axis (fftpower.py:572): False on complex-dtype meshes, which keep all N^3 modes"""
        return not self.pm.cplx

    @staticmethod
    def _layout(pm):
        return pm.complex_shape, _TORCH_CPLX[pm.typestr]

    @property
    def dtype(self):
        return numpy.dtype("c8" if self.pm.typestr == "f4" else "c16")

    @property
    def transposed(self):
        return self.pm.transposed

    def _slab(self):
        """(layout bits, first owned index, count) as the Fourier-space kernels take them (NBK_LAYOUT_*)"""
        pm = self.pm
        full = 2 if pm.cplx else 0
        return (1 | full, pm.y_start, pm.y_n) if pm.transposed else (full, 0, int(pm.Nmesh[0]))

    def c2r(self, out=None):
        """backward FFT, unnormalised.  The complex buffer is preserved."""
        pm = self.pm
        if out is None or out is Ellipsis:
            out = RealField(pm)
        code = _CODE[pm.typestr]
        P = pm.comm.size
        Nx, Ny, Nz = [int(v) for v in pm.Nmesh]
        if pm.cplx:
            # the field is the spectrum of a real array (this path never builds anything else): its stored half is
            # all a c2r needs
            half = torch.empty((Nx, Ny, Nz // 2 + 1), dtype=self.value.dtype, device=self.value.device)
            check(lib().nbk_hermitian_compress(_ptr(self.value), _ptr(half), code, Nx * Ny, Nz, _stream()),
                  "nbk_hermitian_compress")
            if pm.mixed_fft:
                check(lib().nbk_c2r_mr(_ptr(half), _ptr(out.value), code, pm._nmesh_c, None, _stream()), "nbk_c2r_mr")
            else:
                check(lib().nbk_c2r(_ptr(half), _ptr(out.value), code, pm._nmesh_c, None, _stream()), "nbk_c2r")
            out.attrs = dict(self.attrs)
            return out
        if pm.mixed_fft:
            self._c2r_mixed(out)
            out.attrs = dict(self.attrs)
            return out
        st = pm._peer_stage() if P > 1 else None
        if st is not None:
            # inverse x pass scatters rows into the owners' staging buffers over NVLink (the input is only read);
            # inverse y pass + z c2r then run locally on the staging buffer
            view, ptrs, hdl = st
            Nzc = pm.Nzc
            if _transpose_mode() == "push":
                send = torch.empty((P, pm.x_n, pm.y_n, Nzc), dtype=self.value.dtype, device=self.value.device)
                with stage("ifft_x_pack"):
                    check(lib().nbk_fft_lines_pack(_ptr(self.value), _ptr(send), code, Nx, Nzc, pm.y_n, P, 1, 1.0, _stream()),
                          "fft_lines_pack(inverse)")
                hdl.barrier(channel=0)
                with stage("ifft_x_scatter"):
                    check(lib().nbk_slab_push(_ptr(send), ptrs, code, pm.x_n, pm.y_n, Nzc, pm.y_start, P, pm.comm.rank,
                                              _stream()), "slab_push(inverse)")
            else:
                hdl.barrier(channel=0)
                with stage("ifft_x_scatter"):
                    check(lib().nbk_fft_lines_scatter(_ptr(self.value), ptrs, code, Nx, Nzc, pm.y_n, pm.y_start, P, 1, 1.0,
                                                      _stream()), "fft_lines_scatter(inverse)")
            hdl.barrier(channel=1)
            with stage("ifft_zy"):
                check(lib().nbk_fft_zy_backward(_ptr(view), _ptr(out.value), code, pm.x_n, Ny, Nz, _stream()), "fft_zy_backward")
            out.attrs = dict(self.attrs)
            return out
        work = torch.empty_like(self.value)
        if P == 1:
            check(lib().nbk_c2r(_ptr(self.value), _ptr(out.value), code, pm._nmesh_c, _ptr(work), _stream()), "nbk_c2r")
        else:
            Nzc = pm.Nzc
            work.copy_(self.value)
            check(lib().nbk_fft_lines(_ptr(work), code, Nx, Nzc, Nzc, pm.y_n, Nx * Nzc, 1, 1.0, _stream()), "fft_lines(x)")
            send = torch.empty_like(work)
            check(lib().nbk_transpose_pack_back(_ptr(work), _ptr(send), code, pm.y_n, Nx, Nzc, P, _stream()), "pack_back")
            recv = torch.view_as_real(work).view(-1)
            pm.comm.all_to_all_single(recv, torch.view_as_real(send).view(-1))
            slab = torch.view_as_real(send).view(-1)
            check(lib().nbk_transpose_unpack_back(_ptr(recv), _ptr(slab), code, pm.x_n, Ny, Nzc, P, _stream()), "unpack_back")
            check(lib().nbk_fft_zy_backward(_ptr(slab), _ptr(out.value), code, pm.x_n, Ny, Nz, _stream()), "fft_zy_backward")
        out.attrs = dict(self.attrs)
        return out

    def _c2r_mixed(self, out):
        """the mixed-radix inverse: one GPU in one call; P > 1 mirrors _r2c_mixed_slabs (inverse x pass, pack back +
        NCCL all-to-all + unpack back, inverse y and z passes on the x slab).  The complex field is only read."""
        pm = self.pm
        L, code, P = lib(), _CODE[pm.typestr], pm.comm.size
        Nx, Ny, Nz = [int(v) for v in pm.Nmesh]
        work = torch.empty_like(self.value)
        if P == 1:
            with stage("c2r"):
                check(L.nbk_c2r_mr(_ptr(self.value), _ptr(out.value), code, pm._nmesh_c, _ptr(work), _stream()), "nbk_c2r_mr")
            return
        Nzc = pm.Nzc
        with stage("ifft_x"):
            check(L.nbk_fft_mr_lines(_ptr(self.value), _ptr(work), code, Nx, Nzc, Nzc, pm.y_n, Nx * Nzc, 1, 1.0, _stream()),
                  "fft_mr_lines(x)")
        send = torch.empty_like(work)
        with stage("ifft_pack"):
            check(L.nbk_transpose_pack_back(_ptr(work), _ptr(send), code, pm.y_n, Nx, Nzc, P, _stream()), "pack_back")
        recv = torch.view_as_real(work).view(-1)
        with stage("ifft_alltoall"):
            pm.comm.all_to_all_single(recv, torch.view_as_real(send).view(-1))
        slab = torch.view_as_real(send).view(-1)
        with stage("ifft_unpack"):
            check(L.nbk_transpose_unpack_back(_ptr(recv), _ptr(slab), code, pm.x_n, Ny, Nzc, P, _stream()), "unpack_back")
        with stage("ifft_zy"):
            check(L.nbk_fft_mr_lines(_ptr(slab), _ptr(slab), code, Ny, Nzc, Nzc, pm.x_n, Ny * Nzc, 1, 1.0, _stream()),
                  "fft_mr_lines(y)")
            check(L.nbk_fft_mr_z(_ptr(slab), _ptr(out.value), code, pm.x_n * Ny, Nz, 1, 1.0, _stream()), "fft_mr_z")

    def compensate(self, name):
        """v /= window transfer function (source/mesh/catalog.py:449-594), in place"""
        pm = self.pm
        tr, start, count = self._slab()
        with stage("compensate"):
            check(lib().nbk_compensate(_ptr(self.value), _CODE[pm.typestr], _lib.COMP[name], pm._nmesh_c, tr, start, count,
                                       _stream()), "nbk_compensate")
        return self

    def interlace_combine(self, other):
        """self = 0.5 self + 0.5 other exp(0.5j k.H)  (source/mesh/catalog.py:345-347)"""
        pm = self.pm
        tr, start, count = self._slab()
        check(lib().nbk_interlace_combine(_ptr(self.value), _ptr(other.value), _CODE[pm.typestr], pm._nmesh_c, pm._box_c,
                                          tr, start, count, _stream()), "nbk_interlace_combine")
        return self


def _typestr_to_type(typestr):
    if typestr in (RealField, ComplexField):
        return typestr
    if typestr in ("real", None):
        return RealField
    if typestr in ("complex", "transposedcomplex", "untransposedcomplex"):
        return ComplexField
    raise ValueError("unknown field type %s" % str(typestr))
