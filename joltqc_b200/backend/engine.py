"""Python handle on one C-ABI J/K engine (one shell table on one GPU).

torch is used only for device memory and streams (plumbing); all arithmetic happens in
libjoltqc_b200.so.
"""
import ctypes

import numpy as np
import torch

from . import lib as _lib
from .cart2sph import cart2sph_matrix


def _ptr(a, t):
    return a.ctypes.data_as(ctypes.POINTER(t))


class JKEngine:
    def __init__(self, layout, device=None, devices=None):
        if not torch.cuda.is_available():
            raise RuntimeError("joltqc_b200 needs a CUDA device (B200); there is no CPU J/K path")
        self.L = _lib.load()
        if device is None:
            device = devices[0] if devices else torch.cuda.current_device()
        self.device = torch.device("cuda", int(device) if not isinstance(device, torch.device) else device.index or 0)
        self.layout = layout
        packed = np.ascontiguousarray(layout.basis_data_fp64["packed"], dtype=np.float64)
        angs = np.ascontiguousarray(layout.angs, dtype=np.int32)
        nprims = np.ascontiguousarray(layout.nprims, dtype=np.int32)
        ao_loc = np.ascontiguousarray(layout.ao_loc, dtype=np.int32)
        pad = np.ascontiguousarray(layout.pad_id, dtype=np.uint8)
        goff = np.ascontiguousarray(layout.group_offset, dtype=np.int32)
        moff = np.ascontiguousarray(layout.mol_ao_offset, dtype=np.int32)
        c2s = np.ascontiguousarray(np.concatenate([cart2sph_matrix(l).ravel() for l in range(5)]))
        d = _lib.BasisDesc(
            nbas=int(angs.size), records=_ptr(packed, ctypes.c_double), angs=_ptr(angs, ctypes.c_int),
            nprims=_ptr(nprims, ctypes.c_int), ao_loc=_ptr(ao_loc, ctypes.c_int), pad=_ptr(pad, ctypes.c_uint8),
            ngroups=int(goff.size - 1), group_offset=_ptr(goff, ctypes.c_int), mol_ao_offset=_ptr(moff, ctypes.c_int),
            mol_nao=int(layout.mol_nao), mol_cart=int(bool(layout._mol.cart)), c2s=_ptr(c2s, ctypes.c_double))
        h = ctypes.c_void_p()
        _lib.check(self.L.jqc_engine_create(ctypes.byref(d), self.device.index, ctypes.byref(h)))
        self.h = h
        self.nbas, self.nao, self.mol_nao = int(angs.size), int(ao_loc[-1]), int(layout.mol_nao)
        self._q = {}

    def __del__(self):
        h, self.h = getattr(self, "h", None), None
        if h:
            try:
                self.L.jqc_engine_destroy(h)
            except Exception:
                pass

    # ------------------------------------------------------------------ helpers
    def _dev(self, a):
        t = torch.as_tensor(a) if not isinstance(a, torch.Tensor) else a
        return t.to(device=self.device, dtype=torch.float64).contiguous()

    @staticmethod
    def _stream():
        return ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)

    def set_shard(self, rank, world):
        _lib.check(self.L.jqc_engine_set_shard(self.h, int(rank), int(world)))

    def set_profiling(self, on=True):
        _lib.check(self.L.jqc_set_profiling(self.h, int(bool(on))))

    # ------------------------------------------------------------------ pieces
    def q_matrix(self, omega=0.0):
        omega = float(omega or 0.0)
        if omega not in self._q:
            p = ctypes.c_void_p()
            with torch.cuda.device(self.device):
                _lib.check(self.L.jqc_q_matrix(self.h, omega, ctypes.byref(p)))
                # view of the engine-owned buffer (lives as long as the engine), cloned for safety
                view = _wrap_device_buffer(p.value, self.nbas * self.nbas, self.device, "<f4")
                out = view.reshape(self.nbas, self.nbas).clone()
            self._q[omega] = out
        return self._q[omega]

    def dm_from_mol(self, mat):
        m = self._dev(mat)
        n = 1 if m.ndim == 2 else m.shape[0]
        out = torch.empty((n, self.nao, self.nao), dtype=torch.float64, device=self.device)
        with torch.cuda.device(self.device):
            _lib.check(self.L.jqc_dm_from_mol(self.h, m.data_ptr(), n, out.data_ptr(), self._stream()))
        return out[0] if m.ndim == 2 else out

    def dm_to_mol(self, mat):
        m = self._dev(mat)
        n = 1 if m.ndim == 2 else m.shape[0]
        out = torch.empty((n, self.mol_nao, self.mol_nao), dtype=torch.float64, device=self.device)
        with torch.cuda.device(self.device):
            _lib.check(self.L.jqc_dm_to_mol(self.h, m.data_ptr(), n, out.data_ptr(), self._stream()))
        return out[0] if m.ndim == 2 else out

    # ------------------------------------------------------------------ the operator
    def get_jk(self, dm, hermi=0, with_j=True, with_k=True, omega=None, cutoff_fp64=1e-13, cutoff_fp32=1e-13,
               group=None):
        """dm: (nao, nao) or (n, nao, nao) in the molecule's AO basis, any array type.
        Returns device tensors shaped like dm (the one not requested is the int 0), like the
        reference closure (jqc/pyscf/jk.py:109-118, 380).  With a torch.distributed `group` (or
        an initialised default group after set_shard) the partial J/K of all ranks are summed
        with one all_reduce."""
        d = self._dev(dm)
        shape = d.shape
        d3 = d.reshape(-1, shape[-2], shape[-1])
        if d3.shape[-1] != self.mol_nao or d3.shape[-2] != self.mol_nao:
            raise ValueError(f"dm has AO dimension {tuple(shape)}, the molecule has {self.mol_nao}")
        n = d3.shape[0]
        om = 0.0 if omega is None else float(omega)
        vj = torch.empty_like(d3) if with_j else None
        vk = torch.empty_like(d3) if with_k else None
        st = self._stream()
        world = getattr(self, "_world", 1)
        with torch.cuda.device(self.device):
            if world == 1:
                _lib.check(self.L.jqc_get_jk(self.h, d3.data_ptr(), n, int(hermi), int(with_j), int(with_k), om,
                                             float(cutoff_fp64), float(cutoff_fp32),
                                             vj.data_ptr() if with_j else None, vk.data_ptr() if with_k else None, st))
            else:
                self.build_partial_allreduce(d3, hermi, with_j, with_k, om, cutoff_fp64, cutoff_fp32, group)
                _lib.check(self.L.jqc_finalize(self.h, vj.data_ptr() if with_j else None,
                                               vk.data_ptr() if with_k else None, st))
        return (vj.reshape(shape) if with_j else 0), (vk.reshape(shape) if with_k else 0)

    def enable_sharding(self, rank, world):
        self.set_shard(rank, world)
        self._world = int(world)

    def build_partial(self, dm, hermi=0, with_j=True, with_k=True, omega=None, cutoff_fp64=1e-13, cutoff_fp32=1e-13):
        """This rank's share of the kernel-side [J || K] buffer (jqc_build_partial): a torch view of
        engine-owned memory, ready for an all_reduce; follow with finalize()."""
        d = self._dev(dm)
        d3 = d.reshape(-1, d.shape[-2], d.shape[-1])
        self._last_shape = d.shape
        p = ctypes.c_void_p()
        ln = ctypes.c_size_t()
        with torch.cuda.device(self.device):
            _lib.check(self.L.jqc_build_partial(self.h, d3.data_ptr(), d3.shape[0], int(hermi), int(with_j), int(with_k),
                                                0.0 if omega is None else float(omega), float(cutoff_fp64),
                                                float(cutoff_fp32), ctypes.byref(p), ctypes.byref(ln), self._stream()))
        self._last_jk = (bool(with_j), bool(with_k), d3.shape)
        return _wrap_device_buffer(p.value, ln.value, self.device)

    def finalize(self):
        """Post-processing + back-transform of the (reduced) partial buffer (jqc_finalize)."""
        with_j, with_k, shape3 = self._last_jk
        vj = torch.empty(shape3, dtype=torch.float64, device=self.device) if with_j else None
        vk = torch.empty(shape3, dtype=torch.float64, device=self.device) if with_k else None
        with torch.cuda.device(self.device):
            _lib.check(self.L.jqc_finalize(self.h, vj.data_ptr() if with_j else None, vk.data_ptr() if with_k else None,
                                           self._stream()))
        return (vj.reshape(self._last_shape) if with_j else 0), (vk.reshape(self._last_shape) if with_k else 0)

    def build_partial_allreduce(self, d3, hermi, with_j, with_k, om, cutoff_fp64, cutoff_fp32, group=None):
        import torch.distributed as dist
        buf = self.build_partial(d3, hermi, with_j, with_k, om, cutoff_fp64, cutoff_fp32)
        dist.all_reduce(buf, op=dist.ReduceOp.SUM, group=group)
        return buf

    def jk_energy_grad(self, dm, shell_atom, natm, j_factor=1.0, k_factor=1.0, omega=None, cutoff=1e-13, group=None,
                       count=False):
        """Nuclear gradient of E_jk = (j_factor/2) tr(D J[D]) - (k_factor/4) tr(D K[D]) for one symmetric
        density ``dm`` (mol_nao x mol_nao, molecule AO basis) as a (natm, 3) float64 device tensor
        (jqc_jk_energy_grad).  ``shell_atom``: BasisLayout.shell_atom.  With sharding enabled the partial
        gradients of all ranks are summed with one all_reduce, as in get_jk.  ``count=True`` also stores
        the number of quartets this rank evaluated in ``self.last_grad_quartets`` (synchronises)."""
        d = self._dev(dm)
        if d.ndim != 2 or d.shape[0] != self.mol_nao or d.shape[1] != self.mol_nao:
            raise ValueError(f"dm has shape {tuple(d.shape)}, expected ({self.mol_nao}, {self.mol_nao})")
        return self._energy_grad(self.L.jqc_jk_energy_grad, d, shell_atom, natm, j_factor, k_factor, omega, cutoff,
                                 group, count)

    def jk_energy_grad_uhf(self, dm, shell_atom, natm, j_factor=1.0, k_factor=1.0, omega=None, cutoff=1e-13,
                           group=None, count=False):
        """Nuclear gradient of E_U = (j_factor/2) tr(Dt J[Dt]) - (k_factor/2) [tr(Da K[Da]) + tr(Db K[Db])]
        for two symmetric spin densities ``dm = [Da, Db]`` (2 x mol_nao x mol_nao, molecule AO basis) and
        Dt = Da + Db, in one pass over the derivative integrals (jqc_jk_energy_grad_uhf).  Sharding and
        ``count`` as in jk_energy_grad."""
        d = self._dev(dm)
        if d.ndim != 3 or tuple(d.shape) != (2, self.mol_nao, self.mol_nao):
            raise ValueError(f"dm has shape {tuple(d.shape)}, expected (2, {self.mol_nao}, {self.mol_nao})")
        return self._energy_grad(self.L.jqc_jk_energy_grad_uhf, d, shell_atom, natm, j_factor, k_factor, omega,
                                 cutoff, group, count)

    def _energy_grad(self, fn, d, shell_atom, natm, j_factor, k_factor, omega, cutoff, group, count):
        sa = np.ascontiguousarray(shell_atom, dtype=np.int32)
        if sa.shape != (self.nbas,):
            raise ValueError(f"shell_atom has shape {sa.shape}, expected ({self.nbas},)")
        out = torch.empty((int(natm), 3), dtype=torch.float64, device=self.device)
        nq = ctypes.c_longlong(0)
        with torch.cuda.device(self.device):
            _lib.check(fn(self.h, d.data_ptr(), float(j_factor), float(k_factor), 0.0 if omega is None else float(omega),
                          float(cutoff), _ptr(sa, ctypes.c_int), int(natm), out.data_ptr(),
                          ctypes.byref(nq) if count else None, self._stream()))
            if count:
                self.last_grad_quartets = int(nq.value)
            if getattr(self, "_world", 1) > 1:
                import torch.distributed as dist
                dist.all_reduce(out, op=dist.ReduceOp.SUM, group=group)
        return out

    def get_jk_host(self, dm, hermi=0, with_j=True, with_k=True, omega=None, cutoff_fp64=1e-13, cutoff_fp32=1e-13,
                    out=None):
        """Host-buffer entry point (numpy in, numpy out): H2D + build + D2H inside the C call
        (jqc_get_jk_host).  ``out=(vj, vk)``: preallocated C-contiguous float64 arrays shaped like
        ``dm`` (e.g. views of pinned memory) that receive the results."""
        d = np.ascontiguousarray(dm, dtype=np.float64)
        d3 = d.reshape(-1, d.shape[-2], d.shape[-1])
        if out is not None:
            vj, vk = (o.reshape(d3.shape) if o is not None else None for o in out)
            for o, w in ((vj, with_j), (vk, with_k)):
                if w and (o is None or o.dtype != np.float64 or not o.flags.c_contiguous):
                    raise ValueError("out buffers must be C-contiguous float64 arrays shaped like dm")
        else:
            vj = np.empty_like(d3) if with_j else None
            vk = np.empty_like(d3) if with_k else None
        _lib.check(self.L.jqc_get_jk_host(self.h, d3.ctypes.data, d3.shape[0], int(hermi), int(with_j), int(with_k),
                                          0.0 if omega is None else float(omega), float(cutoff_fp64), float(cutoff_fp32),
                                          vj.ctypes.data if with_j else None, vk.ctypes.data if with_k else None))
        return (vj.reshape(d.shape) if with_j else 0), (vk.reshape(d.shape) if with_k else 0)

    def last_stats(self):
        counts = (ctypes.c_longlong * 625)()
        pw = (ctypes.c_longlong * 625)()
        nl = ctypes.c_int()
        _lib.check(self.L.jqc_last_stats(self.h, counts, pw, ctypes.byref(nl)))
        return np.array(counts[:], dtype=np.int64), np.array(pw[:], dtype=np.int64), int(nl.value)

    def last_band_stats(self):
        """(quartets evaluated by the FP64 kernels, by the FP32 kernels), (their device ms when profiling)."""
        n = (ctypes.c_longlong * 2)()
        ms = (ctypes.c_float * 2)()
        _lib.check(self.L.jqc_last_band_stats(self.h, n, ms))
        return (int(n[0]), int(n[1])), (float(ms[0]), float(ms[1]))

    def last_class_ms(self):
        ms = (ctypes.c_float * 625)()
        _lib.check(self.L.jqc_last_class_ms(self.h, ms))
        return np.array(ms[:], dtype=np.float32)


class _CAI:
    """Minimal __cuda_array_interface__ holder so torch can view an engine-owned buffer."""

    def __init__(self, ptr, n, typestr):
        self.__cuda_array_interface__ = {"shape": (n,), "typestr": typestr, "data": (ptr, False), "version": 3,
                                         "strides": None}


def _wrap_device_buffer(ptr, n, device, typestr="<f8"):
    return torch.as_tensor(_CAI(ptr, n, typestr), device=device)


def fp64_peak_probe(device=0):
    L = _lib.load()
    tf, mhz = ctypes.c_double(), ctypes.c_double()
    _lib.check(L.jqc_fp64_peak_probe(int(device), ctypes.byref(tf), ctypes.byref(mhz)))
    return tf.value, mhz.value
