"""Host-side mirror of the reference's public surface (src/blu.rs, src/lib.rs:11-64).

``BLU(m, b_nz)`` has the methods of ``impl BLU`` (blu.rs:61-334) with the same argument
meaning; instead of ``Result<(), Status>`` every method returns the integer status
(``Status.OK`` == ``Ok(())``), numbered as in include/blu_b200.h.
"""
import ctypes
import os
import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_LIB = None

i64p = ctypes.POINTER(ctypes.c_int64)
f64p = ctypes.POINTER(ctypes.c_double)
i32p = ctypes.POINTER(ctypes.c_int)


class Status:
    OK = 0
    REALLOCATE = 1
    WARNING_SINGULAR_MATRIX = 2
    ERROR_INVALID_CALL = -2
    ERROR_ARGUMENT_MISSING = -3
    ERROR_INVALID_ARGUMENT = -4
    ERROR_MAXIMUM_UPDATES = -5
    ERROR_SINGULAR_UPDATE = -6
    ERROR_INTERNAL = -100
    ERROR_CUDA = -101
    ERROR_OUT_OF_MEMORY = -102


# selectors (include/blu_b200.h)
P = dict(droptol=0, abstol=1, reltol=2, nzbias=3, maxsearch=4, pad=5, stretch=6, compress_thres=7,
         sparse_thres=8, search_rows=9, realloc_factor=10, l_mem=11, u_mem=12, w_mem=13,
         threads_per_basis=14, norms=15, dense_k=16, tail_threads=17, split_min=18, tree_min=19, dense_k_big=20)
_INFO_NAMES = ["m", "rank", "bump_size", "bump_nz", "matrix_nz", "l_nz", "u_nz", "r_nz", "nsearch_pivot",
               "nexpand", "ngarbage", "factor_flops", "min_pivot", "max_pivot", "max_eta", "nupdate",
               "nforrest", "nfactorize", "nupdate_total", "nforrest_total", "nsymperm_total", "l_flops",
               "u_flops", "r_flops", "condest_l", "condest_u", "norm_l", "norm_u", "normest_l_inv",
               "normest_u_inv", "onenorm", "infnorm", "residual_test", "pivot_error", "update_cost",
               "time_factorize", "time_solve", "time_update", "elim_bytes", "nelim_div", "pivotlen",
               "rankdef", "internal_error", "status", "nrealloc", "elim_bytes_head", "nruns", "addmem_l", "addmem_u", "addmem_w"]
I = {n: 100 + k for k, n in enumerate(_INFO_NAMES)}
I.update({f"t_phase{q}": 200 + q for q in range(16)})
I.update({f"n_kind{q}": 220 + q for q in range(8)})
I.update({f"norms_cyc{q}": 230 + q for q in range(16)})


def library_path():
    return os.environ.get("BLU_B200_LIB", os.path.join(_HERE, "libblu_b200.so"))


def load_library(path=None):
    """Load the C-ABI library.  Raises if it is missing: there is no fallback."""
    global _LIB
    if _LIB is not None and path is None:
        return _LIB
    path = path or library_path()
    if not os.path.exists(path):
        raise RuntimeError(f"blu_b200: CUDA library not built: {path} (run __graft_entry__.build())")
    L = ctypes.CDLL(path)
    vp = ctypes.c_void_p
    L.blu_create.argtypes = [ctypes.POINTER(vp), ctypes.c_int64, ctypes.c_int64, ctypes.c_int]
    L.blu_destroy.argtypes = [vp]
    L.blu_set_param.argtypes = [vp, ctypes.c_int, ctypes.c_double]
    L.blu_get_param.argtypes = [vp, ctypes.c_int]; L.blu_get_param.restype = ctypes.c_double
    L.blu_get_info.argtypes = [vp, ctypes.c_int]; L.blu_get_info.restype = ctypes.c_double
    L.blu_factorize.argtypes = [vp, i64p, i64p, i64p, f64p]
    L.blu_get_factors.argtypes = [vp, i64p, i64p, i64p, i64p, f64p, i64p, i64p, f64p]
    L.blu_factorize_c0ntinue.argtypes = [vp, i64p, i64p, i64p, f64p, ctypes.c_int]
    L.blu_solve_dense.argtypes = [vp, f64p, f64p, ctypes.c_char]
    L.blu_solve_dense_multi.argtypes = [vp, ctypes.c_int64, f64p, f64p, ctypes.c_char]
    L.blu_solve_sparse_multi.argtypes = [vp, ctypes.c_int64, i64p, i64p, f64p, i64p, i64p, f64p, i32p, ctypes.c_char]
    L.blu_solve_sparse.argtypes = [vp, ctypes.c_int64, i64p, f64p, i64p, i64p, f64p, ctypes.c_char]
    L.blu_solve_for_update.argtypes = [vp, ctypes.c_int64, i64p, f64p, i64p, i64p, f64p, ctypes.c_char]
    L.blu_update.argtypes = [vp, ctypes.c_double]
    L.blu_clone.argtypes = [ctypes.POINTER(vp), vp]
    for f in ("blu_save", "blu_save_dev"):
        getattr(L, f).argtypes = [vp, vp, ctypes.c_int64, i64p]
    for f in ("blu_restore", "blu_restore_dev"):
        getattr(L, f).argtypes = [vp, vp, ctypes.c_int64]
    L.blu_batch_create.argtypes = [ctypes.POINTER(vp), ctypes.c_int64, ctypes.c_int64, ctypes.c_int64, ctypes.c_int]
    L.blu_batch_destroy.argtypes = [vp]
    L.blu_batch_factorize.argtypes = [vp, i64p, i64p, i64p, f64p, ctypes.c_int64, i32p]
    L.blu_batch_solve_dense.argtypes = [vp, f64p, f64p, ctypes.c_char, i32p]
    L.blu_batch_solve_for_update.argtypes = [vp, i64p, i64p, f64p, ctypes.c_int, i64p, i64p, f64p, i32p, ctypes.c_char]
    L.blu_batch_update.argtypes = [vp, f64p, i32p]
    L.blu_batch_solve_sparse.argtypes = [vp, i64p, i64p, i64p, f64p, i64p, i64p, f64p, i32p, ctypes.c_char]
    L.blu_batch_solve_dense_multi.argtypes = [vp, ctypes.c_int64, f64p, f64p, ctypes.c_char, i32p]
    L.blu_batch_maxvolume.argtypes = [vp, ctypes.c_int64, i64p, i64p, i64p, f64p, ctypes.c_int64, i64p, i64p,
                                      ctypes.c_double, i64p, i32p]
    L.blu_batch_factorize_subset.argtypes = [vp, ctypes.c_int64, i64p, i64p, i64p, i64p, f64p, ctypes.c_int64, i32p]
    L.blu_batch_solve_for_update_subset.argtypes = [vp, ctypes.c_int64, i64p, i64p, i64p, f64p, ctypes.c_int, i64p, i64p, f64p,
                                                    i32p, ctypes.c_char]
    L.blu_batch_update_subset.argtypes = [vp, ctypes.c_int64, i64p, f64p, i32p]
    L.blu_batch_get_info.argtypes = [vp, ctypes.c_int64, ctypes.c_int]; L.blu_batch_get_info.restype = ctypes.c_double
    L.blu_batch_get_factors.argtypes = [vp, ctypes.c_int64, i64p, i64p, i64p, i64p, f64p, i64p, i64p, f64p]
    L.blu_batch_upload.argtypes = [vp, i64p, i64p, i64p, f64p, ctypes.c_int64, f64p]
    L.blu_batch_factorize_resident.argtypes = [vp]
    L.blu_batch_solve_dense_resident.argtypes = [vp, ctypes.c_char]
    L.blu_batch_download.argtypes = [vp, f64p, i32p]
    L.blu_batch_factorize_dev.argtypes = [vp, vp, vp, vp, vp, ctypes.c_int64]
    L.blu_batch_solve_dense_dev.argtypes = [vp, vp, vp, ctypes.c_char, vp]
    L.blu_batch_factorize_subset_dev.argtypes = [vp, vp, vp, vp, vp, vp, ctypes.c_int64, vp]
    L.blu_batch_solve_for_update_dev.argtypes = [vp, vp, vp, vp, vp, ctypes.c_int, vp, vp, vp, vp, ctypes.c_char]
    L.blu_batch_update_dev.argtypes = [vp, vp, vp, vp]
    L.blu_batch_solve_sparse_dev.argtypes = [vp, ctypes.c_int64, vp, vp, vp, vp, vp, vp, vp, vp, ctypes.c_char]
    L.blu_batch_solve_dense_multi_dev.argtypes = [vp, ctypes.c_int64, vp, vp, ctypes.c_char, vp]
    L.blu_batch_copy.argtypes = [vp, ctypes.c_int64, i64p, i64p]
    L.blu_batch_copy_dev.argtypes = [vp, vp]
    for f in ("blu_batch_save", "blu_batch_save_dev"):
        getattr(L, f).argtypes = [vp, ctypes.c_int64, i64p, ctypes.POINTER(vp), i64p, i64p]
    for f in ("blu_batch_restore", "blu_batch_restore_dev"):
        getattr(L, f).argtypes = [vp, ctypes.c_int64, i64p, ctypes.POINTER(vp), i64p]
    L.blu_batch_graph_capture.argtypes = [vp, ctypes.c_char]
    L.blu_batch_graph_launch.argtypes = [vp]
    L.blu_batch_stream.argtypes = [vp]; L.blu_batch_stream.restype = vp
    L.blu_batch_set_stream.argtypes = [vp, vp]
    L.blu_batch_synchronize.argtypes = [vp]
    L.blu_batch_last_kernel_ms.argtypes = [vp, ctypes.c_int]; L.blu_batch_last_kernel_ms.restype = ctypes.c_double
    L.blu_batch_launch_count.argtypes = [vp]; L.blu_batch_launch_count.restype = ctypes.c_int64
    L.blu_multi_create.argtypes = [ctypes.POINTER(vp), ctypes.c_int64, ctypes.c_int64, ctypes.c_int64, i32p, ctypes.c_int]
    L.blu_multi_destroy.argtypes = [vp]
    L.blu_multi_factorize_solve.argtypes = [vp, i64p, i64p, i64p, f64p, ctypes.c_int64, f64p, f64p, ctypes.c_char, i32p]
    L.blu_multi_part.argtypes = [vp, ctypes.c_int, i64p, i64p]; L.blu_multi_part.restype = vp
    L.blu_version.restype = ctypes.c_char_p
    if path == library_path():
        _LIB = L
    return L


def _i64(a):
    return np.ascontiguousarray(a, dtype=np.int64)


def _f64(a):
    return np.ascontiguousarray(a, dtype=np.float64)


def _pi(a):
    return a.ctypes.data_as(i64p) if a is not None else None


def _pf(a):
    return a.ctypes.data_as(f64p) if a is not None else None


def _ch(trans):
    return (trans if isinstance(trans, bytes) else str(trans).encode())[:1]


class _Base:
    _get_info_fn = "blu_get_info"

    def set_param(self, name, value):
        return self._L.blu_set_param(self._h, P[name], float(value))

    def get_param(self, name):
        return self._L.blu_get_param(self._h, P[name])

    def __setattr__(self, name, value):
        # the tunables of `LU` are plain pub fields in the reference (lu.rs:10-66)
        if name in P and "_h" in self.__dict__:
            st = self.set_param(name, value)
            if st != 0:
                raise ValueError(f"set {name}={value}: status {st}")
        else:
            object.__setattr__(self, name, value)

    # Device memory as torch tensors (the _dev calls of BLUBatch, BLU.save_dev / restore_dev).

    def _torch_device(self):
        import torch
        if b"emulation" in self._L.blu_version():      # the SIMT emulation build: its "device" memory is host memory
            return torch.device("cpu")
        if getattr(self, "_cuda_index", None) is None:
            object.__setattr__(self, "_cuda_index", self._device if self._device >= 0 else torch.cuda.current_device())
        return torch.device("cuda", self._cuda_index)

    def _tensor(self, t, dtype, numel, name, dev):
        import torch
        if not isinstance(t, torch.Tensor):
            raise TypeError(f"{name}: a torch.Tensor is expected")
        if t.dtype != dtype:
            raise TypeError(f"{name}: dtype {t.dtype}, expected {dtype}")
        if t.device != dev:
            raise ValueError(f"{name}: tensor on {t.device}, the {'batch' if isinstance(self, BLUBatch) else 'object'} is on {dev}")
        if not t.is_contiguous():
            raise ValueError(f"{name}: not contiguous")
        if numel is not None and t.numel() != numel:
            raise ValueError(f"{name}: {t.numel()} elements, expected {numel}")
        return t

    @staticmethod
    def _ptr(t):
        return ctypes.c_void_p(t.data_ptr()) if t is not None and t.numel() > 0 else None

    def _on_stream(self, dev, fn):
        """run fn (one library call) after everything torch has queued on its current stream of dev"""
        import torch
        if dev.type == "cuda":
            s = torch.cuda.ExternalStream(self._L.blu_batch_stream(self._h), device=dev)
            s.wait_stream(torch.cuda.current_stream(dev))
        return fn()

    @staticmethod
    def _aligned_host(nbytes):
        """a numpy.uint8 array of nbytes whose data starts 16-byte aligned"""
        raw = np.zeros(int(nbytes) + 16, np.uint8)
        k = (-raw.ctypes.data) % 16
        return raw[k:k + int(nbytes)]


class BLU(_Base):
    """struct BLU, blu.rs:9-20: `lu` state on the device, `lhs/ilhs/nzlhs` on the host."""

    def __init__(self, m, b_nz, device=-1, lib=None):
        self._L = lib or load_library()
        h = ctypes.c_void_p()
        st = self._L.blu_create(ctypes.byref(h), int(m), int(b_nz), int(device))
        if st != 0:
            raise RuntimeError(f"blu_create failed with status {st} (no CUDA device? there is no CPU path)")
        self._h = h
        self.m = int(m)
        self.lhs = np.zeros(self.m)
        self.ilhs = np.zeros(self.m, dtype=np.int64)
        self.nzlhs = 0
        self._device = int(device)

    def close(self):
        if getattr(self, "_h", None):
            self._L.blu_destroy(self._h)
            object.__setattr__(self, "_h", None)

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def info(self, name):
        return self._L.blu_get_info(self._h, I[name])

    # blu.rs:95
    def factorize(self, b_begin, b_end, b_i, b_x):
        bb, be, bi, bx = _i64(b_begin), _i64(b_end), _i64(b_i), _f64(b_x)
        if len(bb) < self.m or len(be) < self.m:
            raise IndexError("b_begin/b_end shorter than m")
        return self._L.blu_factorize(self._h, _pi(bb), _pi(be), _pi(bi), _pf(bx))

    def factorize_c0ntinue(self, b_begin, b_end, b_i, b_x, c0ntinue):
        """factorize() of the crate's free-function surface (lib.rs:11-19, factorize.rs:34): Reallocate escapes
        (status 1, `addmem_l/u/w` say how much is missing); grow `l_mem`/`u_mem`/`w_mem` and call again with
        c0ntinue=True."""
        bb, be, bi, bx = _i64(b_begin), _i64(b_end), _i64(b_i), _f64(b_x)
        return self._L.blu_factorize_c0ntinue(self._h, _pi(bb), _pi(be), _pi(bi), _pf(bx), 1 if c0ntinue else 0)

    # blu.rs:139
    def get_factors(self, want_l=True, want_u=True):
        m = self.m
        lnz, unz = int(self.info("l_nz")), int(self.info("u_nz"))
        out = dict(rowperm=np.zeros(m, np.int64), colperm=np.zeros(m, np.int64))
        if want_l:
            out.update(l_colptr=np.zeros(m + 1, np.int64), l_rowidx=np.zeros(m + lnz, np.int64), l_value=np.zeros(m + lnz))
        if want_u:
            out.update(u_colptr=np.zeros(m + 1, np.int64), u_rowidx=np.zeros(m + unz, np.int64), u_value=np.zeros(m + unz))
        st = self._L.blu_get_factors(self._h, _pi(out["rowperm"]), _pi(out["colperm"]),
                                     _pi(out.get("l_colptr")), _pi(out.get("l_rowidx")), _pf(out.get("l_value")),
                                     _pi(out.get("u_colptr")), _pi(out.get("u_rowidx")), _pf(out.get("u_value")))
        return st, out

    # blu.rs:182
    def solve_dense(self, rhs, trans="N"):
        r = _f64(rhs)
        if len(r) != self.m:
            raise IndexError("rhs length != m")   # the reference panics here (lu/solve_dense.rs:37)
        x = np.zeros(self.m)
        st = self._L.blu_solve_dense(self._h, _pf(r), _pf(x), _ch(trans))
        return st, x

    def _clear_lhs(self):
        """lu_clear_lhs, blu.rs:380-395: zero what the previous solve scattered."""
        nz = self.nzlhs
        if nz:
            if nz <= int(self.get_param("sparse_thres") * self.m):
                self.lhs[self.ilhs[:nz]] = 0.0
            else:
                self.lhs[:] = 0.0
            self.nzlhs = 0

    def solve_dense_multi(self, rhs, trans="N"):
        """rhs[nrhs, m] -> (status, x[nrhs, m]): solve_dense for every row, up to BLU_B200_SOLVE_UNITS rows in flight
        together."""
        r = _f64(rhs).reshape(-1, self.m)
        x = np.zeros_like(r)
        st = self._L.blu_solve_dense_multi(self._h, r.shape[0], _pf(r), _pf(x), _ch(trans))
        return st, x

    def solve_sparse_multi(self, rhs_list, trans="N"):
        """rhs_list = [(irhs, xrhs), ...] -> (status, [(ilhs, values), ...]): solve_sparse for each, up to
        BLU_B200_SOLVE_UNITS in flight together; entry n of a result is lhs[ilhs[n]] = values[n], in solve_sparse's
        order."""
        n = len(rhs_list)
        begin = np.zeros(n + 1, dtype=np.int64)
        for r, (ii, _) in enumerate(rhs_list):
            begin[r + 1] = begin[r] + len(ii)
        irhs = _i64(np.concatenate([np.asarray(ii, dtype=np.int64) for ii, _ in rhs_list])) if n else np.zeros(0, np.int64)
        xrhs = _f64(np.concatenate([np.asarray(xx, dtype=np.float64) for _, xx in rhs_list])) if n else np.zeros(0)
        nz = np.zeros(n, dtype=np.int64)
        il = np.zeros(n * self.m, dtype=np.int64)
        xl = np.zeros(n * self.m)
        stat = np.zeros(n, dtype=np.int32)
        st = self._L.blu_solve_sparse_multi(self._h, n, _pi(begin), _pi(irhs), _pf(xrhs), _pi(nz), _pi(il), _pf(xl),
                                            stat.ctypes.data_as(i32p), _ch(trans))
        out = []
        for r in range(n):
            k = max(int(nz[r]), 0)
            out.append((il[r * self.m:r * self.m + k].copy(), xl[r * self.m:r * self.m + k].copy()))
        return st, out, stat

    # blu.rs:207: result in self.lhs / self.ilhs / self.nzlhs
    def solve_sparse(self, nzrhs, irhs, xrhs, trans="N"):
        ir, xr = _i64(irhs), _f64(xrhs)
        self._clear_lhs()
        nz = ctypes.c_int64(0)
        st = self._L.blu_solve_sparse(self._h, int(nzrhs), _pi(ir), _pf(xr), ctypes.byref(nz), _pi(self.ilhs), _pf(self.lhs), _ch(trans))
        self.nzlhs = nz.value
        return st

    # blu.rs:257
    def solve_for_update(self, nzrhs, irhs, xrhs, trans="N", want_solution=0):
        ir = _i64(irhs)
        xr = _f64(xrhs) if xrhs is not None else None
        self._clear_lhs()
        # D13 (SURVEY.md section 0) repaired: blu.rs:268-283 passes Some(lhs)
        # even when want_solution == 0; BASICLU semantics = no solution unless asked for.
        if want_solution:
            nz = ctypes.c_int64(0)
            st = self._L.blu_solve_for_update(self._h, int(nzrhs), _pi(ir), _pf(xr), ctypes.byref(nz), _pi(self.ilhs), _pf(self.lhs), _ch(trans))
            self.nzlhs = nz.value
        else:
            st = self._L.blu_solve_for_update(self._h, int(nzrhs), _pi(ir), _pf(xr), None, None, None, _ch(trans))
        return st

    # blu.rs:319
    def update(self, xtbl):
        return self._L.blu_update(self._h, float(xtbl))

    def clone(self):
        """BLU: Clone (blu_clone): a new object on this one's device with its factors, update history, pending
        solve_for_update, getters, parameters, capacities, resident B and lhs / ilhs / nzlhs.  From then on it behaves
        bit for bit as this one would.  Raises on a failed call."""
        h = ctypes.c_void_p()
        st = self._L.blu_clone(ctypes.byref(h), self._h)
        if st != 0:
            raise RuntimeError(f"blu_clone: status {st}")
        c = BLU.__new__(BLU)
        c._L, c._h, c.m, c._device = self._L, h, self.m, self._device
        c.lhs, c.ilhs, c.nzlhs = self.lhs.copy(), self.ilhs.copy(), self.nzlhs
        return c

    def __copy__(self):
        return self.clone()

    def __deepcopy__(self, memo):
        return self.clone()

    # Images (blu_save / blu_restore): the format of BLUBatch.save / restore, so that an image moves a basis between
    # objects and batch slots of the same m.

    def save(self):
        """The object's image as a numpy.uint8 array.  Raises on a failed call."""
        n = ctypes.c_int64(0)
        st = self._L.blu_save(self._h, None, 0, ctypes.byref(n))
        if st != 0:
            raise ValueError(f"blu_save: status {st}")
        a = self._aligned_host(n.value)
        st = self._L.blu_save(self._h, ctypes.c_void_p(a.ctypes.data), a.size, ctypes.byref(n))
        if st != 0:
            raise ValueError(f"blu_save: status {st}")
        return a

    def restore(self, img):
        """The object becomes the basis saved in img (a buffer of bytes: a numpy.uint8 array, bytes, ...).  Returns
        the status."""
        a = np.frombuffer(img, np.uint8) if not isinstance(img, np.ndarray) else np.ascontiguousarray(img).view(np.uint8).reshape(-1)
        if a.ctypes.data % 16:
            b = self._aligned_host(a.size)
            b[:] = a
            a = b
        return self._L.blu_restore(self._h, ctypes.c_void_p(a.ctypes.data), a.size)

    def save_dev(self):
        """The object's image as a 1-D torch.uint8 tensor on its device, 256-byte aligned.  Ordered after torch's
        current stream.  Raises on a failed call."""
        import torch
        dev = self._torch_device()
        n = ctypes.c_int64(0)
        st = self._on_stream(dev, lambda: self._L.blu_save_dev(self._h, None, 0, ctypes.byref(n)))
        if st != 0:
            raise ValueError(f"blu_save_dev: status {st}")
        block = torch.empty(n.value + 256, dtype=torch.uint8, device=dev)
        at = (-block.data_ptr()) % 256
        out = block[at:at + n.value]
        st = self._on_stream(dev, lambda: self._L.blu_save_dev(self._h, ctypes.c_void_p(out.data_ptr()), out.numel(), ctypes.byref(n)))
        if st != 0:
            raise ValueError(f"blu_save_dev: status {st}")
        return out

    def restore_dev(self, img):
        """restore from a contiguous torch.uint8 tensor on the object's device.  Returns the status."""
        import torch
        dev = self._torch_device()
        t = self._tensor(img, torch.uint8, None, "img", dev)
        return self._on_stream(dev, lambda: self._L.blu_restore_dev(self._h, ctypes.c_void_p(t.data_ptr()), t.numel()))


class BLUBatch(_Base):
    """Many independent bases of one dimension on one GPU (one `BLU` per basis on the CPU)."""

    def __init__(self, nmat, m, bnz_cap, device=-1, lib=None):
        self._L = lib or load_library()
        h = ctypes.c_void_p()
        st = self._L.blu_batch_create(ctypes.byref(h), int(nmat), int(m), int(bnz_cap), int(device))
        if st != 0:
            raise RuntimeError(f"blu_batch_create failed with status {st} (no CUDA device? there is no CPU path)")
        self._h = h
        self.nmat, self.m = int(nmat), int(m)
        self._device = int(device)

    def close(self):
        if getattr(self, "_h", None):
            self._L.blu_batch_destroy(self._h)
            object.__setattr__(self, "_h", None)

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def info(self, k, name):
        return self._L.blu_batch_get_info(self._h, int(k), I[name])

    def factorize(self, b_begin, b_end, b_i, b_x):
        bb, be, bi, bx = _i64(b_begin), _i64(b_end), _i64(b_i), _f64(b_x)
        status = np.zeros(self.nmat, dtype=np.int32)
        st = self._L.blu_batch_factorize(self._h, _pi(bb), _pi(be), _pi(bi), _pf(bx), len(bi), status.ctypes.data_as(i32p))
        return st, status

    def solve_dense(self, rhs, trans="N"):
        r = _f64(rhs).reshape(-1)
        x = np.zeros(self.nmat * self.m)
        status = np.zeros(self.nmat, dtype=np.int32)
        st = self._L.blu_batch_solve_dense(self._h, _pf(r), _pf(x), _ch(trans), status.ctypes.data_as(i32p))
        return st, x.reshape(self.nmat, self.m), status

    def solve_for_update(self, rhs_list, trans="N", want_solution=0):
        """rhs_list[k] = (irhs, xrhs or None) for basis k -> (status, per-basis status, [(ilhs, values)] or None)"""
        n = self.nmat
        begin = np.zeros(n + 1, dtype=np.int64)
        for k, (ii, _) in enumerate(rhs_list):
            begin[k + 1] = begin[k] + len(ii)
        irhs = _i64(np.concatenate([np.asarray(ii, dtype=np.int64).reshape(-1) for ii, _ in rhs_list]))
        have_x = rhs_list[0][1] is not None
        xrhs = _f64(np.concatenate([np.asarray(xx, dtype=np.float64) for _, xx in rhs_list])) if have_x else None
        stat = np.zeros(n, dtype=np.int32)
        if want_solution:
            nz = np.zeros(n, dtype=np.int64); il = np.zeros(n * self.m, dtype=np.int64); xl = np.zeros(n * self.m)
            st = self._L.blu_batch_solve_for_update(self._h, _pi(begin), _pi(irhs), _pf(xrhs), 1, _pi(nz), _pi(il), _pf(xl),
                                                    stat.ctypes.data_as(i32p), _ch(trans))
            out = [(il[k * self.m:k * self.m + max(int(nz[k]), 0)].copy(), xl[k * self.m:k * self.m + max(int(nz[k]), 0)].copy()) for k in range(n)]
            return st, stat, out
        st = self._L.blu_batch_solve_for_update(self._h, _pi(begin), _pi(irhs), _pf(xrhs), 0, None, None, None,
                                                stat.ctypes.data_as(i32p), _ch(trans))
        return st, stat, None

    def update(self, xtbl):
        x = _f64(xtbl)
        stat = np.zeros(self.nmat, dtype=np.int32)
        st = self._L.blu_batch_update(self._h, _pf(x), stat.ctypes.data_as(i32p))
        return st, stat

    def factorize_subset(self, sel, b_begin, b_end, b_i, b_x):
        """Refactorize the bases sel only; column j of the r-th is b_i/b_x[b_begin[r*m+j] : b_end[r*m+j]].  The other
        bases keep their factors and update history.  Returns (status, status per selected basis)."""
        s, bb, be, bi, bx = _i64(sel), _i64(b_begin), _i64(b_end), _i64(b_i), _f64(b_x)
        stat = np.zeros(len(s), dtype=np.int32)
        st = self._L.blu_batch_factorize_subset(self._h, len(s), _pi(s), _pi(bb), _pi(be), _pi(bi), _pf(bx), len(bi),
                                                stat.ctypes.data_as(i32p))
        return st, stat

    def solve_for_update_subset(self, sel, rhs_list, trans="N", want_solution=0):
        """solve_for_update on the bases sel only, rhs_list[r] = (irhs, xrhs or None) for basis sel[r] ->
        (status, status per selected basis, [(ilhs, values)] per selected basis or None)"""
        s = _i64(sel)
        n = len(s)
        begin = np.zeros(n + 1, dtype=np.int64)
        for r, (ii, _) in enumerate(rhs_list):
            begin[r + 1] = begin[r] + len(np.asarray(ii).reshape(-1))
        irhs = _i64(np.concatenate([np.asarray(ii, dtype=np.int64).reshape(-1) for ii, _ in rhs_list])) if n else np.zeros(0, np.int64)
        have_x = n > 0 and rhs_list[0][1] is not None
        xrhs = _f64(np.concatenate([np.asarray(xx, dtype=np.float64) for _, xx in rhs_list])) if have_x else None
        stat = np.zeros(n, dtype=np.int32)
        if want_solution:
            nz = np.zeros(n, dtype=np.int64); il = np.zeros(max(n, 1) * self.m, dtype=np.int64); xl = np.zeros(max(n, 1) * self.m)
            st = self._L.blu_batch_solve_for_update_subset(self._h, n, _pi(s), _pi(begin), _pi(irhs), _pf(xrhs), 1, _pi(nz), _pi(il),
                                                           _pf(xl), stat.ctypes.data_as(i32p), _ch(trans))
            out = [(il[r * self.m:r * self.m + max(int(nz[r]), 0)].copy(), xl[r * self.m:r * self.m + max(int(nz[r]), 0)].copy())
                   for r in range(n)]
            return st, stat, out
        st = self._L.blu_batch_solve_for_update_subset(self._h, n, _pi(s), _pi(begin), _pi(irhs), _pf(xrhs), 0, None, None, None,
                                                       stat.ctypes.data_as(i32p), _ch(trans))
        return st, stat, None

    def update_subset(self, sel, xtbl):
        """update on the bases sel only, basis sel[r] with xtbl[r] -> (status, status per selected basis)"""
        s, x = _i64(sel), _f64(xtbl)
        stat = np.zeros(len(s), dtype=np.int32)
        st = self._L.blu_batch_update_subset(self._h, len(s), _pi(s), _pf(x), stat.ctypes.data_as(i32p))
        return st, stat

    def solve_sparse(self, rhs_lists, trans="N"):
        """rhs_lists[k] = [(irhs, xrhs), ...] for basis k -> (status, [[(ilhs, values), ...] per basis],
        [unit status per basis]): solve_sparse for every right-hand side of every basis, one warp each, as
        BLU.solve_sparse_multi does for one basis.  A rejected right-hand side gives empty arrays."""
        if len(rhs_lists) != self.nmat:
            raise IndexError("rhs_lists needs one list per basis")
        counts = np.array([len(r) for r in rhs_lists], dtype=np.int64)
        unit_begin = np.concatenate([[0], np.cumsum(counts)]).astype(np.int64)
        units = [pair for r in rhs_lists for pair in r]
        n = len(units)
        rhs_begin = np.concatenate([[0], np.cumsum([len(ii) for ii, _ in units])]).astype(np.int64)
        irhs = _i64(np.concatenate([np.asarray(ii, dtype=np.int64).reshape(-1) for ii, _ in units])) if n else np.zeros(0, np.int64)
        xrhs = _f64(np.concatenate([np.asarray(xx, dtype=np.float64).reshape(-1) for _, xx in units])) if n else np.zeros(0)
        nz = np.zeros(n, dtype=np.int64)
        il = np.zeros(max(n, 1) * self.m, dtype=np.int64)
        xl = np.zeros(max(n, 1) * self.m)
        stat = np.zeros(max(n, 1), dtype=np.int32)
        st = self._L.blu_batch_solve_sparse(self._h, _pi(unit_begin), _pi(rhs_begin), _pi(irhs), _pf(xrhs), _pi(nz), _pi(il),
                                            _pf(xl), stat.ctypes.data_as(i32p), _ch(trans))
        out, ustat = [], []
        for k in range(self.nmat):
            res = []
            for u in range(unit_begin[k], unit_begin[k + 1]):
                c = max(int(nz[u]), 0)
                res.append((il[u * self.m:u * self.m + c].copy(), xl[u * self.m:u * self.m + c].copy()))
            out.append(res)
            ustat.append(stat[unit_begin[k]:unit_begin[k + 1]].copy())
        return st, out, ustat

    def solve_dense_multi(self, rhs, trans="N"):
        """rhs[nmat, nrhs, m] -> (status, x[nmat, nrhs, m], status[nmat, nrhs]): solve_dense for every right-hand
        side of every basis, one warp each."""
        r = _f64(rhs)
        nrhs = r.size // (self.nmat * self.m)
        r = r.reshape(self.nmat, nrhs, self.m)
        x = np.zeros_like(r)
        stat = np.zeros((self.nmat, nrhs), dtype=np.int32)
        st = self._L.blu_batch_solve_dense_multi(self._h, nrhs, _pf(r), _pf(x), _ch(trans), stat.ctypes.data_as(i32p))
        return st, x, stat

    def maxvolume(self, ncol, a_begin, a_end, a_i, a_x, basis, isbasic, volumetol):
        """maxvolume (maxvolume.rs:64-224) on every basis at once.  Basis k's pool column j is
        a_i/a_x[a_begin[k*ncol+j] : a_end[k*ncol+j]]; basis (nmat*m) and isbasic (nmat*ncol) are updated in place,
        like maxvolume().  Returns (status, per-basis status, per-basis nupdate)."""
        ab, ae, ai, ax = _i64(a_begin), _i64(a_end), _i64(a_i), _f64(a_x)
        bas = _i64(basis).reshape(-1).copy()
        isb = _i64(isbasic).reshape(-1).copy()
        stat = np.zeros(self.nmat, dtype=np.int32)
        nup = np.zeros(self.nmat, dtype=np.int64)
        st = self._L.blu_batch_maxvolume(self._h, int(ncol), _pi(ab), _pi(ae), _pi(ai), _pf(ax), len(ai), _pi(bas), _pi(isb),
                                         float(volumetol), _pi(nup), stat.ctypes.data_as(i32p))
        basis[...] = bas.reshape(np.shape(basis))
        isbasic[...] = isb.reshape(np.shape(isbasic))
        return st, stat, nup

    def get_factors(self, k):
        m = self.m
        lnz, unz = int(self.info(k, "l_nz")), int(self.info(k, "u_nz"))
        out = dict(rowperm=np.zeros(m, np.int64), colperm=np.zeros(m, np.int64),
                   l_colptr=np.zeros(m + 1, np.int64), l_rowidx=np.zeros(m + lnz, np.int64), l_value=np.zeros(m + lnz),
                   u_colptr=np.zeros(m + 1, np.int64), u_rowidx=np.zeros(m + unz, np.int64), u_value=np.zeros(m + unz))
        st = self._L.blu_batch_get_factors(self._h, int(k), _pi(out["rowperm"]), _pi(out["colperm"]),
                                           _pi(out["l_colptr"]), _pi(out["l_rowidx"]), _pf(out["l_value"]),
                                           _pi(out["u_colptr"]), _pi(out["u_rowidx"]), _pf(out["u_value"]))
        return st, out

    # device-resident path (bench)
    def upload(self, b_begin=None, b_end=None, b_i=None, b_x=None, rhs=None):
        bb = _i64(b_begin) if b_begin is not None else None
        be = _i64(b_end) if b_end is not None else None
        bi = _i64(b_i) if b_i is not None else None
        bx = _f64(b_x) if b_x is not None else None
        r = _f64(rhs).reshape(-1) if rhs is not None else None
        return self._L.blu_batch_upload(self._h, _pi(bb), _pi(be), _pi(bi), _pf(bx), len(bi) if bi is not None else 0, _pf(r))

    def factorize_resident(self):
        return self._L.blu_batch_factorize_resident(self._h)

    def factorize_dev(self, d_b_begin, d_b_end, d_b_i, d_b_x, bnz_total):
        """B in caller-owned device memory (raw device pointers as ints, e.g. torch.Tensor.data_ptr())."""
        return self._L.blu_batch_factorize_dev(self._h, d_b_begin, d_b_end, d_b_i, d_b_x, int(bnz_total))

    def solve_dense_dev(self, d_rhs, d_lhs, trans="N", d_status=None):
        return self._L.blu_batch_solve_dense_dev(self._h, d_rhs, d_lhs, _ch(trans), d_status)

    # The basis-change step on torch tensors in device memory (blu_batch_*_dev).  Index arrays are int64, values
    # float64, masks and statuses int32 (a mask may also be bool); every tensor is contiguous and on the batch's CUDA
    # device.  On the SIMT emulator library, "device" memory is host memory, and CPU tensors are what it takes.
    # Outputs come back as tensors; out tensors passed in are written in place, and the entries of bases or units that
    # do not run keep what they held (zeros when the call allocates them).

    def _out(self, t, dtype, numel, name, dev, shape):
        import torch
        if t is None:
            return torch.zeros(shape, dtype=dtype, device=dev)
        return self._tensor(t, dtype, numel, name, dev)

    def _run_mask(self, run, dev):
        import torch
        if run is None:
            return None
        if isinstance(run, torch.Tensor) and run.dtype == torch.bool:
            self._tensor(run, torch.bool, self.nmat, "run", dev)
            return run.to(torch.int32)
        return self._tensor(run, torch.int32, self.nmat, "run", dev)

    def factorize_subset_dev(self, b_begin, b_end, b_i, b_x, run=None, status=None):
        """Refactorize the bases whose run flag is set (every basis for run=None) from B in device memory: column j of
        basis k is b_i/b_x[b_begin[k*m+j] : b_end[k*m+j]].  Returns (status, status per basis)."""
        import torch
        dev = self._torch_device()
        n, m = self.nmat, self.m
        bb = self._tensor(b_begin, torch.int64, n * m, "b_begin", dev)
        be = self._tensor(b_end, torch.int64, n * m, "b_end", dev)
        bi = self._tensor(b_i, torch.int64, None, "b_i", dev)
        bx = self._tensor(b_x, torch.float64, bi.numel(), "b_x", dev)
        r = self._run_mask(run, dev)
        stat = self._out(status, torch.int32, n, "status", dev, (n,))
        st = self._on_stream(dev, lambda: self._L.blu_batch_factorize_subset_dev(
            self._h, self._ptr(r), self._ptr(bb), self._ptr(be), self._ptr(bi), self._ptr(bx), bi.numel(), self._ptr(stat)))
        return st, stat

    def solve_for_update_dev(self, rhs_begin, irhs, xrhs=None, trans="N", want_solution=0, run=None,
                             status=None, nzlhs=None, ilhs=None, xlhs=None):
        """solve_for_update on the bases whose run flag is set: basis k's right-hand side is
        irhs/xrhs[rhs_begin[k] : rhs_begin[k+1]].  Returns (status, status[nmat], nzlhs[nmat], ilhs[nmat, m],
        xlhs[nmat, m]); the last three are None without want_solution.  Entry n of basis k's solution is
        lhs[ilhs[k, n]] = xlhs[k, n] for n < nzlhs[k]."""
        import torch
        dev = self._torch_device()
        n, m = self.nmat, self.m
        rb = self._tensor(rhs_begin, torch.int64, n + 1, "rhs_begin", dev)
        ir = self._tensor(irhs, torch.int64, None, "irhs", dev)
        xr = self._tensor(xrhs, torch.float64, ir.numel(), "xrhs", dev) if xrhs is not None else None
        r = self._run_mask(run, dev)
        stat = self._out(status, torch.int32, n, "status", dev, (n,))
        nz = il = xl = None
        if want_solution:
            nz = self._out(nzlhs, torch.int64, n, "nzlhs", dev, (n,))
            il = self._out(ilhs, torch.int64, n * m, "ilhs", dev, (n, m))
            xl = self._out(xlhs, torch.float64, n * m, "xlhs", dev, (n, m))
        st = self._on_stream(dev, lambda: self._L.blu_batch_solve_for_update_dev(
            self._h, self._ptr(r), self._ptr(rb), self._ptr(ir), self._ptr(xr), 1 if want_solution else 0,
            self._ptr(nz), self._ptr(il), self._ptr(xl), self._ptr(stat), _ch(trans)))
        return st, stat, nz, il, xl

    def update_dev(self, xtbl, run=None, status=None):
        """update on the bases whose run flag is set, basis k with xtbl[k].  Returns (status, status[nmat])."""
        import torch
        dev = self._torch_device()
        x = self._tensor(xtbl, torch.float64, self.nmat, "xtbl", dev)
        r = self._run_mask(run, dev)
        stat = self._out(status, torch.int32, self.nmat, "status", dev, (self.nmat,))
        st = self._on_stream(dev, lambda: self._L.blu_batch_update_dev(self._h, self._ptr(r), self._ptr(x), self._ptr(stat)))
        return st, stat

    def solve_sparse_dev(self, unit_begin, rhs_begin, irhs, xrhs, trans="N", nunits=None,
                         status=None, nzlhs=None, ilhs=None, xlhs=None):
        """solve_sparse for every unit: basis k owns units unit_begin[k] : unit_begin[k+1], unit u solves with
        irhs/xrhs[rhs_begin[u] : rhs_begin[u+1]].  nunits is read from unit_begin[-1] when not given (one small copy
        to the host).  Returns (status, status[nunits], nzlhs[nunits], ilhs[nunits, m], xlhs[nunits, m])."""
        import torch
        dev = self._torch_device()
        m = self.m
        ub = self._tensor(unit_begin, torch.int64, self.nmat + 1, "unit_begin", dev)
        nu = int(ub[-1].item()) if nunits is None else int(nunits)
        if nu < 0:
            raise ValueError("nunits < 0")
        rb = self._tensor(rhs_begin, torch.int64, nu + 1, "rhs_begin", dev)
        ir = self._tensor(irhs, torch.int64, None, "irhs", dev)
        xr = self._tensor(xrhs, torch.float64, ir.numel(), "xrhs", dev)
        stat = self._out(status, torch.int32, nu, "status", dev, (nu,))
        nz = self._out(nzlhs, torch.int64, nu, "nzlhs", dev, (nu,))
        il = self._out(ilhs, torch.int64, nu * m, "ilhs", dev, (nu, m))
        xl = self._out(xlhs, torch.float64, nu * m, "xlhs", dev, (nu, m))
        st = self._on_stream(dev, lambda: self._L.blu_batch_solve_sparse_dev(
            self._h, nu, self._ptr(ub), self._ptr(rb), self._ptr(ir), self._ptr(xr), self._ptr(nz), self._ptr(il), self._ptr(xl),
            self._ptr(stat), _ch(trans)))
        return st, stat, nz, il, xl

    def solve_dense_multi_dev(self, rhs, trans="N", lhs=None, status=None):
        """rhs[nmat, nrhs, m] (any contiguous tensor of nmat*nrhs*m values) -> (status, lhs[nmat, nrhs, m],
        status[nmat, nrhs]): solve_dense for every right-hand side of every basis."""
        import torch
        dev = self._torch_device()
        n, m = self.nmat, self.m
        r = self._tensor(rhs, torch.float64, None, "rhs", dev)
        if r.numel() % (n * m):
            raise ValueError("rhs: not a whole number of right-hand sides per basis")
        nrhs = r.numel() // (n * m)
        x = self._out(lhs, torch.float64, r.numel(), "lhs", dev, (n, nrhs, m))
        stat = self._out(status, torch.int32, n * nrhs, "status", dev, (n, nrhs))
        st = self._on_stream(dev, lambda: self._L.blu_batch_solve_dense_multi_dev(
            self._h, nrhs, self._ptr(r), self._ptr(x), _ch(trans), self._ptr(stat)))
        return st, x, stat

    def copy(self, dst, src):
        """Basis dst[r] becomes a copy of basis src[r] (factors, update history, a pending solve_for_update, getters,
        store capacities and resident B): from then on it behaves as src[r] would.  Returns the status."""
        d, s = _i64(dst).reshape(-1), _i64(src).reshape(-1)
        if len(d) != len(s):
            raise ValueError("dst and src differ in length")
        return self._L.blu_batch_copy(self._h, len(d), _pi(d), _pi(s))

    def copy_dev(self, from_):
        """copy with the map in device memory: from_ is an int32 tensor of nmat entries on the batch's device,
        from_[k] = -1 keeps basis k, otherwise basis k becomes a copy of basis from_[k].  Returns the status."""
        import torch
        dev = self._torch_device()
        f = self._tensor(from_, torch.int32, self.nmat, "from_", dev)
        return self._on_stream(dev, lambda: self._L.blu_batch_copy_dev(self._h, self._ptr(f)))

    # Images (blu_batch_save / blu_batch_restore): a basis' factorization and update history as bytes the caller owns,
    # restorable into any slot of any batch of the same m.

    def _save(self, fn, idx, bufs):
        """one save call; bufs = None: the size query.  Returns (status, sizes)."""
        s = _i64(idx).reshape(-1)
        n = len(s)
        nbytes = np.zeros(n, np.int64)
        if bufs is None:
            return fn(self._h, n, _pi(s), None, None, _pi(nbytes)), nbytes
        ptrs = (ctypes.c_void_p * max(n, 1))(*[b[0] for b in bufs])
        cap = _i64([b[1] for b in bufs])
        return fn(self._h, n, _pi(s), ptrs, _pi(cap), _pi(nbytes)), nbytes

    def save(self, idx):
        """The images of bases idx (repeats allowed) as a list of numpy.uint8 arrays.  Raises on a failed call."""
        L = self._L.blu_batch_save
        st, nbytes = self._save(L, idx, None)
        if st != 0:
            raise ValueError(f"blu_batch_save: status {st}")
        out = [self._aligned_host(b) for b in nbytes]
        st, _ = self._save(L, idx, [(a.ctypes.data, a.size) for a in out])
        if st != 0:
            raise ValueError(f"blu_batch_save: status {st}")
        return out

    def restore(self, dst, images):
        """Basis dst[r] becomes the basis saved in images[r] (a buffer of bytes: numpy.uint8 arrays, bytes, ...).
        Returns the status."""
        d = _i64(dst).reshape(-1)
        if len(d) != len(images):
            raise ValueError("dst and images differ in length")
        bufs = []
        for im in images:
            a = np.frombuffer(im, np.uint8) if not isinstance(im, np.ndarray) else np.ascontiguousarray(im).view(np.uint8).reshape(-1)
            if a.ctypes.data % 16:
                b = self._aligned_host(a.size)
                b[:] = a
                a = b
            bufs.append(a)
        ptrs = (ctypes.c_void_p * max(len(d), 1))(*[a.ctypes.data for a in bufs])
        cap = _i64([a.size for a in bufs])
        return self._L.blu_batch_restore(self._h, len(d), _pi(d), ptrs, _pi(cap))

    def save_dev(self, idx):
        """The images of bases idx as a list of 1-D torch.uint8 tensors on the batch's device: views into one
        allocation, each starting 256-byte aligned.  Ordered after torch's current stream.  Raises on a failed call."""
        import torch
        dev = self._torch_device()
        L = self._L.blu_batch_save_dev
        st, nbytes = self._on_stream(dev, lambda: self._save(L, idx, None))
        if st != 0:
            raise ValueError(f"blu_batch_save_dev: status {st}")
        size = [(int(b) + 255) & ~255 for b in nbytes]
        block = torch.empty(sum(size) + 256, dtype=torch.uint8, device=dev)
        at = (-block.data_ptr()) % 256
        out = []
        for b, z in zip(nbytes, size):
            out.append(block[at:at + int(b)])
            at += z
        st, _ = self._on_stream(dev, lambda: self._save(L, idx, [(t.data_ptr(), t.numel()) for t in out]))
        if st != 0:
            raise ValueError(f"blu_batch_save_dev: status {st}")
        return out

    def restore_dev(self, dst, images):
        """restore from contiguous torch.uint8 tensors on the batch's device.  Returns the status."""
        import torch
        dev = self._torch_device()
        d = _i64(dst).reshape(-1)
        if len(d) != len(images):
            raise ValueError("dst and images differ in length")
        ts = [self._tensor(t, torch.uint8, None, f"images[{r}]", dev) for r, t in enumerate(images)]
        ptrs = (ctypes.c_void_p * max(len(d), 1))(*[t.data_ptr() for t in ts])
        cap = _i64([t.numel() for t in ts])
        return self._on_stream(dev, lambda: self._L.blu_batch_restore_dev(self._h, len(d), _pi(d), ptrs, _pi(cap)))

    def graph_capture(self, trans="N"):
        return self._L.blu_batch_graph_capture(self._h, _ch(trans))

    def graph_launch(self):
        return self._L.blu_batch_graph_launch(self._h)

    def solve_dense_resident(self, trans="N"):
        return self._L.blu_batch_solve_dense_resident(self._h, _ch(trans))

    def download(self):
        x = np.zeros(self.nmat * self.m)
        status = np.zeros(self.nmat, dtype=np.int32)
        st = self._L.blu_batch_download(self._h, _pf(x), status.ctypes.data_as(i32p))
        return st, x.reshape(self.nmat, self.m), status

    def last_kernel_ms(self, which):
        return self._L.blu_batch_last_kernel_ms(self._h, int(which))

    def launch_count(self):
        return self._L.blu_batch_launch_count(self._h)

    def set_stream(self, stream_ptr):
        return self._L.blu_batch_set_stream(self._h, ctypes.c_void_p(stream_ptr))

    def synchronize(self):
        return self._L.blu_batch_synchronize(self._h)


class BLUMulti:
    """One batch of independent bases spread over several GPUs of this process (blu_multi_*: contiguous
    ranges per device, one host thread and stream each, no collective -- SURVEY.md 8e)."""

    def __init__(self, nmat, m, bnz_cap, devices, lib=None):
        self._L = lib or load_library()
        self.nmat, self.m = int(nmat), int(m)
        dev = np.ascontiguousarray(devices, dtype=np.int32)
        h = ctypes.c_void_p()
        st = self._L.blu_multi_create(ctypes.byref(h), self.nmat, self.m, int(bnz_cap), dev.ctypes.data_as(i32p), len(dev))
        if st != 0:
            raise RuntimeError(f"blu_multi_create failed with status {st} (no CUDA device? there is no CPU path)")
        self._h = h
        self.ndev = len(dev)

    def factorize_solve(self, b_begin, b_end, b_i, b_x, rhs=None, trans="N"):
        bb, be, bi, bx = _i64(b_begin), _i64(b_end), _i64(b_i), _f64(b_x)
        status = np.zeros(self.nmat, dtype=np.int32)
        r = _f64(rhs).reshape(-1) if rhs is not None else None
        x = np.zeros(self.nmat * self.m) if rhs is not None else None
        st = self._L.blu_multi_factorize_solve(self._h, _pi(bb), _pi(be), _pi(bi), _pf(bx), len(bi), _pf(r), _pf(x), _ch(trans), status.ctypes.data_as(i32p))
        return st, (x.reshape(self.nmat, self.m) if x is not None else None), status

    def part(self, d):
        """(batch handle usable with blu_batch_get_info / get_factors, first basis, number of bases) of device slot d"""
        first, count = ctypes.c_int64(), ctypes.c_int64()
        h = self._L.blu_multi_part(self._h, int(d), ctypes.byref(first), ctypes.byref(count))
        return h, first.value, count.value

    def info(self, k, name):
        for d in range(self.ndev):
            h, first, count = self.part(d)
            if first <= k < first + count:
                return self._L.blu_batch_get_info(h, int(k - first), I[name])
        raise IndexError(k)

    def close(self):
        if getattr(self, "_h", None):
            self._L.blu_multi_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass
