"""ctypes binding of the C-ABI in include/moolib_b200.h (used by tests, bench.py and __graft_entry__.smoke()).

There is deliberately NO fallback: if libmoolib_b200.so is missing or a call fails, this raises.
"""
import ctypes
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "lib", "libmoolib_b200.so")

MB_OK, MB_EINVAL, MB_ECUDA, MB_ETIMEOUT, MB_ESTATE, MB_ENOMEM = 0, -1, -2, -3, -4, -5
MB_AR_ALGO_AUTO, MB_AR_ALGO_ONESHOT, MB_AR_ALGO_TWOSHOT = 0, 1, 2
MB_AR_HANDLE_BYTES = 192
MB_AR_MAX_WORLD = 8
MB_AR_MAX_SLOTS = 4
MB_AR_BUFS_PER_SLOT = 3
MB_AR_SHORT = 1
MB_COPY_MAX_INLINE_JOBS = 512
MB_SRC_UNKNOWN, MB_SRC_DEVICE, MB_SRC_HOST_MAPPED = 0, 1, 2
MB_DT_F32, MB_DT_BF16, MB_DT_F16 = 0, 1, 2

# every symbol include/moolib_b200.h declares (tests check the .so exports all of them)
SYMBOLS = [
    "mb_version", "mb_last_error", "mb_sm_count",
    "mb_copy2d_batch", "mb_copy2d_batch_ex", "mb_copy_ctx_create", "mb_copy_ctx_destroy", "mb_copy2d_table",
    "mb_gather_rows", "mb_stack_slot", "mb_cat_narrow", "mb_scatter_actions",
    "mb_ar_ctx_create", "mb_ar_ctx_destroy", "mb_ar_ctx_export", "mb_ar_ctx_import", "mb_ar_ctx_reset",
    "mb_ar_staging", "mb_ar_world", "mb_ar_rank", "mb_ar_stage", "mb_ar_allreduce", "mb_ar_result",
    "mb_ar_flat_numel", "mb_ar_abort", "mb_ar_buffer", "mb_ar_slot_advance", "mb_ar_reduce_gated", "mb_ar_round_times", "mb_vtrace_f32", "mb_u8_to_f32", "mb_ar_xfer_pack", "mb_ar_xfer_unpack", "mb_ar_algo_for",
    "mb_ar_layout", "mb_ar_stage_ex", "mb_ar_allreduce_ex", "mb_ar_reduce_gated_ex",
]


class MoolibB200Error(RuntimeError):
    def __init__(self, code, msg):
        super().__init__(f"moolib_b200 error {code}: {msg}")
        self.code = code


class CopyJob(ctypes.Structure):
    _fields_ = [
        ("src", ctypes.c_void_p), ("dst", ctypes.c_void_p), ("row_bytes", ctypes.c_uint64),
        ("rows", ctypes.c_uint64), ("src_pitch", ctypes.c_int64), ("dst_pitch", ctypes.c_int64),
    ]


class ArHdr(ctypes.Structure):
    _fields_ = [
        ("num_gradients", ctypes.c_uint64), ("num_skipped", ctypes.c_uint64), ("batch_size", ctypes.c_uint64),
        ("has_grads", ctypes.c_uint64),
    ]


class ArSegment(ctypes.Structure):
    _fields_ = [("begin", ctypes.c_uint64), ("end", ctypes.c_uint64), ("dtype", ctypes.c_int32),
                ("reserved", ctypes.c_int32)]


class ArHandle(ctypes.Structure):
    _fields_ = [("bytes", ctypes.c_ubyte * MB_AR_HANDLE_BYTES)]


_lib = None


def load():
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise ImportError(
            f"{LIB_PATH} is missing: build it with `python moolib_b200/build.py` (nvcc, sm_100a). "
            "There is no CPU fallback for the moolib_b200 hot paths.")
    L = ctypes.CDLL(LIB_PATH)
    vp, u64, i64, ci, u32 = ctypes.c_void_p, ctypes.c_uint64, ctypes.c_int64, ctypes.c_int, ctypes.c_uint32
    L.mb_version.restype = ci
    L.mb_last_error.restype = ctypes.c_char_p
    L.mb_sm_count.argtypes = [ci]
    L.mb_copy2d_batch.argtypes = [ctypes.POINTER(CopyJob), ci, vp]
    L.mb_copy2d_batch_ex.argtypes = [ctypes.POINTER(CopyJob), ci, ci, vp]
    L.mb_copy_ctx_create.argtypes = [ci, u32, ctypes.POINTER(vp)]
    L.mb_copy_ctx_destroy.argtypes = [vp]
    L.mb_copy2d_table.argtypes = [vp, ctypes.POINTER(CopyJob), ci, ci, vp]
    L.mb_gather_rows.argtypes = [vp, u64, vp, u64, u64, vp]
    L.mb_stack_slot.argtypes = [vp, u64, u64, u64, u64, vp, vp]
    L.mb_cat_narrow.argtypes = [vp, vp, u64, u64, u64, u64, u64, u64, u64, vp]
    L.mb_scatter_actions.argtypes = [vp, u64, vp, u64, vp]
    L.mb_ar_ctx_create.argtypes = [ci, ci, ci, u64, ci, ctypes.POINTER(vp)]
    L.mb_ar_ctx_destroy.argtypes = [vp]
    L.mb_ar_ctx_export.argtypes = [vp, ctypes.POINTER(ArHandle)]
    L.mb_ar_ctx_import.argtypes = [vp, ci, ctypes.POINTER(ArHandle)]
    L.mb_ar_ctx_reset.argtypes = [vp, ci, ci]
    L.mb_ar_staging.argtypes = [vp, ci]
    L.mb_ar_staging.restype = vp
    L.mb_ar_world.argtypes = [vp]
    L.mb_ar_rank.argtypes = [vp]
    L.mb_ar_stage.argtypes = [vp, ci, ctypes.POINTER(vp), ctypes.POINTER(u64), ci, ci, ci, vp]
    L.mb_ar_allreduce.argtypes = [vp, ci, ctypes.POINTER(ArHdr), ctypes.POINTER(vp), ctypes.POINTER(u64), ci, vp,
                                  u64, ci, ci, u32, vp]
    L.mb_ar_result.argtypes = [vp, ci, ctypes.POINTER(ArHdr), ctypes.POINTER(ci)]
    L.mb_ar_flat_numel.argtypes = [ctypes.POINTER(u64), ci]
    L.mb_ar_flat_numel.restype = u64
    L.mb_ar_abort.argtypes = [vp]
    L.mb_ar_algo_for.argtypes = [vp, u64]
    L.mb_ar_xfer_pack.argtypes = [vp, ctypes.POINTER(vp), ctypes.POINTER(u64), ci, vp]
    L.mb_ar_xfer_unpack.argtypes = [vp, ci, ctypes.POINTER(vp), ctypes.POINTER(u64), ci, vp]
    L.mb_vtrace_f32.argtypes = [vp, vp, vp, vp, vp, ci, ctypes.c_float, ci, ctypes.c_float, u64, u64, vp, vp, vp]
    L.mb_u8_to_f32.argtypes = [vp, vp, u64, ctypes.c_float, vp]
    L.mb_ar_buffer.argtypes = [vp, ci, ci]
    L.mb_ar_buffer.restype = vp
    L.mb_ar_slot_advance.argtypes = [vp, ci]
    L.mb_ar_reduce_gated.argtypes = [vp, ci, ctypes.POINTER(ArHdr), u64, ctypes.POINTER(vp), ctypes.POINTER(u64), ci, vp,
                                     u64, ci, ci, u32, vp]
    L.mb_ar_round_times.argtypes = [vp, ci, ctypes.POINTER(ctypes.c_float), ctypes.POINTER(ctypes.c_float)]
    i32p = ctypes.POINTER(ctypes.c_int32)
    L.mb_ar_layout.argtypes = [ctypes.POINTER(u64), i32p, ci, ctypes.POINTER(u64), ctypes.POINTER(u64),
                               ctypes.POINTER(ArSegment)]
    L.mb_ar_stage_ex.argtypes = [vp, ci, ctypes.POINTER(vp), ctypes.POINTER(u64), i32p, ci, ci, ci, vp]
    L.mb_ar_allreduce_ex.argtypes = [vp, ci, ctypes.POINTER(ArHdr), ctypes.POINTER(vp), ctypes.POINTER(u64), i32p, ci,
                                     vp, u64, ci, ci, u32, vp]
    L.mb_ar_reduce_gated_ex.argtypes = [vp, ci, ctypes.POINTER(ArHdr), u64, ctypes.POINTER(vp), ctypes.POINTER(u64),
                                        i32p, ci, vp, u64, ci, ci, u32, vp]
    _lib = L
    return L


def check(rc):
    """Raise on a negative return code; pass the (non-negative) value through."""
    if rc < 0:
        raise MoolibB200Error(rc, load().mb_last_error().decode("utf-8", "replace"))
    return rc


def _stream_ptr(stream):
    if stream is None:
        import torch
        return ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)
    if isinstance(stream, int):
        return ctypes.c_void_p(stream)
    return ctypes.c_void_p(stream.cuda_stream)


# ---------------------------------------------------------------------------------------------------------------
# thin helpers over torch tensors (torch is only the owner of device memory and streams here)
# ---------------------------------------------------------------------------------------------------------------

def make_jobs(jobs):
    """jobs: iterable of (src_ptr, dst_ptr, row_bytes, rows, src_pitch, dst_pitch)."""
    arr = (CopyJob * len(jobs))()
    for i, j in enumerate(jobs):
        arr[i].src, arr[i].dst, arr[i].row_bytes, arr[i].rows, arr[i].src_pitch, arr[i].dst_pitch = j
    return arr


def copy2d_batch(jobs, stream=None):
    arr = jobs if isinstance(jobs, ctypes.Array) else make_jobs(list(jobs))
    return check(load().mb_copy2d_batch(arr, len(arr), _stream_ptr(stream)))


class CopyContext:
    """Staging for device-resident job tables (mb_copy_ctx): any number of pitched copies in one launch."""

    def __init__(self, device, max_jobs=8192):
        self.L = load()
        self._ctx = ctypes.c_void_p()
        check(self.L.mb_copy_ctx_create(device, max_jobs, ctypes.byref(self._ctx)))

    def close(self):
        if self._ctx:
            self.L.mb_copy_ctx_destroy(self._ctx)
            self._ctx = ctypes.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def copy(self, jobs, src_kind=MB_SRC_UNKNOWN, stream=None):
        arr = jobs if isinstance(jobs, ctypes.Array) else make_jobs(list(jobs))
        return check(self.L.mb_copy2d_table(self._ctx, arr, len(arr), src_kind, _stream_ptr(stream)))


def stack_slot(dst, slot, src, dim=0, stream=None):
    """dst.select(dim, slot).copy_(src) for contiguous dst/src through mb_stack_slot."""
    assert dst.is_contiguous() and src.is_contiguous()
    outer = 1
    for s in dst.shape[:dim]:
        outer *= s
    size = dst.shape[dim]
    inner = dst.element_size()
    for s in dst.shape[dim + 1:]:
        inner *= s
    assert src.numel() * src.element_size() == outer * inner, "shape mismatch"
    return check(load().mb_stack_slot(dst.data_ptr(), outer, size, slot, inner, src.data_ptr(), _stream_ptr(stream)))


def cat_narrow(dst, dst_off, src, src_off, n, dim=0, stream=None):
    """dst.narrow(dim, dst_off, n).copy_(src.narrow(dim, src_off, n)) for contiguous tensors."""
    assert dst.is_contiguous() and src.is_contiguous()
    outer = 1
    for s in dst.shape[:dim]:
        outer *= s
    inner = dst.element_size()
    for s in dst.shape[dim + 1:]:
        inner *= s
    return check(load().mb_cat_narrow(dst.data_ptr(), src.data_ptr(), outer, dst.shape[dim], dst_off, src.shape[dim],
                                      src_off, n, inner, _stream_ptr(stream)))


def gather_rows(dst, src_row_ptrs_dev, row_bytes, nrows, dst_pitch=None, stream=None):
    return check(load().mb_gather_rows(dst.data_ptr(), dst_pitch or row_bytes, src_row_ptrs_dev.data_ptr(), row_bytes,
                                       nrows, _stream_ptr(stream)))


class ArContext:
    """One rank's allreduce context (mb_ar_ctx)."""

    def __init__(self, rank, world, device, max_bytes, nslots=1):
        self.L = load()
        self._ctx = ctypes.c_void_p()
        check(self.L.mb_ar_ctx_create(rank, world, device, max_bytes, nslots, ctypes.byref(self._ctx)))
        self.rank, self.world, self.device, self.max_bytes, self.nslots = rank, world, device, max_bytes, nslots

    def close(self):
        if self._ctx:
            self.L.mb_ar_ctx_destroy(self._ctx)
            self._ctx = ctypes.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def export(self) -> bytes:
        h = ArHandle()
        check(self.L.mb_ar_ctx_export(self._ctx, ctypes.byref(h)))
        return bytes(h.bytes)

    def import_peer(self, peer_rank, handle_bytes: bytes):
        h = ArHandle()
        ctypes.memmove(h.bytes, handle_bytes, MB_AR_HANDLE_BYTES)
        check(self.L.mb_ar_ctx_import(self._ctx, peer_rank, ctypes.byref(h)))

    def reset(self, rank, world):
        check(self.L.mb_ar_ctx_reset(self._ctx, rank, world))
        self.rank, self.world = rank, world

    def abort(self):
        check(self.L.mb_ar_abort(self._ctx))

    def staging_ptr(self, slot=0):
        return self.L.mb_ar_staging(self._ctx, slot)

    @staticmethod
    def _lists(tensors):
        n = len(tensors)
        ptrs = (ctypes.c_void_p * n)(*[t.data_ptr() for t in tensors])
        numel = (ctypes.c_uint64 * n)(*[t.numel() for t in tensors])
        return ptrs, numel, n

    def stage(self, tensors, slot=0, accumulate=False, zero_src=False, stream=None):
        ptrs, numel, n = self._lists(tensors)
        return check(self.L.mb_ar_stage(self._ctx, slot, ptrs, numel, n, int(accumulate), int(zero_src),
                                        _stream_ptr(stream)))

    def allreduce(self, dst_tensors, hdr=(1, 0, 1, 1), slot=0, scale=True, algo=MB_AR_ALGO_AUTO, timeout_ms=30000,
                  stream=None):
        ptrs, numel, n = self._lists(dst_tensors)
        h = ArHdr(*hdr)
        return check(self.L.mb_ar_allreduce(self._ctx, slot, ctypes.byref(h), ptrs, numel, n, None, 0, int(scale),
                                            algo, timeout_ms, _stream_ptr(stream)))

    def allreduce_flat(self, dst, hdr=(1, 0, 1, 1), slot=0, scale=False, algo=MB_AR_ALGO_AUTO, timeout_ms=30000,
                       stream=None):
        h = ArHdr(*hdr)
        return check(self.L.mb_ar_allreduce(self._ctx, slot, ctypes.byref(h), None, None, 0, dst.data_ptr(),
                                            dst.numel(), int(scale), algo, timeout_ms, _stream_ptr(stream)))

    def buffer_ptr(self, slot=0, ahead=0):
        return self.L.mb_ar_buffer(self._ctx, slot, ahead)

    def buffer(self, numel, slot=0, ahead=0):
        """The ring buffer `ahead` positions after the slot's current staging buffer, as a flat fp32 torch tensor
        (no copy: gradients written here are staged by construction)."""
        import torch

        class _Mem:
            pass

        m = _Mem()
        m.__cuda_array_interface__ = {"shape": (int(numel),), "typestr": "<f4", "version": 3,
                                      "data": (int(self.buffer_ptr(slot, ahead)), False)}
        with torch.cuda.device(self.device):
            return torch.as_tensor(m, device=f"cuda:{self.device}")

    def algo_for(self, nbytes):
        return check(self.L.mb_ar_algo_for(self._ctx, nbytes))

    def advance(self, slot=0):
        check(self.L.mb_ar_slot_advance(self._ctx, slot))

    def reduce_gated(self, min_batch, dst_tensors=None, flat_dst=None, hdr=(1, 0, 1, 1), slot=0, scale=True,
                     algo=MB_AR_ALGO_AUTO, timeout_ms=30000, stream=None):
        """K-A0 gate + K-A2 reduce; the caller advances the ring after seeing status MB_OK."""
        h = ArHdr(*hdr)
        if dst_tensors is not None:
            ptrs, numel, n = self._lists(dst_tensors)
            return check(self.L.mb_ar_reduce_gated(self._ctx, slot, ctypes.byref(h), min_batch, ptrs, numel, n, None, 0,
                                                   int(scale), algo, timeout_ms, _stream_ptr(stream)))
        return check(self.L.mb_ar_reduce_gated(self._ctx, slot, ctypes.byref(h), min_batch, None, None, 0,
                                               flat_dst.data_ptr(), flat_dst.numel(), int(scale), algo, timeout_ms,
                                               _stream_ptr(stream)))

    def round_times(self, slot=0):
        g, r = ctypes.c_float(), ctypes.c_float()
        check(self.L.mb_ar_round_times(self._ctx, slot, ctypes.byref(g), ctypes.byref(r)))
        return g.value, r.value

    def xfer_pack(self, tensors, stream=None):
        ptrs, numel, n = self._lists(tensors)
        return check(self.L.mb_ar_xfer_pack(self._ctx, ptrs, numel, n, _stream_ptr(stream)))

    def xfer_unpack(self, src_rank, tensors, stream=None):
        ptrs, numel, n = self._lists(tensors)
        return check(self.L.mb_ar_xfer_unpack(self._ctx, src_rank, ptrs, numel, n, _stream_ptr(stream)))

    # ---- mixed-dtype lists (fp32 / bf16 / fp16): the _ex entry points, layout of mb_ar_layout ----
    @staticmethod
    def _lists_ex(tensors):
        n = len(tensors)
        ptrs = (ctypes.c_void_p * n)(*[t.data_ptr() for t in tensors])
        numel = (ctypes.c_uint64 * n)(*[t.numel() for t in tensors])
        dts = (ctypes.c_int32 * n)(*[dtype_code(t.dtype) for t in tensors])
        return ptrs, numel, dts, n

    def stage_ex(self, tensors, slot=0, accumulate=False, zero_src=False, stream=None):
        ptrs, numel, dts, n = self._lists_ex(tensors)
        return check(self.L.mb_ar_stage_ex(self._ctx, slot, ptrs, numel, dts, n, int(accumulate), int(zero_src),
                                           _stream_ptr(stream)))

    def _reduce_ex(self, gated, min_batch, tensors, flat_dst, hdr, slot, scale, algo, timeout_ms, stream):
        """tensors: the destination list, or (flat_dst given) tensors / (numel, torch dtype) pairs describing the
        layout of the flat uint8 result buffer."""
        h = ArHdr(*hdr)
        if flat_dst is None:
            ptrs, numel, dts, n = self._lists_ex(tensors)
            flat_ptr, flat_bytes = None, 0
        else:
            desc = [(t.numel(), t.dtype) if hasattr(t, "numel") else t for t in tensors]
            n = len(desc)
            ptrs = None
            numel = (ctypes.c_uint64 * n)(*[m for m, _ in desc])
            dts = (ctypes.c_int32 * n)(*[dtype_code(d) for _, d in desc])
            flat_ptr, flat_bytes = flat_dst.data_ptr(), flat_dst.numel() * flat_dst.element_size()
        if gated:
            return check(self.L.mb_ar_reduce_gated_ex(self._ctx, slot, ctypes.byref(h), min_batch, ptrs, numel, dts, n,
                                                      flat_ptr, flat_bytes, int(scale), algo, timeout_ms,
                                                      _stream_ptr(stream)))
        return check(self.L.mb_ar_allreduce_ex(self._ctx, slot, ctypes.byref(h), ptrs, numel, dts, n, flat_ptr,
                                               flat_bytes, int(scale), algo, timeout_ms, _stream_ptr(stream)))

    def allreduce_ex(self, tensors, flat_dst=None, hdr=(1, 0, 1, 1), slot=0, scale=True, algo=MB_AR_ALGO_AUTO,
                     timeout_ms=30000, stream=None):
        return self._reduce_ex(False, 0, tensors, flat_dst, hdr, slot, scale, algo, timeout_ms, stream)

    def reduce_gated_ex(self, min_batch, tensors, flat_dst=None, hdr=(1, 0, 1, 1), slot=0, scale=True,
                        algo=MB_AR_ALGO_AUTO, timeout_ms=30000, stream=None):
        return self._reduce_ex(True, min_batch, tensors, flat_dst, hdr, slot, scale, algo, timeout_ms, stream)

    def buffer_bytes(self, nbytes, slot=0, ahead=0):
        """Like buffer(), as a flat uint8 tensor of `nbytes` (view it per tensor with layout() offsets)."""
        import torch

        class _Mem:
            pass

        m = _Mem()
        m.__cuda_array_interface__ = {"shape": (int(nbytes),), "typestr": "|u1", "version": 3,
                                      "data": (int(self.buffer_ptr(slot, ahead)), False)}
        with torch.cuda.device(self.device):
            return torch.as_tensor(m, device=f"cuda:{self.device}")

    def result(self, slot=0):
        h = ArHdr()
        st = ctypes.c_int()
        check(self.L.mb_ar_result(self._ctx, slot, ctypes.byref(h), ctypes.byref(st)))
        return (h.num_gradients, h.num_skipped, h.batch_size, h.has_grads), st.value


def flat_numel(numels):
    arr = (ctypes.c_uint64 * len(numels))(*numels)
    return load().mb_ar_flat_numel(arr, len(numels))


def dtype_code(dt):
    """MB_DT_* of a torch dtype (or of the strings 'f32', 'bf16', 'f16')."""
    name = str(dt).replace("torch.", "")
    codes = {"float32": MB_DT_F32, "f32": MB_DT_F32, "bfloat16": MB_DT_BF16, "bf16": MB_DT_BF16,
             "float16": MB_DT_F16, "f16": MB_DT_F16}
    if name not in codes:
        raise ValueError(f"unsupported allreduce dtype {dt}; supported: float32, bfloat16, float16")
    return codes[name]


def layout(numels, dtypes):
    """mb_ar_layout: (per-tensor byte offsets, total bytes, [(begin, end, MB_DT_*) per dtype segment])."""
    n = len(numels)
    nm = (ctypes.c_uint64 * max(n, 1))(*numels)
    dt = (ctypes.c_int32 * max(n, 1))(*[dtype_code(d) if not isinstance(d, int) else d for d in dtypes])
    off = (ctypes.c_uint64 * max(n, 1))()
    total = ctypes.c_uint64()
    segs = (ArSegment * 3)()
    nseg = check(load().mb_ar_layout(nm, dt, n, off, ctypes.byref(total), segs))
    return list(off)[:n], total.value, [(segs[k].begin, segs[k].end, segs[k].dtype) for k in range(nseg)]
