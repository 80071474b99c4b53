"""ctypes mirror of the library's C-ABI, with the reference's own names.

``VfgsHw`` exposes the ten functions of the reference's ``src/vfgs_hw.h:51-62`` (bound to the CUDA
shim) plus the additive frame entry points of ``include/vfgs_b200.h``. Like the reference there is
ONE hardware state per process (``src/vfgs_hw.c:49-63`` are file-scope statics), so every instance
talks to the same state. ``Session`` objects (``VfgsHw.create_session``) hold independent copies of
it, one per video stream, which ``VfgsHw.add_grain_jobs_device`` serves in one batched call. Nothing
here computes grain: without the compiled CUDA library the import of the library fails loudly.
"""
from __future__ import annotations

import ctypes as C
import os

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, "libvfgs_b200.so")

HW_SYMBOLS = (
    "vfgs_set_luma_pattern", "vfgs_set_chroma_pattern", "vfgs_set_scale_lut", "vfgs_set_pattern_lut",
    "vfgs_set_seed", "vfgs_set_scale_shift", "vfgs_set_depth", "vfgs_set_legal_range",
    "vfgs_set_chroma_subsampling", "vfgs_add_grain_line",
)
B200_SYMBOLS = (
    "vfgs_b200_init", "vfgs_b200_reset", "vfgs_b200_last_error", "vfgs_b200_frame_bytes",
    "vfgs_b200_add_grain_frames_device", "vfgs_b200_add_grain_planes_device",
    "vfgs_b200_add_grain_frames_host", "vfgs_b200_skip_frames", "vfgs_b200_get_lfsr",
    "vfgs_b200_set_lfsr", "vfgs_b200_host_alloc", "vfgs_b200_host_free", "vfgs_b200_launch_count",
    "vfgs_b200_last_launch", "vfgs_b200_get_state", "vfgs_b200_kernel_timing", "vfgs_b200_kernel_time",
    "vfgs_b200_force_general_kernel", "vfgs_b200_pipeline_stats", "vfgs_b200_init_sei", "vfgs_b200_init_afgs1",
    "vfgs_b200_add_grain_semiplanar_device", "vfgs_b200_session_create", "vfgs_b200_session_destroy",
    "vfgs_b200_session_get_lfsr", "vfgs_b200_session_set_lfsr", "vfgs_b200_session_skip_frames",
    "vfgs_b200_session_get_state", "vfgs_b200_add_grain_jobs_device", "vfgs_b200_session_set_seed",
    "vfgs_b200_session_init_metadata",
)
NV12, P010 = 1, 2  # VFGS_B200_NV12 / VFGS_B200_P010


class VfgsError(RuntimeError):
    pass


class Planes(C.Structure):
    """vfgs_b200_planes (include/vfgs_b200.h)."""
    _fields_ = [("y", C.c_void_p), ("u", C.c_void_p), ("v", C.c_void_p),
                ("stride_y", C.c_int64), ("stride_c", C.c_int64), ("frame_stride", C.c_int64)]


class SemiPlanes(C.Structure):
    """vfgs_b200_semiplanar (include/vfgs_b200.h): a Y plane and one plane of interleaved U,V pairs."""
    _fields_ = [("y", C.c_void_p), ("uv", C.c_void_p), ("stride_y", C.c_int64), ("stride_uv", C.c_int64),
                ("frame_stride", C.c_int64), ("format", C.c_int)]


def surface_planes(t, height: int, fmt: int) -> SemiPlanes:
    """The usual decoder surface: a CUDA tensor of shape (n, height + ch, pitch) (uint8 for NV12, 16-bit for P010;
    pitch in samples) holding per frame `height` Y rows and then the `ch` UV rows, all at the same pitch."""
    if t.dim() != 3 or not t.is_contiguous():
        raise VfgsError("surface must be a contiguous (n, height + ch, pitch) tensor")
    if t.element_size() != (2 if fmt == P010 else 1):
        raise VfgsError("NV12 surfaces hold 8-bit samples, P010 surfaces 16-bit ones")
    pitch = t.shape[2] * t.element_size()
    base = t.data_ptr()
    return SemiPlanes(base, base + height * pitch, pitch, pitch, t.shape[1] * pitch, fmt)


class _CMetadata(C.Structure):
    """vfgs_b200_session_metadata (include/vfgs_fw.h)."""
    _fields_ = [("session", C.c_void_p), ("sei", C.c_void_p), ("afgs1", C.c_void_p)]


class _CJob(C.Structure):
    """vfgs_b200_job (include/vfgs_b200.h)."""
    _fields_ = [("session", C.c_void_p), ("in_", C.POINTER(Planes)), ("out", C.POINTER(Planes)),
                ("sp_in", C.POINTER(SemiPlanes)), ("sp_out", C.POINTER(SemiPlanes)),
                ("nframes", C.c_int), ("width", C.c_int), ("height", C.c_int), ("out_depth", C.c_int)]


def _state_dict(raw: np.ndarray) -> dict:
    o = 2 * 9 * 64 * 64
    return {
        "pattern": raw[:o].view(np.int8).reshape(2, 9, 64, 64).copy(),
        "slut": raw[o:o + 768].reshape(3, 256).copy(),
        "plut": raw[o + 768:o + 1536].reshape(3, 256).copy(),
        "lfsr": raw[o + 1536:o + 1552].view(np.uint32).copy(),
        "scalars": raw[o + 1552:o + 1584].view(np.int32).copy(),
    }


_lib = None


def load_library(global_symbols: bool = False) -> C.CDLL:
    """dlopen libvfgs_b200.so (building it first if the sources are newer). ``global_symbols`` makes
    the vfgs_* symbols visible to libraries loaded afterwards (the reference firmware layer)."""
    global _lib
    if _lib is not None and not global_symbols:
        return _lib
    from .build import build
    build()
    if not os.path.exists(LIB_PATH):
        raise VfgsError(f"{LIB_PATH} is missing: the CUDA extension was not built")
    L = C.CDLL(LIB_PATH, mode=C.RTLD_GLOBAL if global_symbols else C.DEFAULT_MODE)
    vp, ci = C.c_void_p, C.c_int
    L.vfgs_set_luma_pattern.argtypes = [ci, vp]
    L.vfgs_set_chroma_pattern.argtypes = [ci, vp]
    L.vfgs_set_scale_lut.argtypes = [ci, vp]
    L.vfgs_set_pattern_lut.argtypes = [ci, vp]
    L.vfgs_set_seed.argtypes = [C.c_uint32]
    L.vfgs_set_scale_shift.argtypes = [ci]
    L.vfgs_set_depth.argtypes = [ci]
    L.vfgs_set_legal_range.argtypes = [ci]
    L.vfgs_set_chroma_subsampling.argtypes = [ci, ci]
    L.vfgs_add_grain_line.argtypes = [vp, vp, vp, ci, ci]
    for name in HW_SYMBOLS:
        getattr(L, name).restype = None
    L.vfgs_b200_init.argtypes = [ci]
    L.vfgs_b200_last_error.restype = C.c_char_p
    L.vfgs_b200_frame_bytes.argtypes = [ci, ci, ci]
    L.vfgs_b200_frame_bytes.restype = C.c_size_t
    L.vfgs_b200_add_grain_frames_device.argtypes = [vp, vp, ci, ci, ci, ci, vp]
    L.vfgs_b200_add_grain_planes_device.argtypes = [C.POINTER(Planes), C.POINTER(Planes), ci, ci, ci, ci, vp]
    L.vfgs_b200_add_grain_semiplanar_device.argtypes = [C.POINTER(SemiPlanes), C.POINTER(SemiPlanes), ci, ci, ci, vp]
    L.vfgs_b200_add_grain_frames_host.argtypes = [vp, vp, ci, ci, ci, ci]
    L.vfgs_b200_skip_frames.argtypes = [C.c_int64, ci, ci]
    L.vfgs_b200_get_lfsr.argtypes = [vp]
    L.vfgs_b200_get_lfsr.restype = None
    L.vfgs_b200_set_lfsr.argtypes = [vp]
    L.vfgs_b200_set_lfsr.restype = None
    L.vfgs_b200_host_alloc.argtypes = [C.c_size_t]
    L.vfgs_b200_host_alloc.restype = vp
    L.vfgs_b200_host_free.argtypes = [vp]
    L.vfgs_b200_host_free.restype = None
    L.vfgs_b200_launch_count.restype = C.c_uint64
    L.vfgs_b200_last_launch.argtypes = [vp]
    L.vfgs_b200_last_launch.restype = None
    L.vfgs_b200_kernel_timing.argtypes = [ci]
    L.vfgs_b200_kernel_time.argtypes = [C.POINTER(C.c_double), C.POINTER(C.c_uint64)]
    L.vfgs_b200_force_general_kernel.argtypes = [ci]
    L.vfgs_b200_force_general_kernel.restype = None
    L.vfgs_b200_init_sei.argtypes = [vp]
    L.vfgs_b200_init_afgs1.argtypes = [vp]
    L.vfgs_b200_get_state.argtypes = [vp, C.c_size_t]
    L.vfgs_b200_get_state.restype = C.c_size_t
    L.vfgs_b200_session_create.argtypes = [C.POINTER(vp)]
    L.vfgs_b200_session_destroy.argtypes = [vp]
    L.vfgs_b200_session_destroy.restype = None
    L.vfgs_b200_session_get_lfsr.argtypes = [vp, vp]
    L.vfgs_b200_session_get_lfsr.restype = None
    L.vfgs_b200_session_set_lfsr.argtypes = [vp, vp]
    L.vfgs_b200_session_set_lfsr.restype = None
    L.vfgs_b200_session_skip_frames.argtypes = [vp, C.c_int64, ci, ci]
    L.vfgs_b200_session_get_state.argtypes = [vp, vp, C.c_size_t]
    L.vfgs_b200_session_get_state.restype = C.c_size_t
    L.vfgs_b200_add_grain_jobs_device.argtypes = [C.POINTER(_CJob), ci, vp]
    L.vfgs_b200_session_set_seed.argtypes = [vp, C.c_uint32]
    L.vfgs_b200_session_init_metadata.argtypes = [C.POINTER(_CMetadata), ci, vp]
    _lib = L
    return L


def _np_ptr(a: np.ndarray):
    if not a.flags["C_CONTIGUOUS"]:
        raise VfgsError("array must be C-contiguous")
    return a.ctypes.data_as(C.c_void_p)


class VfgsHw:
    """The hardware layer, CUDA back end. Method names and argument meaning follow vfgs_hw.h."""

    def __init__(self, device: int | None = None, global_symbols: bool = False):
        self.L = load_library(global_symbols)
        if device is not None:
            self._chk(self.L.vfgs_b200_init(device))

    def _chk(self, rc: int) -> None:
        if rc != 0:
            raise VfgsError(f"vfgs_b200 error {rc}: {self.L.vfgs_b200_last_error().decode()}")

    # ---- vfgs_hw.h:51-62 ------------------------------------------------------------------
    def vfgs_set_luma_pattern(self, index, P): self.L.vfgs_set_luma_pattern(index, _np_ptr(P))
    def vfgs_set_chroma_pattern(self, index, P): self.L.vfgs_set_chroma_pattern(index, _np_ptr(P))
    def vfgs_set_scale_lut(self, c, lut): self.L.vfgs_set_scale_lut(c, _np_ptr(lut))
    def vfgs_set_pattern_lut(self, c, lut): self.L.vfgs_set_pattern_lut(c, _np_ptr(lut))
    def vfgs_set_seed(self, seed): self.L.vfgs_set_seed(seed & 0xFFFFFFFF)
    def vfgs_set_scale_shift(self, shift): self.L.vfgs_set_scale_shift(shift)
    def vfgs_set_depth(self, depth): self.L.vfgs_set_depth(depth)
    def vfgs_set_legal_range(self, legal): self.L.vfgs_set_legal_range(legal)
    def vfgs_set_chroma_subsampling(self, subx, suby): self.L.vfgs_set_chroma_subsampling(subx, suby)

    def vfgs_add_grain_line(self, Y, U, V, y, width):
        """One picture line of host memory (numpy arrays), in place."""
        self.L.vfgs_add_grain_line(_np_ptr(Y), _np_ptr(U), _np_ptr(V), y, width)

    # ---- vfgs_fw.h: the firmware layer with the pattern synthesis on the device ---------------
    def init_sei(self, raw: bytes):
        """raw: the bytes of an fgs_sei struct (src/vfgs_fw.h:53-62)."""
        buf = (C.c_uint8 * len(raw)).from_buffer_copy(raw)
        self._chk(self.L.vfgs_b200_init_sei(buf))

    def init_afgs1(self, raw: bytes):
        """raw: the bytes of an fgs_afgs1 struct (src/vfgs_fw.h:64-91)."""
        buf = (C.c_uint8 * len(raw)).from_buffer_copy(raw)
        self._chk(self.L.vfgs_b200_init_afgs1(buf))

    # ---- vfgs_b200.h ------------------------------------------------------------------------
    def reset(self): self._chk(self.L.vfgs_b200_reset())
    def frame_bytes(self, width, height, depth): return self.L.vfgs_b200_frame_bytes(width, height, depth)
    def skip_frames(self, n, width, height): self._chk(self.L.vfgs_b200_skip_frames(n, width, height))
    def launch_count(self) -> int: return int(self.L.vfgs_b200_launch_count())

    def kernel_timing(self, enable: bool): self._chk(self.L.vfgs_b200_kernel_timing(1 if enable else 0))

    def kernel_time(self):
        """(accumulated grain-kernel device ms, launches) since timing was enabled."""
        ms, n = C.c_double(0), C.c_uint64(0)
        self._chk(self.L.vfgs_b200_kernel_time(C.byref(ms), C.byref(n)))
        return ms.value, int(n.value)

    def force_general_kernel(self, mode): self.L.vfgs_b200_force_general_kernel(int(mode))

    def last_launch(self) -> dict:
        a = (C.c_int * 5)()
        self.L.vfgs_b200_last_launch(a)
        kernels = [n for bit, n in ((1, "fgs_apply_fast_kernel"), (8, "fgs_apply_fast_kernel<EDGE>"), (4, "fgs_apply_gather_kernel"), (2, "fgs_apply_kernel"),
                                           (16, "fgs_apply_fast_kernel<interleaved UV>")) if a[4] & bit]
        return {"grid": a[0], "block": a[1], "smem": a[2], "sms": a[3], "kernels": kernels}

    def state(self) -> dict:
        """Mirrored hw state as arrays (same keys as the oracle's/reference's state dumps)."""
        n = self.L.vfgs_b200_get_state(None, 0)
        buf = (C.c_uint8 * n)()
        self.L.vfgs_b200_get_state(buf, n)
        return _state_dict(np.frombuffer(bytes(buf), dtype=np.uint8))

    def get_lfsr(self):
        r = (C.c_uint32 * 4)()
        self.L.vfgs_b200_get_lfsr(r)
        return [int(v) for v in r]

    def set_lfsr(self, regs):
        r = (C.c_uint32 * 4)(*[int(v) & 0xFFFFFFFF for v in regs])
        self.L.vfgs_b200_set_lfsr(r)

    def add_grain_frames_device(self, src, dst, nframes, width, height, out_depth=0, stream=None):
        """src/dst: torch CUDA tensors (flat packed planar frames). Asynchronous on ``stream``
        (a torch.cuda.Stream; default: torch's current stream)."""
        import torch
        if stream is None:
            stream = torch.cuda.current_stream(src.device)
        self._chk(self.L.vfgs_b200_add_grain_frames_device(
            C.c_void_p(src.data_ptr()), C.c_void_p(dst.data_ptr()), nframes, width, height, out_depth,
            C.c_void_p(stream.cuda_stream)))

    def add_grain_frames_device_ptr(self, src_ptr, dst_ptr, nframes, width, height, out_depth=0, stream_ptr=0):
        self._chk(self.L.vfgs_b200_add_grain_frames_device(
            C.c_void_p(src_ptr), C.c_void_p(dst_ptr), nframes, width, height, out_depth, C.c_void_p(stream_ptr)))

    def add_grain_planes_device(self, pin: Planes, pout: Planes, nframes, width, height, out_depth=0, stream_ptr=0):
        self._chk(self.L.vfgs_b200_add_grain_planes_device(
            C.byref(pin), C.byref(pout), nframes, width, height, out_depth, C.c_void_p(stream_ptr)))

    def add_grain_semiplanar_device(self, pin: SemiPlanes, pout: SemiPlanes, nframes, width, height, stream_ptr=0):
        """Semi-planar (NV12 / P010) frames in device memory, see vfgs_b200_add_grain_semiplanar_device."""
        self._chk(self.L.vfgs_b200_add_grain_semiplanar_device(
            C.byref(pin), C.byref(pout), nframes, width, height, C.c_void_p(stream_ptr)))

    def add_grain_surfaces(self, src, dst, nframes, width, height, out_format=None, stream=None):
        """src/dst: decoder-style surfaces, CUDA tensors of shape (n, height + ch, pitch) (surface_planes). The input
        format follows the configured depth (NV12 for 8, P010 for 10); out_format defaults to the input format
        (NV12 from P010 is the fused 10 -> 8 conversion). src is dst for in place."""
        import torch
        if stream is None:
            stream = torch.cuda.current_stream(src.device)
        in_fmt = P010 if src.element_size() == 2 else NV12
        self.add_grain_semiplanar_device(surface_planes(src, height, in_fmt), surface_planes(dst, height, out_format or in_fmt),
                                         nframes, width, height, stream.cuda_stream)

    def add_grain_frames_host(self, src, dst, nframes, width, height, out_depth=0):
        """src/dst: host buffers (numpy arrays or pinned torch CPU tensors)."""
        def ptr(x):
            return _np_ptr(x) if isinstance(x, np.ndarray) else C.c_void_p(x.data_ptr())
        self._chk(self.L.vfgs_b200_add_grain_frames_host(ptr(src), ptr(dst), nframes, width, height, out_depth))

    # ---- sessions: one grain state per video stream, many streams per call -------------------------
    def create_session(self) -> "Session":
        """Snapshot of the current hardware state (registers included) as an independent session."""
        h = C.c_void_p()
        self._chk(self.L.vfgs_b200_session_create(C.byref(h)))
        return Session(self, h.value)

    def add_grain_jobs_device(self, jobs, stream=None):
        """jobs: a list of ``Job``s (device memory). One batched call, asynchronous on ``stream`` (a torch.cuda.Stream;
        default: torch's current stream), equal to one single-job call per job in list order."""
        import torch
        if stream is None:
            stream = torch.cuda.current_stream()
        arr = (_CJob * max(len(jobs), 1))()
        for k, j in enumerate(jobs):
            c = arr[k]
            c.session = j.session.handle if j.session is not None else None
            if isinstance(j.src, SemiPlanes) or isinstance(j.dst, SemiPlanes):
                c.sp_in, c.sp_out = (C.pointer(j.src) if j.src is not None else None), (C.pointer(j.dst) if j.dst is not None else None)
            else:
                c.in_, c.out = (C.pointer(j.src) if j.src is not None else None), (C.pointer(j.dst) if j.dst is not None else None)
            c.nframes, c.width, c.height, c.out_depth = j.nframes, j.width, j.height, j.out_depth
        self._chk(self.L.vfgs_b200_add_grain_jobs_device(arr, len(jobs), C.c_void_p(stream.cuda_stream)))

    def init_sessions(self, entries, stream=None):
        """entries: a list of ``(session, kind, raw)`` with kind ``"sei"`` or ``"afgs1"`` and raw the bytes of an fgs_sei /
        fgs_afgs1 struct. Re-programs every session from its metadata in one asynchronous device call on ``stream`` (a
        torch.cuda.Stream; default: torch's current stream), see vfgs_b200_session_init_metadata."""
        import torch
        if stream is None:
            stream = torch.cuda.current_stream()
        arr = (_CMetadata * max(len(entries), 1))()
        keep = []
        for k, (session, kind, raw) in enumerate(entries):
            if kind not in ("sei", "afgs1"):
                raise VfgsError(f"metadata kind {kind!r}: 'sei' or 'afgs1'")
            buf = (C.c_uint8 * len(raw)).from_buffer_copy(raw)
            keep.append(buf)
            arr[k].session = session.handle if session is not None else None
            setattr(arr[k], kind, C.cast(buf, C.c_void_p))
        self._chk(self.L.vfgs_b200_session_init_metadata(arr, len(entries), C.c_void_p(stream.cuda_stream)))


class Session:
    """One video stream's grain state (vfgs_b200_session): patterns, LUTs, scalars and LFSR registers, independent of
    the global state and of other sessions. ``close()`` (or leaving a ``with`` block) frees it once the kernels that
    read it are done."""

    def __init__(self, hw: VfgsHw, handle: int):
        self.hw, self.L, self.handle = hw, hw.L, handle
        sc = self.get_state()["scalars"]
        self.depth, self.csubx, self.csuby = 8 + int(sc[1]), int(sc[6]), int(sc[7])

    def close(self):
        if self.handle:
            self.L.vfgs_b200_session_destroy(C.c_void_p(self.handle))
            self.handle = None

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def get_lfsr(self):
        r = (C.c_uint32 * 4)()
        self.L.vfgs_b200_session_get_lfsr(C.c_void_p(self.handle), r)
        return [int(v) for v in r]

    def set_lfsr(self, regs):
        r = (C.c_uint32 * 4)(*[int(v) & 0xFFFFFFFF for v in regs])
        self.L.vfgs_b200_session_set_lfsr(C.c_void_p(self.handle), r)

    def skip_frames(self, n, width, height):
        self.hw._chk(self.L.vfgs_b200_session_skip_frames(C.c_void_p(self.handle), n, width, height))

    def set_seed(self, seed):
        """vfgs_set_seed on the session's registers."""
        self.hw._chk(self.L.vfgs_b200_session_set_seed(C.c_void_p(self.handle), seed & 0xFFFFFFFF))

    def init_sei(self, raw: bytes, stream=None):
        """This session's FGC SEI metadata (the bytes of an fgs_sei struct): VfgsHw.init_sessions with one entry."""
        self.hw.init_sessions([(self, "sei", raw)], stream)

    def init_afgs1(self, raw: bytes, stream=None):
        """This session's AFGS1 metadata (the bytes of an fgs_afgs1 struct): VfgsHw.init_sessions with one entry."""
        self.hw.init_sessions([(self, "afgs1", raw)], stream)

    def get_state(self) -> dict:
        n = self.L.vfgs_b200_session_get_state(C.c_void_p(self.handle), None, 0)
        buf = (C.c_uint8 * n)()
        self.L.vfgs_b200_session_get_state(C.c_void_p(self.handle), buf, n)
        return _state_dict(np.frombuffer(bytes(buf), dtype=np.uint8))

    def frame_bytes(self, width, height, depth):
        """Bytes of one packed planar frame with this session's chroma subsampling."""
        s = 2 if depth > 8 else 1
        return (width * height + 2 * (width // self.csubx) * (height // self.csuby)) * s


class Job:
    """One job of VfgsHw.add_grain_jobs_device: ``nframes`` frames of ``session`` from ``src`` to ``dst`` (a ``Planes``
    or a ``SemiPlanes`` pair). ``tensors`` keeps the buffers the planes point into alive."""

    def __init__(self, session, src, dst, nframes, width, height, out_depth=0, tensors=()):
        self.session, self.src, self.dst = session, src, dst
        self.nframes, self.width, self.height, self.out_depth = nframes, width, height, out_depth
        self.tensors = tensors

    @classmethod
    def packed(cls, session: Session, src, dst, nframes, width, height, out_depth=0) -> "Job":
        """Packed planar frames (the layout of add_grain_frames_device) in CUDA tensors, with the session's subsampling."""
        def planes(t, depth):
            s = 2 if depth > 8 else 1
            cw, ch = width // session.csubx, height // session.csuby
            b = t.data_ptr()
            return Planes(b, b + width * height * s, b + (width * height + cw * ch) * s, width * s, cw * s,
                          session.frame_bytes(width, height, depth))
        od = out_depth or session.depth
        return cls(session, planes(src, session.depth), planes(dst, od), nframes, width, height, out_depth, (src, dst))

    @classmethod
    def surfaces(cls, session: Session, src, dst, nframes, width, height, out_format=None) -> "Job":
        """Decoder-style surfaces (surface_planes): CUDA tensors of shape (n, height + ch, pitch)."""
        in_fmt = P010 if src.element_size() == 2 else NV12
        return cls(session, surface_planes(src, height, in_fmt), surface_planes(dst, height, out_format or in_fmt), nframes,
                   width, height, 0, (src, dst))
