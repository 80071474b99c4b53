"""Planar <-> semi-planar (NV12 / P010) conversion for the tests of vfgs_b200_add_grain_semiplanar_device, and a driver
for its host emulation (tests/emu/emu_semiplanar.cpp, emu_add_grain_semiplanar)."""
from __future__ import annotations

import ctypes as C
import os
import subprocess

import numpy as np

from oracle.pyoracle import RefState, _ptr, frame_samples
from tests.util import aligned_empty

INTERLEAVED = 128  # emu mask bit: the fast task code's interleaved U/V lane ran


def split_planar(frames: np.ndarray, n: int, w: int, h: int, fmt: str):
    """Packed planar frames -> (Y (n, h, w), U (n, ch, cw), V (n, ch, cw))."""
    ys, cs, cw, ch = frame_samples(w, h, fmt)
    f = frames.reshape(n, ys + 2 * cs)
    return (f[:, :ys].reshape(n, h, w), f[:, ys:ys + cs].reshape(n, ch, cw), f[:, ys + cs:].reshape(n, ch, cw))


def planar_to_semi(frames: np.ndarray, n: int, w: int, h: int, fmt: str, p010: bool, rng=None):
    """(Y (n, h, w), UV (n, ch, 2 cw)) with U and V interleaved; P010: samples << 6, plus random low bits from rng."""
    Y, U, V = split_planar(frames, n, w, h, fmt)
    UV = np.empty(U.shape[:2] + (2 * U.shape[2],), dtype=frames.dtype)
    UV[:, :, 0::2], UV[:, :, 1::2] = U, V
    Y = Y.copy()
    if p010:
        Y, UV = (Y.astype(np.uint16) << 6), (UV.astype(np.uint16) << 6)
        if rng is not None:
            Y |= rng.integers(0, 64, size=Y.shape, dtype=np.uint16)
            UV |= rng.integers(0, 64, size=UV.shape, dtype=np.uint16)
    return Y, UV


def semi_to_planar(Y: np.ndarray, UV: np.ndarray, p010: bool) -> np.ndarray:
    """Inverse of planar_to_semi: packed planar frames (P010: samples >> 6)."""
    n = Y.shape[0]
    if p010:
        Y, UV = Y >> 6, UV >> 6
    return np.concatenate([Y.reshape(n, -1), UV[:, :, 0::2].reshape(n, -1), UV[:, :, 1::2].reshape(n, -1)], axis=1).reshape(-1)


class Surface:
    """Host buffer of n semi-planar frames: per frame `h` Y rows at pitch_y bytes, then `ch` UV rows at pitch_uv bytes,
    frames frame_pad bytes apart beyond that; the buffer starts `offset` bytes after a 64-byte boundary."""

    def __init__(self, n, w, h, ch, sample, pitch_y=None, pitch_uv=None, offset=0, frame_pad=0):
        self.n, self.w, self.h, self.ch, self.sample = n, w, h, ch, sample
        self.pitch_y = pitch_y or w * sample
        self.pitch_uv = pitch_uv or w // 2 * 2 * sample  # 2 cw samples, cw = w / 2
        self.frame = h * self.pitch_y + ch * self.pitch_uv + frame_pad
        self.buf = aligned_empty(n * self.frame + 64, np.uint8, offset)
        self.base = self.buf.ctypes.data
        self.uv_off = h * self.pitch_y

    def _view(self, off, rows, pitch, cols):
        dt = np.uint16 if self.sample == 2 else np.uint8
        out = np.empty((self.n, rows, cols), dtype=dt)
        for f in range(self.n):
            for r in range(rows):
                a = f * self.frame + off + r * pitch
                out[f, r] = self.buf[a:a + cols * self.sample].view(dt)
        return out

    def _fill(self, arr, off, pitch):
        for f in range(arr.shape[0]):
            for r in range(arr.shape[1]):
                a = f * self.frame + off + r * pitch
                self.buf[a:a + arr.shape[2] * self.sample] = arr[f, r].view(np.uint8)

    def fill(self, Y, UV):
        self._fill(Y, 0, self.pitch_y)
        self._fill(UV, self.uv_off, self.pitch_uv)

    def planes(self):
        return self._view(0, self.h, self.pitch_y, self.w), self._view(self.uv_off, self.ch, self.pitch_uv, 2 * (self.w // 2))

    def args(self):
        """y, uv, stride_y, stride_uv, frame_stride"""
        return (C.c_void_p(self.base), C.c_void_p(self.base + self.uv_off), self.pitch_y, self.pitch_uv, self.frame)


def load_emu():
    """Host build of the semi-planar task code (tests/emu/emu_semiplanar.cpp, test tool only), rebuilt when a source is
    newer than the library."""
    here = os.path.join(os.path.dirname(os.path.abspath(__file__)), "emu")
    so, src = os.path.join(here, "libemu_semiplanar.so"), os.path.join(here, "emu_semiplanar.cpp")
    csrc = os.path.join(os.path.dirname(here), "..", "versatilefilmgrain_b200", "csrc")
    deps = [src] + [os.path.join(csrc, n) for n in os.listdir(csrc) if n.endswith(".h")]
    if not os.path.exists(so) or any(os.path.getmtime(d) > os.path.getmtime(so) for d in deps):
        # -Bsymbolic: the shared headers' inline functions bind to this library's copies, not to another loaded library's
        subprocess.run(["g++", "-O2", "-std=c++17", "-fPIC", "-shared", "-Wl,-Bsymbolic", "-Wno-unknown-pragmas", "-o", so, src], check=True)
    L = C.CDLL(so)
    assert L.emus_state_size() == C.sizeof(RefState)
    return bind_emu(L)


def bind_emu(L):
    L.emu_add_grain_semiplanar.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_longlong, C.c_longlong, C.c_longlong,
                                           C.c_void_p, C.c_void_p, C.c_longlong, C.c_longlong, C.c_longlong] + [C.c_int] * 6
    return L


def run_emu_semi(emu, o, src: Surface, dst: Surface, n, w, h, p010_out, first=0, mode=0):
    """Emulated semi-planar call with the state of oracle `o` (whose registers it does not advance); returns the mask."""
    st = RefState()
    o.L.oracle_get_state(o.h, C.byref(st))
    return emu.emu_add_grain_semiplanar(C.byref(st), *src.args(), *dst.args(), n, w, h, int(p010_out), first, mode)
