"""Text inputs of ``prepare-orfs``, ``orfs-seq``, ``count-orfs`` and ``count-orfs-codon``: plain text, or BGZF
inflated on the GPU.

``open_texts(paths, command)`` looks at the first bytes of every input (DESIGN.md section 12):

    plain text      the path itself: the native loader reads the file, as it always has
    BGZF            a ``NativeText`` from ``Engine.inflate_bgzf`` (bgzf_inflate_kernel), which a ``*_load_text`` loader
                    takes over without a copy
    other gzip      refused: one serial DEFLATE stream cannot be split across warps

The loaders accept either and name ``NativeText.path``, the path the user gave, in their messages.
"""
from __future__ import annotations

import ctypes as C
import struct
import time

import numpy as np

from . import _lib

GZIP_MAGIC = b"\x1f\x8b"


class NativeText:
    """An owned ``rt_text`` buffer holding the text of ``path``.  A ``*_load_text`` loader takes it over (``take``);
    until then it is freed with this object."""

    def __init__(self, handle: C.c_void_p, path: str):
        self._lib = _lib.load()
        self.handle = handle
        self.path = str(path)

    @classmethod
    def alloc(cls, n: int, path: str) -> "NativeText":
        """An uninitialised text of ``n`` bytes, to be filled through ``view()``."""
        lib = _lib.load()
        h = C.c_void_p()
        if lib.rt_text_alloc(int(n), C.byref(h)) != 0:
            raise MemoryError(f"cannot allocate {n} bytes for the text of {path}")
        return cls(h, path)

    def __len__(self) -> int:
        return int(self._lib.rt_text_len(self.handle)) if self.handle else 0

    def view(self) -> np.ndarray:
        """The text as a writable uint8 array over the native buffer (valid until the text is taken or freed)."""
        n = len(self)
        if not n:
            return np.zeros(0, np.uint8)
        return np.ctypeslib.as_array((C.c_uint8 * n).from_address(self._lib.rt_text_data(self.handle)))

    def take(self) -> C.c_void_p:
        """The handle, for a loader that takes the buffer over; this object no longer owns it."""
        if not self.handle:
            raise ValueError(f"the text of {self.path} has already been handed to a loader")
        h, self.handle = self.handle, None
        return h

    def __del__(self):
        try:
            if getattr(self, "handle", None):
                self._lib.rt_text_free(self.handle)
                self.handle = None
        except Exception:
            pass


def is_bgzf_header(head: bytes) -> bool:
    """The first member header of a BGZF file (SAM spec 4.1): gzip magic, CM 8, FEXTRA and a 'BC' subfield of length 2.
    This mirrors the header checks of ``parse_block`` (csrc/rt_bgzf.h), which ``rt_bgzf_inflate`` then applies to every
    member.  What only the whole member can show (its BSIZE within the file, ISIZE at most 64 KiB) is left to that walk,
    so a file whose first member has a BGZF header but a bad size is reported as BGZF block 0 (rule 4), not as plain
    gzip."""
    if len(head) < 12 or head[:3] != b"\x1f\x8b\x08" or not head[3] & 4:
        return False
    xlen = struct.unpack_from("<H", head, 10)[0]
    extra = head[12:12 + xlen]
    x = 0
    while x + 4 <= len(extra):
        slen = struct.unpack_from("<H", extra, x + 2)[0]
        if extra[x:x + 2] == b"BC" and slen == 2:
            return True
        x += 4 + slen
    return False


def sniff(path: str) -> str:
    """"plain", "bgzf" or "gzip" from the first bytes of the file."""
    with open(path, "rb") as fh:
        head = fh.read(12)
        if head[:2] != GZIP_MAGIC:
            return "plain"
        if len(head) == 12:
            head += fh.read(struct.unpack_from("<H", head, 10)[0])
    return "bgzf" if is_bgzf_header(head) else "gzip"


def open_texts(paths, command: str) -> list:
    """Per input, the path for plain text or a ``NativeText`` for BGZF.  Every input is sniffed, and the first plain
    gzip one refused with a ValueError, before any is inflated."""
    kinds = [sniff(p) for p in paths]
    for path, kind in zip(paths, kinds):
        if kind == "gzip":
            raise ValueError(f"{path} is gzip-compressed; {command} reads plain text only")
    if "bgzf" not in kinds:
        return list(paths)
    from .detect_orfs import get_engine

    return [get_engine().inflate_bgzf(p) if kind == "bgzf" else p for p, kind in zip(paths, kinds)]


def open_text(path: str, command: str):
    """``open_texts`` of one input."""
    return open_texts([path], command)[0]


class StageClock:
    """Stage times of one command in milliseconds, written into ``times`` (a new dict when None): ``lap(name)`` records
    the host time since the previous lap, ``device(names, ms)`` the device stage times a native call reported, each as
    ``"device:" + name``."""

    def __init__(self, times: dict | None = None):
        self.times = {} if times is None else times
        self._clock = time.perf_counter()

    def lap(self, name: str) -> None:
        now = time.perf_counter()
        self.times[name] = (now - self._clock) * 1e3
        self._clock = now

    def device(self, names, ms) -> None:
        for name, v in zip(names, ms.tolist()):
            self.times["device:" + name] = v
