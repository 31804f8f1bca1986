"""Host front end (include/vp8_parse.h): .webp bytes -> decoded frames, one image per host thread.

Counterpart of the reference's m01 + m02 + m05 call sequence in main.c:556-600
(webp_parse_simple_lossy -> vp8_parse_keyframe_header -> vp8_decode_decoded_frame).
"""
from __future__ import annotations

import ctypes as C
import os

import numpy as np

from .abi import DecodedFrame, KeyFrameHeader


class CompactFrame(C.Structure):
    """Vp8CompactFrame (include/vp8_parse.h)."""
    _fields_ = [("f", DecodedFrame), ("base", C.c_void_p), ("head_off", C.c_size_t), ("packed_off", C.c_size_t), ("bytes", C.c_size_t),
                ("n_blocks", C.c_uint32), ("width", C.c_uint32), ("height", C.c_uint32), ("owned", C.c_uint32)]

_L = None


def bind(L):
    global _L
    vp, sz = C.c_void_p, C.c_size_t
    L.vp8_parse_arena_bytes.argtypes = [C.c_uint32, C.c_uint32]
    L.vp8_parse_arena_bytes.restype = sz
    L.vp8_parse_webp_size.argtypes = [vp, sz, C.POINTER(C.c_uint32), C.POINTER(C.c_uint32)]
    L.vp8_parse_webp.argtypes = [vp, sz, vp, vp, vp, sz]
    L.vp8_parse_vp8.argtypes = [vp, sz, vp, vp, vp, sz]
    L.vp8_parse_free.argtypes = [vp]
    L.vp8_parse_free.restype = None
    L.vp8_parse_batch.argtypes = [vp, vp, C.c_int, C.c_int, vp, vp, vp, vp, vp]
    L.vp8_parse_compact_bytes.argtypes = [C.c_uint32, C.c_uint32]
    L.vp8_parse_compact_bytes.restype = sz
    L.vp8_parse_webp_compact.argtypes = [vp, sz, vp, vp, vp, sz]
    L.vp8_parse_compact_free.argtypes = [vp]
    L.vp8_parse_compact_free.restype = None
    L.vp8_parse_batch_compact.argtypes = [vp, vp, C.c_int, C.c_int, vp, vp, vp, sz, vp, vp]
    L.vp8_compact_rebase.argtypes = [vp, vp]
    L.vp8_compact_rebase.restype = None
    L.vp8_parse_webp_info.argtypes = [vp, sz, C.POINTER(C.c_uint32), C.POINTER(C.c_uint32), C.POINTER(C.c_int)]
    L.vp8_parse_alpha.argtypes = [vp, sz, vp, sz]
    _L = L


def _lib():
    if _L is None:
        from . import load_library
        load_library()
    return _L


class ParsedFrames:
    """n parsed frames: `.kfs[i]` / `.frames[i]` are the ctypes structs the GPU entry points take.
    The coefficient/mode arrays live either in calloc memory or in one pinned buffer (pinned=True)."""

    def __init__(self, n):
        self.n = n
        self.kfs = (KeyFrameHeader * n)()
        self.frames = (DecodedFrame * n)()
        self._pinned = None
        self._owned = True

    def free(self):
        if self._owned and self.frames is not None:
            L = _lib()
            for i in range(self.n):
                L.vp8_parse_free(C.addressof(self.frames[i]))
            self._owned = False
        if self._pinned is not None:
            self._pinned.close()
            self._pinned = None

    def __del__(self):
        try:
            self.free()
        except Exception:
            pass

    def kf_list(self):
        return [self.kfs[i] for i in range(self.n)]

    def frame_list(self):
        return [self.frames[i] for i in range(self.n)]

    def array(self, i, name):
        """numpy view of one per-frame array (for tests)."""
        f = self.frames[i]
        mb = f.mb_total
        count = {"segment_id": mb, "skip_coeff": mb, "has_coeff": mb, "ymode": mb, "uv_mode": mb, "bmode": mb * 16,
                 "coeff_y2": mb * 16, "coeff_y": mb * 256, "coeff_u": mb * 64, "coeff_v": mb * 64}[name]
        return np.ctypeslib.as_array(getattr(f, name), shape=(count,))


def webp_size(data: bytes):
    w, h = C.c_uint32(), C.c_uint32()
    buf = (C.c_uint8 * len(data)).from_buffer_copy(data)
    if _lib().vp8_parse_webp_size(buf, len(data), C.byref(w), C.byref(h)) != 0:
        e = C.get_errno()
        raise OSError(e, "not a simple lossy WebP key frame")
    return w.value, h.value


def webp_info(data: bytes):
    """(width, height, has_alpha) of a simple or extended (VP8X) lossy file (vp8_parse_webp_info)."""
    w, h, a = C.c_uint32(), C.c_uint32(), C.c_int()
    buf = (C.c_uint8 * len(data)).from_buffer_copy(data)
    if _lib().vp8_parse_webp_info(buf, len(data), C.byref(w), C.byref(h), C.byref(a)) != 0:
        e = C.get_errno()
        raise OSError(e, f"not a lossy WebP key frame: {os.strerror(e)}")
    return w.value, h.value, bool(a.value)


def alpha_plane(data: bytes):
    """The unfiltered alpha plane of a .webp file as an (h, w) uint8 array, decoded on the host (vp8_parse_alpha); None for a
    file without an ALPH chunk."""
    w, h, has_alpha = webp_info(data)
    if not has_alpha:
        return None
    out = np.empty((h, w), np.uint8)
    buf = (C.c_uint8 * len(data)).from_buffer_copy(data)
    if _lib().vp8_parse_alpha(buf, len(data), out.ctypes.data, out.nbytes) != 0:
        e = C.get_errno()
        raise OSError(e, f"alpha plane: {os.strerror(e)}")
    return out


def parse_batch(files, threads: int | None = None, pinned: bool = False) -> ParsedFrames:
    """Parse a list of .webp byte strings on `threads` host threads (default: all cores)."""
    L = _lib()
    n = len(files)
    assert n > 0
    threads = threads or os.cpu_count() or 1
    bufs = [(C.c_uint8 * len(d)).from_buffer_copy(d) for d in files]
    fp = (C.c_void_p * n)(*[C.addressof(b) for b in bufs])
    sizes = (C.c_size_t * n)(*[len(d) for d in files])
    out = ParsedFrames(n)
    status = (C.c_int * n)()
    arenas = arena_sizes = None
    if pinned:
        from . import PinnedBuffer
        need = []
        for d in files:
            w, h = webp_size(d)
            need.append(int(L.vp8_parse_arena_bytes(w, h)))
        offs = np.concatenate([[0], np.cumsum(need)])
        out._pinned = PinnedBuffer(int(offs[-1]))
        base = out._pinned.array.ctypes.data
        arenas = (C.c_void_p * n)(*[base + int(o) for o in offs[:-1]])
        arena_sizes = (C.c_size_t * n)(*need)
    failed = L.vp8_parse_batch(fp, sizes, n, threads, out.kfs, out.frames, arenas, arena_sizes, status)
    if failed:
        bad = [(i, status[i]) for i in range(n) if status[i]]
        out.free()
        raise OSError(bad[0][1], f"{failed} of {n} files failed to parse; first: file {bad[0][0]}: {os.strerror(bad[0][1])}")
    return out


def parse_webp(data: bytes) -> ParsedFrames:
    return parse_batch([data], threads=1)


class _HostBuffer:
    """Pageable stand-in for PinnedBuffer (256-byte aligned numpy memory)."""

    def __init__(self, nbytes):
        self._raw = np.zeros(nbytes + 256, np.uint8)
        off = (-self._raw.ctypes.data) % 256
        self.array = self._raw[off:off + nbytes]

    def close(self):
        self.array = self._raw = None


_PTR_FIELDS = ("segment_id", "skip_coeff", "has_coeff", "ymode", "uv_mode", "bmode", "coeff_y2", "coeff_y", "coeff_u", "coeff_v")
_ARENA_MAGIC = 0x564138415245414E  # stats_opaque[21] of frames whose arrays are one block ([22] base, [23] bytes): vp8_parse.cpp


def replicate_dense(pf: ParsedFrames, order, pinned: bool = True) -> ParsedFrames:
    """A batch of len(order) dense frames, frame k a private copy of pf.frames[order[k]] in ONE pinned buffer.
    For benchmarks: n structs pointing at the same arrays would let the host caches serve a 6.9 GB input."""
    n = len(order)
    out = ParsedFrames(n)
    out._owned = False
    sizes = []
    for i in range(pf.n):
        f = pf.frames[i]
        assert f.stats_opaque[21] == _ARENA_MAGIC, "frame was not parsed into an arena"
        sizes.append((int(f.stats_opaque[23]) + 255) // 256 * 256)
    total = sum(sizes[i] for i in order)
    if pinned:
        from . import PinnedBuffer
        out._pinned = PinnedBuffer(total)
    else:
        out._pinned = _HostBuffer(total)
    out.nbytes = total
    at = out._pinned.array.ctypes.data
    ptr_off = {name: getattr(DecodedFrame, name).offset for name in _PTR_FIELDS}
    for k, i in enumerate(order):
        src = pf.frames[i]
        base = int(src.stats_opaque[22])
        C.memmove(at, base, int(src.stats_opaque[23]))
        dst_addr = C.addressof(out.frames[k])
        C.memmove(dst_addr, C.addressof(src), C.sizeof(DecodedFrame))
        C.memmove(C.addressof(out.kfs[k]), C.addressof(pf.kfs[i]), C.sizeof(KeyFrameHeader))
        for name, off in ptr_off.items():
            slot = C.c_uint64.from_address(dst_addr + off)
            if slot.value:
                slot.value = slot.value - base + at
        out.frames[k].stats_opaque[22] = at
        out.frames[k].stats_opaque[24] = 0  # not owned by the frame
        at += sizes[i]
    return out


class CompactFrames:
    """n compact frames (vp8_parse_batch_compact): `.frames[i]` are the structs vp8_gpu_decode_compact takes. With
    pinned=True they sit back to back in one pinned buffer, so a chunk crosses the link as one transfer."""

    def __init__(self, n):
        self.n = n
        self.kfs = (KeyFrameHeader * n)()
        self.frames = (CompactFrame * n)()
        self._pinned = None
        self.used = 0

    def frame_list(self):
        return [self.frames[i] for i in range(self.n)]

    def head(self, i):
        """(mb_mask, mb_first, packed blocks as int16[n_blocks, 16]) numpy views of frame i (for tests)."""
        f = self.frames[i]
        mb = f.f.mb_total
        base = f.base + f.head_off
        mask = np.ctypeslib.as_array(C.cast(base, C.POINTER(C.c_uint32)), shape=(mb,))
        first = np.ctypeslib.as_array(C.cast(base + 4 * mb, C.POINTER(C.c_uint32)), shape=(mb,))
        blocks = np.ctypeslib.as_array(C.cast(f.base + f.packed_off, C.POINTER(C.c_int16)), shape=(max(f.n_blocks, 1), 16))[:f.n_blocks]
        return mask, first, blocks

    def free(self):
        if self.frames is not None and self._pinned is None:
            L = _lib()
            for i in range(self.n):
                L.vp8_parse_compact_free(C.addressof(self.frames[i]))
        self.frames = None
        if self._pinned is not None:
            self._pinned.close()
            self._pinned = None

    def __del__(self):
        try:
            self.free()
        except Exception:
            pass


def parse_batch_compact(files, threads: int | None = None, pinned: bool = False, contiguous: bool | None = None,
                        replicate: int = 1) -> CompactFrames:
    """Parse .webp byte strings straight into the compact wire format (vp8_parse_batch_compact).
    contiguous (default: same as pinned): the frames end up back to back in ONE buffer in index order - pinned memory
    if pinned, else pageable. replicate > 1 (contiguous only): the buffer holds `replicate` interleaved copies of the
    parsed frames, each with its own memory (benchmarks: a batch of n*replicate frames whose host bytes are all
    distinct, unlike n structs pointing at the same arrays)."""
    L = _lib()
    n = len(files)
    assert n > 0
    contiguous = pinned if contiguous is None else contiguous
    assert contiguous or (not pinned and replicate == 1)
    threads = threads or os.cpu_count() or 1
    bufs = [(C.c_uint8 * len(d)).from_buffer_copy(d) for d in files]
    fp = (C.c_void_p * n)(*[C.addressof(b) for b in bufs])
    sizes = (C.c_size_t * n)(*[len(d) for d in files])
    status = (C.c_int * n)()
    out = CompactFrames(n)

    def buffer(nbytes):
        if pinned:
            from . import PinnedBuffer
            return PinnedBuffer(nbytes)
        return _HostBuffer(nbytes)

    arena, arena_bytes = None, 0
    if contiguous:
        arena_bytes = sum((int(L.vp8_parse_compact_bytes(*webp_size(d))) + 255) // 256 * 256 for d in files)
        out._pinned = buffer(arena_bytes)
        arena = out._pinned.array.ctypes.data
    used = C.c_size_t(0)
    failed = L.vp8_parse_batch_compact(fp, sizes, n, threads, out.kfs, out.frames, arena, arena_bytes, C.byref(used), status)
    if failed:
        bad = [(i, status[i]) for i in range(n) if status[i]]
        out.free()
        raise OSError(bad[0][1], f"{failed} of {n} files failed to parse; first: file {bad[0][0]}: {os.strerror(bad[0][1])}")
    out.used = used.value
    if replicate > 1:
        lens = [(out.frames[i].bytes + 255) // 256 * 256 for i in range(n)]
        big = buffer(sum(lens) * replicate)
        rep = CompactFrames(n * replicate)
        at = 0
        for k in range(n * replicate):
            i = k % n
            src = out.frames[i]
            start = src.base + src.head_off
            C.memmove(big.array.ctypes.data + at, start, src.bytes)
            C.memmove(C.addressof(rep.frames[k]), C.addressof(src), C.sizeof(CompactFrame))
            C.memmove(C.addressof(rep.kfs[k]), C.addressof(out.kfs[i]), C.sizeof(KeyFrameHeader))
            L.vp8_compact_rebase(C.addressof(rep.frames[k]), big.array.ctypes.data + at)
            rep.frames[k].owned = 0
            at += lens[i]
        rep._pinned = big
        rep.used = at
        out.free()
        return rep
    return out
