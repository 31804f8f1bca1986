"""webp-decoder_b200: B200-native pixel path of a VP8 key-frame (lossy WebP) decoder.

Python face of libvp8gpu.so (include/vp8_gpu.h). It mirrors the reference decoder's module interface for
this path - same names, argument meaning and error behaviour:

    vp8_reconstruct_keyframe_yuv(kf, decoded)            reference src/m06_recon/vp8_recon.h:25
    vp8_reconstruct_keyframe_yuv_filtered(kf, decoded)   reference src/m06_recon/vp8_recon.h:28
    vp8_loopfilter_apply_keyframe(y, u, v, decoded)      reference src/m07_loopfilter/vp8_loopfilter.h:14
    yuv420_write_ppm(i420, w, h)                         reference src/m08_yuv2rgb_ppm/yuv2rgb_ppm.h:10
    yuv420_write_png(i420, w, h)                         reference src/m09_png/yuv2rgb_png.h:10

plus the batch interface (`Context`, `Batch`) that keeps many frames resident on the device.

Everything here is plumbing around the C-ABI; all pixels come from the CUDA kernels. If the shared library is
missing or no CUDA device is usable, calls raise - there is no CPU fallback.
"""
from __future__ import annotations

import ctypes as C
import errno as _errno
import os
from pathlib import Path

import numpy as np

from .abi import DecodedFrame, KeyFrameHeader, Yuv420Image  # noqa: F401

_HERE = Path(__file__).resolve().parent
LIB_PATH = _HERE / "libvp8gpu.so"

TIGHT, PADDED = 0, 1
OUT_I420, OUT_PPM, OUT_PNG = 0, 1, 2  # what the pipelined calls' `ppm` argument selects ("png" / OUT_PNG: -png files)


def _fmt(ppm) -> int:
    if isinstance(ppm, str):
        return {"i420": OUT_I420, "ppm": OUT_PPM, "png": OUT_PNG}[ppm]
    return OUT_PNG if ppm is OUT_PNG or (not isinstance(ppm, bool) and ppm == OUT_PNG) else int(bool(ppm))

EXPORTS = [
    # reference module interfaces
    "yuv420_alloc", "yuv420_free", "vp8_reconstruct_keyframe_yuv", "vp8_reconstruct_keyframe_yuv_filtered",
    "vp8_loopfilter_apply_keyframe", "yuv420_write_ppm_fd", "yuv420_write_png_fd",
    # batch interface
    "vp8_gpu_init", "vp8_gpu_destroy", "vp8_gpu_sync", "vp8_gpu_trim", "vp8_gpu_last_error", "vp8_gpu_set_tuning",
    "vp8_gpu_host_alloc", "vp8_gpu_host_free", "vp8_gpu_upload", "vp8_gpu_batch_free", "vp8_gpu_recon",
    "vp8_gpu_filter", "vp8_gpu_rgb", "vp8_gpu_run", "vp8_gpu_i420_bytes", "vp8_gpu_ppm_bytes",
    "vp8_gpu_download_i420", "vp8_gpu_download_ppm", "vp8_gpu_download_images", "vp8_gpu_download_padded",
    "vp8_gpu_batch_size", "vp8_gpu_launch_count", "vp8_gpu_h2d_bytes", "vp8_gpu_d2h_bytes",
    "vp8_gpu_last_launch_config", "vp8_gpu_frame_params", "vp8_gpu_kernel_time", "vp8_gpu_rgb_time",
    "vp8_gpu_decode_i420", "vp8_gpu_decode_ppm", "vp8_gpu_decode_bytes", "vp8_gpu_set_kernel",
    "vp8_gpu_png_bound", "vp8_gpu_png_frame", "vp8_gpu_set_transport",
    "vp8_gpu_png", "vp8_gpu_png_bytes", "vp8_gpu_download_png", "vp8_gpu_decode_png", "vp8_gpu_png_time", "vp8_gpu_set_png_deflate",
    "vp8_gpu_set_cluster", "vp8_gpu_set_cluster_split", "vp8_gpu_last_split", "vp8_gpu_last_cluster", "vp8_gpu_last_groups", "vp8_gpu_last_segments",
    "vp8_gpu_decode_compact", "vp8_gpu_decode_webp", "vp8_gpu_decode_webp_bytes", "vp8_gpu_last_call_profile", "vp8_gpu_bind_host", "vp8_gpu_last_transport", "vp8_gpu_last_dense_frames",
    # encoder in-loop reconstruction (include/vp8_enc.h)
    "enc_vp8_encode_dc_pred_inloop", "enc_vp8_encode_i16x16_uv_sad_inloop", "enc_vp8_encode_i16x16_sad_inloop",
    "enc_vp8_encode_bpred_uv_sad_inloop", "vp8_gpu_enc_i16_inloop", "vp8_gpu_enc_bpred_inloop", "vp8_gpu_enc_mb_total",
    "vp8_gpu_enc_last_kernel_ms",
]

_lib = None


class Vp8GpuError(OSError):
    pass


def load_library() -> C.CDLL:
    """Loads libvp8gpu.so (built in-tree by build.py / __graft_entry__.build()). Fails loudly when absent."""
    global _lib
    if _lib is not None:
        return _lib
    path = Path(os.environ.get("VP8_GPU_LIB", LIB_PATH))  # VP8_GPU_LIB: development override (kernel A/B builds)
    if not path.exists():
        raise Vp8GpuError(_errno.ENOENT, f"{path} is missing: run `python __graft_entry__.py build` "
                                         "(the CUDA library is the only implementation; there is no CPU fallback)")
    L = C.CDLL(str(path), use_errno=True)
    vp, sz, pp = C.c_void_p, C.c_size_t, C.POINTER(C.c_void_p)
    L.vp8_gpu_init.argtypes = [C.c_int, vp, pp]
    L.vp8_gpu_destroy.argtypes = [vp]
    L.vp8_gpu_destroy.restype = None
    L.vp8_gpu_sync.argtypes = [vp]
    L.vp8_gpu_trim.argtypes = [vp]
    L.vp8_gpu_last_error.restype = C.c_char_p
    L.vp8_gpu_set_tuning.argtypes = [vp, C.c_int, C.c_int]
    L.vp8_gpu_set_kernel.argtypes = [vp, C.c_int]
    L.vp8_gpu_set_transport.argtypes = [vp, C.c_int, C.c_int]
    L.vp8_gpu_set_cluster.argtypes = [vp, C.c_int]
    L.vp8_gpu_set_cluster_split.argtypes = [vp, C.c_int]
    L.vp8_gpu_last_split.argtypes = [vp]
    L.vp8_gpu_last_cluster.argtypes = [vp]
    L.vp8_gpu_last_groups.argtypes = [vp]
    L.vp8_gpu_last_segments.argtypes = [vp]
    L.vp8_gpu_host_alloc.argtypes = [sz]
    L.vp8_gpu_host_alloc.restype = vp
    L.vp8_gpu_host_free.argtypes = [vp]
    L.vp8_gpu_host_free.restype = None
    L.vp8_gpu_upload.argtypes = [vp, pp, pp, C.c_int, pp]
    L.vp8_gpu_recon.argtypes = [vp, pp, pp, C.c_int, pp]
    L.vp8_gpu_batch_free.argtypes = [vp, vp]
    L.vp8_gpu_batch_free.restype = None
    L.vp8_gpu_filter.argtypes = [vp, vp]
    L.vp8_gpu_rgb.argtypes = [vp, vp]
    L.vp8_gpu_run.argtypes = [vp, vp, C.c_int, C.c_int]
    L.vp8_gpu_i420_bytes.argtypes = [vp]
    L.vp8_gpu_i420_bytes.restype = sz
    L.vp8_gpu_ppm_bytes.argtypes = [vp]
    L.vp8_gpu_ppm_bytes.restype = sz
    L.vp8_gpu_download_i420.argtypes = [vp, vp, vp, sz, vp, vp]
    L.vp8_gpu_download_ppm.argtypes = [vp, vp, vp, sz, vp, vp]
    L.vp8_gpu_png.argtypes = [vp, vp]
    L.vp8_gpu_png_bytes.argtypes = [vp]
    L.vp8_gpu_png_bytes.restype = sz
    L.vp8_gpu_download_png.argtypes = [vp, vp, vp, sz, vp, vp]
    L.vp8_gpu_decode_png.argtypes = [vp, pp, pp, C.c_int, vp, sz, vp, vp, C.c_int]
    L.vp8_gpu_png_time.argtypes = [vp, C.POINTER(C.c_double), C.POINTER(C.c_int)]
    L.vp8_gpu_set_png_deflate.argtypes = [vp, C.c_int]
    L.vp8_gpu_download_images.argtypes = [vp, vp, vp]
    L.vp8_gpu_download_padded.argtypes = [vp, vp, C.c_int, vp, vp, vp]
    L.vp8_gpu_batch_size.argtypes = [vp]
    for fn in ("vp8_gpu_launch_count", "vp8_gpu_h2d_bytes", "vp8_gpu_d2h_bytes"):
        getattr(L, fn).argtypes = [vp]
        getattr(L, fn).restype = C.c_uint64
    L.vp8_gpu_last_launch_config.argtypes = [vp, C.POINTER(C.c_int), C.POINTER(C.c_int), C.POINTER(C.c_int)]
    L.vp8_gpu_kernel_time.argtypes = [vp, C.POINTER(C.c_double), C.POINTER(C.c_int)]
    L.vp8_gpu_rgb_time.argtypes = [vp, C.POINTER(C.c_double), C.POINTER(C.c_int)]
    L.vp8_gpu_frame_params.argtypes = [vp, vp, vp]
    L.vp8_gpu_frame_params.restype = None
    L.vp8_gpu_decode_i420.argtypes = [vp, pp, pp, C.c_int, C.c_int, vp, sz, vp, vp, C.c_int]
    L.vp8_gpu_decode_ppm.argtypes = [vp, pp, pp, C.c_int, vp, sz, vp, vp, C.c_int]
    L.vp8_gpu_decode_bytes.argtypes = [pp, C.c_int, C.c_int]
    L.vp8_gpu_decode_bytes.restype = sz
    L.vp8_gpu_decode_compact.argtypes = [vp, pp, C.c_int, C.c_int, C.c_int, vp, sz, vp, vp, C.c_int]
    L.vp8_gpu_decode_webp.argtypes = [vp, pp, vp, C.c_int, C.c_int, C.c_int, vp, sz, vp, vp, C.c_int]
    L.vp8_gpu_decode_webp_bytes.argtypes = [pp, vp, C.c_int, C.c_int]
    L.vp8_gpu_decode_webp_bytes.restype = sz
    L.vp8_gpu_last_call_profile.argtypes = [vp, C.POINTER(C.c_double), C.POINTER(C.c_double), C.POINTER(C.c_double)]
    L.vp8_gpu_bind_host.argtypes = [vp, C.c_int, C.c_int]
    L.vp8_gpu_last_transport.argtypes = [vp, C.POINTER(C.c_int), C.POINTER(C.c_int)]
    L.vp8_gpu_last_dense_frames.argtypes = [vp]
    L.yuv420_alloc.argtypes = [vp, C.c_uint32, C.c_uint32]
    L.yuv420_free.argtypes = [vp]
    L.yuv420_free.restype = None
    L.vp8_reconstruct_keyframe_yuv.argtypes = [vp, vp, vp]
    L.vp8_reconstruct_keyframe_yuv_filtered.argtypes = [vp, vp, vp]
    L.vp8_loopfilter_apply_keyframe.argtypes = [vp, vp]
    L.yuv420_write_ppm_fd.argtypes = [C.c_int, vp]
    L.yuv420_write_png_fd.argtypes = [C.c_int, vp]
    if hasattr(L, "vp8_parse_webp"):
        from . import parse as _parse
        _parse.bind(L)
    _lib = L
    return L


def _check(rc: int, what: str):
    if rc != 0:
        e = C.get_errno()
        msg = load_library().vp8_gpu_last_error().decode(errors="replace")
        raise Vp8GpuError(e, f"{what}: {os.strerror(e)} ({msg})")


def _addr(obj) -> int:
    return C.addressof(obj)


def frame_params(decoded):
    """(dq[4][6], lf[4][2][4]) exactly as the library derives them for the kernels."""
    L = load_library()
    dq = np.zeros((4, 6), np.int16)
    lf = np.zeros((4, 2, 4), np.uint8)
    L.vp8_gpu_frame_params(_addr(decoded), dq.ctypes.data, lf.ctypes.data)
    return dq, lf


class PinnedBuffer:
    """Page-locked host memory from the library, exposed as a numpy uint8 array."""

    def __init__(self, nbytes: int):
        L = load_library()
        self._p = L.vp8_gpu_host_alloc(nbytes)
        if not self._p:
            raise Vp8GpuError(_errno.ENOMEM, "vp8_gpu_host_alloc failed")
        self.nbytes = nbytes
        self.array = np.ctypeslib.as_array(C.cast(self._p, C.POINTER(C.c_uint8)), shape=(max(nbytes, 1),))[:nbytes]

    def close(self):
        if self._p:
            self.array = None
            load_library().vp8_gpu_host_free(self._p)
            self._p = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class WebpFiles:
    """n .webp byte strings laid out for the C-ABI (pointer and size arrays); keeps the bytes alive."""

    def __init__(self, datas):
        self.n = len(datas)
        self._bufs = [(C.c_uint8 * len(d)).from_buffer_copy(d) for d in datas]
        self.ptrs = (C.c_void_p * self.n)(*[C.addressof(b) for b in self._bufs])
        self.sizes = (C.c_size_t * self.n)(*[len(d) for d in datas])


class Batch:
    """n decoded frames resident on one GPU."""

    def __init__(self, ctx: "Context", handle: int, sizes):
        self.ctx, self._h, self.sizes = ctx, handle, list(sizes)

    @property
    def n(self):
        return len(self.sizes)

    def free(self):
        if self._h:
            self.ctx._L.vp8_gpu_batch_free(self.ctx._h, self._h)
            self._h = None

    def __del__(self):
        try:
            self.free()
        except Exception:
            pass


class Context:
    """One GPU, one stream. `stream` is a raw cudaStream_t (int), e.g. torch.cuda.current_stream().cuda_stream."""

    def __init__(self, device: int = 0, stream: int | None = None):
        self._L = load_library()
        h = C.c_void_p()
        _check(self._L.vp8_gpu_init(device, C.c_void_p(stream or 0), C.byref(h)), "vp8_gpu_init")
        self._h = h.value
        self.device = device

    def close(self):
        if self._h:
            self._L.vp8_gpu_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def set_tuning(self, warps_per_image: int = 0, images_per_sm: int = 0):
        _check(self._L.vp8_gpu_set_tuning(self._h, warps_per_image, images_per_sm), "vp8_gpu_set_tuning")

    def set_kernel(self, version: int):
        """1 = warp per macroblock, 2 = half-warp per macroblock (two rows per warp)."""
        _check(self._L.vp8_gpu_set_kernel(self._h, version), "vp8_gpu_set_kernel")

    def set_cluster(self, ctas_per_image: int = 0, split: bool | None = None):
        """CTAs per image in cluster mode: 0 automatic, 1 never, 2/4/8 upper bound. split: clusters of 4 / 8 CTAs in the fused
        mode run vp8_mb_split (reconstruction warp + filter warp per row pair; the default) or not."""
        _check(self._L.vp8_gpu_set_cluster(self._h, ctas_per_image), "vp8_gpu_set_cluster")
        if split is not None:
            _check(self._L.vp8_gpu_set_cluster_split(self._h, int(bool(split))), "vp8_gpu_set_cluster_split")

    def set_transport(self, compact=True, host_threads: int = 0):
        """compact: True / False, or "auto" (chosen chunk by chunk, the library's default)."""
        mode = 2 if compact == "auto" else int(bool(compact))
        _check(self._L.vp8_gpu_set_transport(self._h, mode, host_threads), "vp8_gpu_set_transport")

    def set_png_deflate(self, on: bool):
        """Compressed -png files from every -png call of this context (per-row PNG filters, run-length fixed-Huffman
        deflate, all on the device; never longer than the stored files) - or, off (the default), the reference's bytes.
        The files then lie back to back: read offsets / sizes."""
        _check(self._L.vp8_gpu_set_png_deflate(self._h, int(bool(on))), "vp8_gpu_set_png_deflate")

    def last_dense_frames(self):
        """Frames of the last pipelined call that crossed dense inside compact chunks (vp8_gpu_last_dense_frames)."""
        return int(self._L.vp8_gpu_last_dense_frames(self._h))

    def last_transport(self):
        d, c = C.c_int(), C.c_int()
        _check(self._L.vp8_gpu_last_transport(self._h, C.byref(d), C.byref(c)), "vp8_gpu_last_transport")
        return {"dense_chunks": d.value, "compact_chunks": c.value}

    def sync(self):
        _check(self._L.vp8_gpu_sync(self._h), "vp8_gpu_sync")

    def trim(self):
        """Returns the context's cached device blocks to the driver."""
        _check(self._L.vp8_gpu_trim(self._h), "vp8_gpu_trim")

    # ---- staging -----------------------------------------------------------------------------------------
    def _ptr_arrays(self, kfs, frames):
        n = len(frames)
        assert n == len(kfs) and n > 0
        kp = (C.c_void_p * n)(*[_addr(k) for k in kfs])
        fp = (C.c_void_p * n)(*[_addr(f) for f in frames])
        return n, kp, fp

    def upload(self, kfs, frames) -> Batch:
        """Host -> device staging of the frames' arrays (vp8_gpu_upload)."""
        n, kp, fp = self._ptr_arrays(kfs, frames)
        h = C.c_void_p()
        _check(self._L.vp8_gpu_upload(self._h, kp, fp, n, C.byref(h)), "vp8_gpu_upload")
        return Batch(self, h.value, [(k.width, k.height) for k in kfs])

    def recon(self, kfs, frames) -> Batch:
        """vp8_gpu_recon: staging + m06 into macroblock-aligned planes."""
        n, kp, fp = self._ptr_arrays(kfs, frames)
        h = C.c_void_p()
        _check(self._L.vp8_gpu_recon(self._h, kp, fp, n, C.byref(h)), "vp8_gpu_recon")
        return Batch(self, h.value, [(k.width, k.height) for k in kfs])

    # ---- kernels -----------------------------------------------------------------------------------------
    def run(self, batch: Batch, filtered: bool, layout: int = TIGHT):
        _check(self._L.vp8_gpu_run(self._h, batch._h, int(bool(filtered)), layout), "vp8_gpu_run")

    def filter(self, batch: Batch):
        _check(self._L.vp8_gpu_filter(self._h, batch._h), "vp8_gpu_filter")

    def rgb(self, batch: Batch):
        _check(self._L.vp8_gpu_rgb(self._h, batch._h), "vp8_gpu_rgb")

    def png(self, batch: Batch):
        """m09 on the device (after rgb): the -png file of every image, framed and checksummed in HBM."""
        _check(self._L.vp8_gpu_png(self._h, batch._h), "vp8_gpu_png")

    # ---- results -----------------------------------------------------------------------------------------
    def _download(self, fn, total_fn, batch: Batch, out: np.ndarray | None):
        total = total_fn(batch._h)
        if out is None:
            out = np.empty(total, np.uint8)
        assert out.dtype == np.uint8 and out.flags.c_contiguous and out.nbytes >= total
        offs = np.zeros(batch.n, np.uint64)
        sizes = np.zeros(batch.n, np.uint64)
        _check(fn(self._h, batch._h, out.ctypes.data, out.nbytes, offs.ctypes.data, sizes.ctypes.data), fn.__name__)
        return out, offs, sizes

    def download_i420(self, batch: Batch, out: np.ndarray | None = None):
        """Returns (buffer, offsets, sizes): frame i's -yuv/-yuvf bytes are buffer[offsets[i]:offsets[i]+sizes[i]]."""
        return self._download(self._L.vp8_gpu_download_i420, self._L.vp8_gpu_i420_bytes, batch, out)

    def download_ppm(self, batch: Batch, out: np.ndarray | None = None):
        """Same for the -ppm bytes (header + RGB)."""
        return self._download(self._L.vp8_gpu_download_ppm, self._L.vp8_gpu_ppm_bytes, batch, out)

    def download_png(self, batch: Batch, out: np.ndarray | None = None):
        """Same for the -png files."""
        return self._download(self._L.vp8_gpu_download_png, self._L.vp8_gpu_png_bytes, batch, out)

    def download_padded(self, batch: Batch, i: int):
        w, h = batch.sizes[i]
        pw, ph = (w + 15) // 16 * 16, (h + 15) // 16 * 16
        y, u, v = np.empty((ph, pw), np.uint8), np.empty((ph // 2, pw // 2), np.uint8), np.empty((ph // 2, pw // 2), np.uint8)
        _check(self._L.vp8_gpu_download_padded(self._h, batch._h, i, y.ctypes.data, u.ctypes.data, v.ctypes.data),
               "vp8_gpu_download_padded")
        return y, u, v

    # ---- whole path, pipelined ---------------------------------------------------------------------------
    def decode_bytes(self, kfs, ppm: bool = False) -> int:
        n = len(kfs)
        kp = (C.c_void_p * n)(*[_addr(k) for k in kfs])
        return int(self._L.vp8_gpu_decode_bytes(kp, n, _fmt(ppm)))

    def decode_into(self, kfs, frames, out: np.ndarray, filtered: bool = True, ppm: bool = False, chunk: int = 0):
        """vp8_gpu_decode_i420 / vp8_gpu_decode_ppm: upload, kernels and download overlapped chunk by chunk.
        `out` is a uint8 buffer (ideally a PinnedBuffer's array); returns (offsets, sizes)."""
        n, kp, fp = self._ptr_arrays(kfs, frames)
        assert out.dtype == np.uint8 and out.flags.c_contiguous
        offs, sizes = np.zeros(n, np.uint64), np.zeros(n, np.uint64)
        if _fmt(ppm) == OUT_PNG:
            rc = self._L.vp8_gpu_decode_png(self._h, kp, fp, n, out.ctypes.data, out.nbytes, offs.ctypes.data, sizes.ctypes.data, chunk)
        elif ppm:
            rc = self._L.vp8_gpu_decode_ppm(self._h, kp, fp, n, out.ctypes.data, out.nbytes, offs.ctypes.data, sizes.ctypes.data, chunk)
        else:
            rc = self._L.vp8_gpu_decode_i420(self._h, kp, fp, n, int(bool(filtered)), out.ctypes.data, out.nbytes,
                                             offs.ctypes.data, sizes.ctypes.data, chunk)
        _check(rc, "vp8_gpu_decode")
        return offs, sizes

    def decode_compact_into(self, frames, out: np.ndarray, filtered: bool = True, ppm: bool = False, chunk: int = 0):
        """vp8_gpu_decode_compact: frames = list of parse.CompactFrame structs (vp8_parse_*_compact output)."""
        n = len(frames)
        fp = (C.c_void_p * n)(*[_addr(f) for f in frames])
        offs, sizes = np.zeros(n, np.uint64), np.zeros(n, np.uint64)
        _check(self._L.vp8_gpu_decode_compact(self._h, fp, n, int(bool(filtered)), _fmt(ppm), out.ctypes.data, out.nbytes,
                                              offs.ctypes.data, sizes.ctypes.data, chunk), "vp8_gpu_decode_compact")
        return offs, sizes

    def decode_webp_into(self, files: "WebpFiles", out: np.ndarray, filtered: bool = True, ppm: bool = False, chunk: int = 0):
        """vp8_gpu_decode_webp: .webp bytes in (a WebpFiles pack), -yuv/-yuvf or -ppm bytes out; host threads parse
        chunk k while the GPU works on the chunks before it."""
        offs, sizes = np.zeros(files.n, np.uint64), np.zeros(files.n, np.uint64)
        _check(self._L.vp8_gpu_decode_webp(self._h, files.ptrs, files.sizes, files.n, int(bool(filtered)), _fmt(ppm), out.ctypes.data,
                                           out.nbytes, offs.ctypes.data, sizes.ctypes.data, chunk), "vp8_gpu_decode_webp")
        return offs, sizes

    def decode_webp_bytes(self, files: "WebpFiles", ppm: bool = False) -> int:
        return int(self._L.vp8_gpu_decode_webp_bytes(files.ptrs, files.sizes, files.n, _fmt(ppm)))

    def last_call_profile(self):
        t, h, w = C.c_double(), C.c_double(), C.c_double()
        _check(self._L.vp8_gpu_last_call_profile(self._h, C.byref(t), C.byref(h), C.byref(w)), "vp8_gpu_last_call_profile")
        return {"total_ms": t.value, "host_work_ms": h.value, "wait_ms": w.value}

    def bind_host(self, index: int = 0, share: int = 1) -> int:
        """Bind this thread (and the context's future worker threads) to the CPUs local to the GPU."""
        return int(self._L.vp8_gpu_bind_host(self._h, index, share))

    # ---- convenience -------------------------------------------------------------------------------------
    def decode_i420(self, kfs, frames, filtered: bool = True):
        """List of tight I420 byte arrays, one per frame (what `decoder -yuv` / `-yuvf` writes)."""
        b = self.upload(kfs, frames)
        try:
            self.run(b, filtered, TIGHT)
            buf, offs, sizes = self.download_i420(b)
            return [buf[int(o):int(o) + int(s)].copy() for o, s in zip(offs, sizes)]
        finally:
            b.free()

    def decode_ppm(self, kfs, frames):
        """List of PPM byte strings, one per frame (what `decoder -ppm` writes)."""
        b = self.upload(kfs, frames)
        try:
            self.run(b, True, TIGHT)
            self.rgb(b)
            buf, offs, sizes = self.download_ppm(b)
            return [buf[int(o):int(o) + int(s)].tobytes() for o, s in zip(offs, sizes)]
        finally:
            b.free()

    def decode_png(self, kfs, frames):
        """List of PNG byte strings, one per frame (what `decoder -png` writes), framed on the device."""
        b = self.upload(kfs, frames)
        try:
            self.run(b, True, TIGHT)
            self.rgb(b)
            self.png(b)
            buf, offs, sizes = self.download_png(b)
            return [buf[int(o):int(o) + int(s)].tobytes() for o, s in zip(offs, sizes)]
        finally:
            b.free()

    # ---- counters ----------------------------------------------------------------------------------------
    @property
    def launches(self) -> int:
        return int(self._L.vp8_gpu_launch_count(self._h))

    @property
    def h2d_bytes(self) -> int:
        return int(self._L.vp8_gpu_h2d_bytes(self._h))

    @property
    def d2h_bytes(self) -> int:
        return int(self._L.vp8_gpu_d2h_bytes(self._h))

    def kernel_time(self):
        """(total_ms, launches) of the wavefront launches since the previous call, timed with CUDA events."""
        ms, n = C.c_double(), C.c_int()
        _check(self._L.vp8_gpu_kernel_time(self._h, C.byref(ms), C.byref(n)), "vp8_gpu_kernel_time")
        return ms.value, n.value

    def rgb_time(self):
        """(total_ms, launches) of the m08 RGB launches since the previous call."""
        ms, n = C.c_double(), C.c_int()
        _check(self._L.vp8_gpu_rgb_time(self._h, C.byref(ms), C.byref(n)), "vp8_gpu_rgb_time")
        return ms.value, n.value

    def png_time(self):
        """(total_ms, launch pairs) of the m09 launches (vp8_png_frame + vp8_png_finish) since the previous call."""
        ms, n = C.c_double(), C.c_int()
        _check(self._L.vp8_gpu_png_time(self._h, C.byref(ms), C.byref(n)), "vp8_gpu_png_time")
        return ms.value, n.value

    def last_launch_config(self):
        w, g, s = C.c_int(), C.c_int(), C.c_int()
        _check(self._L.vp8_gpu_last_launch_config(self._h, C.byref(w), C.byref(g), C.byref(s)), "launch config")
        return {"warps_per_image": w.value, "grid": g.value, "smem_bytes": s.value,
                "ctas_per_image": int(self._L.vp8_gpu_last_cluster(self._h)),
                "split": bool(self._L.vp8_gpu_last_split(self._h)),
                "images_per_cta": int(self._L.vp8_gpu_last_groups(self._h)),
                "segments": int(self._L.vp8_gpu_last_segments(self._h))}


# -------------------------------------------------------------------------------------------- reference-shaped calls
def _image_to_i420(img: Yuv420Image) -> np.ndarray:
    w, h = img.width, img.height
    cw, ch = (w + 1) // 2, (h + 1) // 2
    y = np.ctypeslib.as_array(img.y, shape=(h * img.stride_y,))
    u = np.ctypeslib.as_array(img.u, shape=(ch * img.stride_uv,))
    v = np.ctypeslib.as_array(img.v, shape=(ch * img.stride_uv,))
    return np.concatenate([y, u, v]).copy()


def _reconstruct(fn_name: str, kf, decoded) -> np.ndarray:
    L = load_library()
    img = Yuv420Image()
    _check(getattr(L, fn_name)(_addr(kf), _addr(decoded), _addr(img)), fn_name)
    try:
        return _image_to_i420(img)
    finally:
        L.yuv420_free(_addr(img))


def vp8_reconstruct_keyframe_yuv(kf, decoded) -> np.ndarray:
    """m06: tight I420 of the visible frame, loop filter not applied."""
    return _reconstruct("vp8_reconstruct_keyframe_yuv", kf, decoded)


def vp8_reconstruct_keyframe_yuv_filtered(kf, decoded) -> np.ndarray:
    """m06 + m07."""
    return _reconstruct("vp8_reconstruct_keyframe_yuv_filtered", kf, decoded)


def _host_image(y: np.ndarray, u: np.ndarray, v: np.ndarray) -> Yuv420Image:
    u8p = C.POINTER(C.c_uint8)
    return Yuv420Image(y.shape[1], y.shape[0], y.strides[0], u.strides[0], y.ctypes.data_as(u8p), u.ctypes.data_as(u8p),
                       v.ctypes.data_as(u8p))


def vp8_loopfilter_apply_keyframe(y: np.ndarray, u: np.ndarray, v: np.ndarray, decoded) -> None:
    """m07 in place on macroblock-aligned 2-D uint8 planes."""
    img = _host_image(y, u, v)
    _check(load_library().vp8_loopfilter_apply_keyframe(_addr(img), _addr(decoded)), "vp8_loopfilter_apply_keyframe")


def _write_via_fd(fn_name: str, i420: np.ndarray, w: int, h: int) -> bytes:
    import threading
    cw, ch = (w + 1) // 2, (h + 1) // 2
    i420 = np.ascontiguousarray(i420, np.uint8)
    yv = i420[:w * h].reshape(h, w)
    uv = i420[w * h:w * h + cw * ch].reshape(ch, cw)
    vv = i420[w * h + cw * ch:].reshape(ch, cw)
    img = _host_image(yv, uv, vv)
    r, wfd = os.pipe()
    chunks = []

    def drain():
        with os.fdopen(r, "rb") as fp:
            chunks.append(fp.read())
    t = threading.Thread(target=drain)
    t.start()
    try:
        rc = getattr(load_library(), fn_name)(wfd, _addr(img))
        e = C.get_errno()
    finally:
        os.close(wfd)
        t.join()
    if rc != 0:
        C.set_errno(e)
        _check(rc, fn_name)
    return chunks[0]


def yuv420_write_ppm(i420: np.ndarray, w: int, h: int) -> bytes:
    """m08: the bytes yuv420_write_ppm_fd emits for a tight I420 image."""
    return _write_via_fd("yuv420_write_ppm_fd", i420, w, h)


def yuv420_write_png(i420: np.ndarray, w: int, h: int) -> bytes:
    """m09: the bytes yuv420_write_png_fd emits."""
    return _write_via_fd("yuv420_write_png_fd", i420, w, h)
