"""Host-side mirror of the sea-codec crate API over libsea_b200.so (ctypes -> C-ABI -> sm_100a kernels).

Names, argument meaning and error behaviour follow the reference:
  sea_encode / sea_decode / SeaDecodeInfo      src/lib.rs:13-63
  EncoderSettings                              src/encoder.rs:16-35
  SeaEncoder.encode_frame / flush / finalize   src/encoder.rs:50-159
  SeaDecoder.decode_frame / get_header         src/decoder.rs:22-72
  SeaError variants                            src/codec/common.rs:53-64
plus the additive batch API (encode_batch / decode_batch) that the throughput numbers use.

There is no CPU path: importing works anywhere, but every codec call needs libsea_b200.so and a CUDA device and
raises SeaError(CUDA) otherwise.
"""
from __future__ import annotations

import ctypes as C
import os
import weakref
from dataclasses import dataclass
from typing import BinaryIO, List, Optional, Sequence

import numpy as np

from . import build as _build

OK = 0
ERR_READ, ERR_INVALID_PARAMETERS, ERR_INVALID_FILE, ERR_INVALID_FRAME = -1, -2, -3, -4
ERR_ENCODER_CLOSED, ERR_UNSUPPORTED_VERSION, ERR_TOO_MANY_FRAMES, ERR_METADATA_TOO_LARGE, ERR_IO = -5, -6, -7, -8, -9
ERR_CAPACITY, ERR_DOMAIN, ERR_CUDA, ERR_NOMEM = -20, -21, -30, -31
RANGE_SKIP_METADATA, WINDOW_F32_PLANAR = 1, 2  # flag bits of decode_range / decode_windows_device

_NAMES = {
    ERR_READ: "ReadError", ERR_INVALID_PARAMETERS: "InvalidParameters", ERR_INVALID_FILE: "InvalidFile",
    ERR_INVALID_FRAME: "InvalidFrame", ERR_ENCODER_CLOSED: "EncoderClosed", ERR_UNSUPPORTED_VERSION: "UnsupportedVersion",
    ERR_TOO_MANY_FRAMES: "TooManyFrames", ERR_METADATA_TOO_LARGE: "MetadataTooLarge", ERR_IO: "IoError",
    ERR_CAPACITY: "Capacity", ERR_DOMAIN: "Domain", ERR_CUDA: "Cuda", ERR_NOMEM: "NoMem",
}


class SeaError(RuntimeError):
    """SeaError (common.rs:53-64) plus the library's own Capacity / Domain / Cuda codes."""

    def __init__(self, code: int, detail: str = ""):
        self.code = code
        self.kind = _NAMES.get(code, str(code))
        super().__init__(f"SeaError::{self.kind}" + (f": {detail}" if detail else ""))


class _Settings(C.Structure):
    _fields_ = [("scale_factor_bits", C.c_uint8), ("scale_factor_frames", C.c_uint8), ("frames_per_chunk", C.c_uint16),
                ("residual_bits", C.c_float), ("vbr", C.c_uint8), ("reserved", C.c_uint8 * 3)]


class _Header(C.Structure):
    _fields_ = [("version", C.c_uint8), ("channels", C.c_uint8), ("chunk_size", C.c_uint16), ("frames_per_chunk", C.c_uint16),
                ("reserved", C.c_uint16), ("sample_rate", C.c_uint32), ("total_frames", C.c_uint32), ("metadata_size", C.c_uint32)]


@dataclass
class EncoderSettings:
    """encoder.rs:16-35 (same field names and defaults)."""

    scale_factor_bits: int = 4
    scale_factor_frames: int = 20
    residual_bits: float = 3.0
    frames_per_chunk: int = 5120
    vbr: bool = False

    def _c(self) -> _Settings:
        return _Settings(self.scale_factor_bits, self.scale_factor_frames, self.frames_per_chunk, float(self.residual_bits),
                         1 if self.vbr else 0)


@dataclass
class SeaFileHeader:
    """file.rs:21-30."""

    version: int
    channels: int
    chunk_size: int
    frames_per_chunk: int
    sample_rate: int
    total_frames: int
    metadata_size: int = 0


@dataclass
class SeaDecodeInfo:
    """lib.rs:38-42."""

    samples: np.ndarray
    sample_rate: int
    channels: int


_u64p = C.POINTER(C.c_uint64)
_u32p = C.POINTER(C.c_uint32)

# every symbol include/sea_b200.h declares: (restype, argtypes)
SYMBOLS = {
    "sea_b200_ctx_create": (C.c_int, [C.c_int, C.POINTER(C.c_void_p)]),
    "sea_b200_ctx_destroy": (None, [C.c_void_p]),
    "sea_b200_ctx_set_stream": (C.c_int, [C.c_void_p, C.c_void_p]),
    "sea_b200_ctx_stream": (C.c_void_p, [C.c_void_p]),
    "sea_b200_strerror": (C.c_char_p, [C.c_int]),
    "sea_b200_last_error": (C.c_char_p, [C.c_void_p]),
    "sea_b200_abi_version": (C.c_int, []),
    "sea_b200_ctx_launch_count": (C.c_uint64, [C.c_void_p]),
    "sea_b200_host_alloc": (C.c_void_p, [C.c_size_t]),
    "sea_b200_host_free": (None, [C.c_void_p]),
    "sea_b200_default_settings": (None, [C.POINTER(_Settings)]),
    "sea_b200_parse_header": (C.c_int, [C.c_void_p, C.c_uint64, C.POINTER(_Header)]),
    "sea_b200_encode_bound": (C.c_int, [C.c_uint64, C.c_uint32, C.POINTER(_Settings), _u64p]),
    "sea_b200_full_chunk_bytes": (C.c_int, [C.c_uint32, C.POINTER(_Settings), _u32p]),
    "sea_b200_vbr_plan": (C.c_int, [C.POINTER(_Settings), C.c_uint64, C.POINTER(C.c_float), _u32p, C.POINTER(C.c_uint64 * 4)]),
    "sea_b200_tables": (C.c_int, [C.c_uint32, C.c_uint32, C.c_void_p, C.c_void_p]),
    "sea_b200_encode": (C.c_int, [C.c_void_p, C.c_void_p, C.c_uint64, C.c_uint32, C.c_uint32, C.POINTER(_Settings), C.c_void_p,
                                  C.c_uint64, _u64p]),
    "sea_b200_decode": (C.c_int, [C.c_void_p, C.c_void_p, C.c_uint64, C.c_void_p, C.c_uint64, _u64p, _u32p, _u32p]),
    "sea_b200_encode_batch": (C.c_int, [C.c_void_p, C.c_uint32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint32, C.c_uint32,
                                        C.POINTER(_Settings), C.c_void_p, C.c_void_p, C.c_void_p]),
    "sea_b200_decode_batch": (C.c_int, [C.c_void_p, C.c_uint32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                        C.c_void_p, C.c_void_p]),
    "sea_b200_encode_batch_device": (C.c_int, [C.c_void_p, C.c_uint32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint32, C.c_uint32,
                                               C.POINTER(_Settings), C.c_void_p, C.c_void_p, C.c_void_p]),
    "sea_b200_decode_batch_device": (C.c_int, [C.c_void_p, C.c_uint32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                               C.c_void_p, C.c_void_p, C.c_void_p]),
    "sea_b200_encoder_create": (C.c_int, [C.c_void_p, C.c_uint32, C.c_uint32, C.POINTER(_Settings), C.POINTER(C.c_void_p)]),
    "sea_b200_encoder_make_chunk": (C.c_int, [C.c_void_p, C.c_void_p, C.c_uint64, C.c_void_p, C.c_uint64, _u64p]),
    "sea_b200_encoder_chunk_size": (C.c_uint32, [C.c_void_p]),
    "sea_b200_encoder_destroy": (None, [C.c_void_p]),
    "sea_b200_decoder_create": (C.c_int, [C.c_void_p, C.c_void_p, C.c_uint64, C.POINTER(C.c_void_p)]),
    "sea_b200_decoder_header": (C.c_int, [C.c_void_p, C.POINTER(_Header)]),
    "sea_b200_decoder_decode_chunk": (C.c_int, [C.c_void_p, C.c_void_p, C.c_uint64, C.c_int64, C.c_void_p, C.c_uint64, _u64p]),
    "sea_b200_decoder_destroy": (None, [C.c_void_p]),
    "sea_b200_encoder_make_chunks": (C.c_int, [C.c_void_p, C.c_void_p, C.c_uint64, C.c_void_p, C.c_uint64, _u64p, _u32p]),
    "sea_b200_decoder_decode_chunks": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint64, C.c_int64, C.c_void_p, C.c_uint64, _u64p]),
    "sea_b200_decode_range": (C.c_int, [C.c_void_p, C.c_void_p, C.c_uint64, C.c_uint64, C.c_uint64, C.c_uint32, C.c_void_p, C.c_uint64,
                                        _u64p, _u32p, _u32p]),
    "sea_b200_decode_windows_device": (C.c_int, [C.c_void_p, C.c_uint32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint32,
                                                 C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint32, C.c_void_p, C.c_void_p, C.c_void_p]),
    "sea_b200_corpus_create": (C.c_int, [C.c_void_p, C.c_uint32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint32,
                                         C.POINTER(C.c_void_p)]),
    "sea_b200_corpus_destroy": (None, [C.c_void_p]),
    "sea_b200_corpus_info": (C.c_int, [C.c_void_p, _u32p, C.c_void_p, _u32p]),
    "sea_b200_corpus_decode_windows_async": (C.c_int, [C.c_void_p, C.c_uint32, C.c_void_p, C.c_void_p, C.c_uint32, C.c_uint32,
                                                       C.c_void_p, C.c_void_p, C.c_void_p]),
    "sea_b200_wasm_setup": (None, []),
    "sea_b200_wasm_sea_encode": (C.c_size_t, [C.c_void_p, C.c_size_t, C.c_uint32, C.c_uint32, C.c_float, C.c_bool, C.c_void_p, C.c_size_t]),
    "sea_b200_wasm_sea_decode": (C.c_size_t, [C.c_void_p, C.c_size_t, C.c_void_p, C.c_size_t, _u32p, _u32p]),
    "sea_b200_wasm_allocate": (C.c_void_p, [C.c_size_t]),
    "sea_b200_wasm_deallocate": (None, [C.c_void_p, C.c_size_t]),
    "sea_b200_wasm_status": (C.c_int, []),
    "sea_b200_csea_decode": (C.c_int, [C.c_void_p, C.c_uint32, _u32p, _u32p, C.c_void_p, _u32p]),
    "sea_b200_int32_peak": (C.c_int, [C.c_void_p, C.c_int, C.POINTER(C.c_double), C.POINTER(C.c_double)]),
    "sea_b200_last_kernel_ms": (C.c_double, [C.c_void_p]),
    "sea_b200_last_vbr_ties": (C.c_uint64, [C.c_void_p]),
    "sea_b200_multi_create": (C.c_int, [C.c_void_p, C.c_uint32, C.POINTER(C.c_void_p)]),
    "sea_b200_multi_destroy": (None, [C.c_void_p]),
    "sea_b200_multi_device_count": (C.c_uint32, [C.c_void_p]),
    "sea_b200_multi_ctx": (C.c_void_p, [C.c_void_p, C.c_uint32]),
    "sea_b200_multi_last_error": (C.c_char_p, [C.c_void_p]),
    "sea_b200_multi_encode_batch": (C.c_int, [C.c_void_p, C.c_uint32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint32, C.c_uint32,
                                              C.POINTER(_Settings), C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "sea_b200_multi_decode_batch": (C.c_int, [C.c_void_p, C.c_uint32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                              C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "sea_b200_last_vbr_ties_per_stream": (C.c_int, [C.c_void_p, C.c_void_p, C.c_uint32]),
    "sea_b200_synth_pcm_device": (C.c_int, [C.c_void_p, C.c_void_p, C.c_uint64, C.c_uint32, C.c_uint32, C.c_uint32, C.c_void_p, C.c_void_p,
                                            C.c_void_p, C.c_uint64, C.c_int32, C.c_int32]),
}

_lib = None


def lib() -> C.CDLL:
    """Loads (building first when the sources are newer) sea_codec_b200/libsea_b200.so.  Fails loudly if absent."""
    global _lib
    if _lib is None:
        path = os.environ.get("SEA_B200_LIB") or _build.LIB  # override: a tuning build of the same C-ABI (tools/build_variant.py)
        try:
            if path == _build.LIB and _build.is_stale():
                _build.build()
        except Exception as e:  # no nvcc on this box: use the prebuilt library if there is one
            if not os.path.exists(path):
                raise SeaError(ERR_CUDA, f"libsea_b200.so is not built and cannot be built here ({e})")
        L = C.CDLL(path)
        for name, (res, args) in SYMBOLS.items():
            fn = getattr(L, name)
            fn.restype = res
            fn.argtypes = args
        _lib = L
    return _lib


def _u64(a) -> np.ndarray:
    return np.ascontiguousarray(a, dtype=np.uint64)


class Context:
    """One GPU + one CUDA stream (sea_b200_ctx).  Use from one thread at a time."""

    def __init__(self, device: int = 0):
        self._h = C.c_void_p()
        self._L = lib()
        rc = self._L.sea_b200_ctx_create(device, C.byref(self._h))
        if rc:
            raise SeaError(rc, "no usable CUDA device for libsea_b200 (there is no CPU fallback)")
        self.device = device
        self._corpora = weakref.WeakSet()  # sea_b200_corpus_destroy uses its context: they are closed before it

    def close(self):
        if getattr(self, "_h", None) and self._h.value:
            for corpus in list(getattr(self, "_corpora", ())):
                corpus.close()
            self._L.sea_b200_ctx_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _check(self, rc: int):
        if rc < 0:
            raise SeaError(rc, self._L.sea_b200_last_error(self._h).decode(errors="replace"))
        return rc

    def set_stream(self, cuda_stream: int):
        self._check(self._L.sea_b200_ctx_set_stream(self._h, C.c_void_p(cuda_stream)))

    @property
    def stream(self) -> int:
        return self._L.sea_b200_ctx_stream(self._h) or 0

    @property
    def launch_count(self) -> int:
        return self._L.sea_b200_ctx_launch_count(self._h)

    @property
    def last_kernel_ms(self) -> float:
        return self._L.sea_b200_last_kernel_ms(self._h)

    @property
    def last_vbr_ties(self) -> int:
        return self._L.sea_b200_last_vbr_ties(self._h)

    def last_vbr_ties_per_stream(self, n_streams: int) -> np.ndarray:
        out = np.zeros(n_streams, dtype=np.uint64)
        self._check(self._L.sea_b200_last_vbr_ties_per_stream(self._h, out.ctypes.data, n_streams))
        return out

    def synth_pcm_device(self, d_pcm: int, stream_stride_samples: int, stream_ids, n_frames: int, channels: int, rate: int) -> None:
        """Fills device memory with the synthetic streams synth.gen_stream(id, n_frames, channels, rate) of the given ids."""
        from . import synth

        ids = np.ascontiguousarray(stream_ids, dtype=np.uint32)
        steps = np.array([synth._step(int(k), rate) for k in ids], dtype=np.uint32)
        tab = np.ascontiguousarray(synth.sine_table(), dtype=np.int32)
        self._check(self._L.sea_b200_synth_pcm_device(self._h, C.c_void_p(d_pcm), stream_stride_samples, ids.size, n_frames, channels,
                                                      ids.ctypes.data, steps.ctypes.data, tab.ctypes.data, synth.SEED, synth._A,
                                                      synth._NOISE_AMP))

    def int32_peak(self, mode: int):
        ops, ms = C.c_double(0), C.c_double(0)
        self._check(self._L.sea_b200_int32_peak(self._h, mode, C.byref(ops), C.byref(ms)))
        return ops.value, ms.value

    # ---- one-shot ------------------------------------------------------------------------------------------
    def sea_encode(self, input_samples, sample_rate: int, channels: int, settings: EncoderSettings) -> bytes:
        s = np.ascontiguousarray(input_samples, dtype=np.int16).reshape(-1)
        st = settings._c()
        bound = C.c_uint64(0)
        if channels <= 0:
            raise SeaError(ERR_INVALID_PARAMETERS, "channels must be positive")
        self._check(self._L.sea_b200_encode_bound(s.size // channels, channels, C.byref(st), C.byref(bound)))
        out = np.empty(bound.value + 64, dtype=np.uint8)
        n = C.c_uint64(0)
        self._check(self._L.sea_b200_encode(self._h, s.ctypes.data, s.size, sample_rate, channels, C.byref(st), out.ctypes.data,
                                            out.size, C.byref(n)))
        return out[: n.value].tobytes()

    def sea_decode(self, encoded: bytes) -> SeaDecodeInfo:
        buf = np.frombuffer(encoded, dtype=np.uint8)
        n, rate, ch = C.c_uint64(0), C.c_uint32(0), C.c_uint32(0)
        self._check(self._L.sea_b200_decode(self._h, buf.ctypes.data, buf.size, None, 0, C.byref(n), C.byref(rate), C.byref(ch)))
        out = np.empty(max(int(n.value), 1), dtype=np.int16)
        self._check(self._L.sea_b200_decode(self._h, buf.ctypes.data, buf.size, out.ctypes.data, out.size, C.byref(n), C.byref(rate),
                                            C.byref(ch)))
        return SeaDecodeInfo(out[: n.value], rate.value, ch.value)

    def decode_range(self, encoded: bytes, first_frame: int, n_frames: int, skip_metadata: bool = False) -> SeaDecodeInfo:
        """Random access: frames [first_frame, first_frame + n_frames) of a .sea file; only the covering chunks are decoded."""
        buf = np.frombuffer(encoded, dtype=np.uint8)
        n, rate, ch = C.c_uint64(0), C.c_uint32(0), C.c_uint32(0)
        flags = 1 if skip_metadata else 0
        self._check(self._L.sea_b200_decode_range(self._h, buf.ctypes.data, buf.size, first_frame, n_frames, flags, None, 0, C.byref(n),
                                                  C.byref(rate), C.byref(ch)))
        out = np.empty(max(int(n.value), 1), dtype=np.int16)
        self._check(self._L.sea_b200_decode_range(self._h, buf.ctypes.data, buf.size, first_frame, n_frames, flags, out.ctypes.data,
                                                  out.size, C.byref(n), C.byref(rate), C.byref(ch)))
        return SeaDecodeInfo(out[: n.value], rate.value, ch.value)

    # ---- batch, host buffers ---------------------------------------------------------------------------------
    def encode_bound(self, n_frames: int, channels: int, settings: EncoderSettings) -> int:
        st = settings._c()
        b = C.c_uint64(0)
        self._check(self._L.sea_b200_encode_bound(n_frames, channels, C.byref(st), C.byref(b)))
        return b.value

    def encode_batch(self, streams: Sequence[np.ndarray], sample_rate: int, channels: int, settings: EncoderSettings) -> List[bytes]:
        """n independent sea_encode calls in one launch.  streams: interleaved int16 arrays."""
        arrs = [np.ascontiguousarray(a, dtype=np.int16).reshape(-1) for a in streams]
        frames = np.array([a.size // channels for a in arrs], dtype=np.uint32)
        pcm_off = np.zeros(len(arrs), dtype=np.uint64)
        total = 0
        for i, a in enumerate(arrs):
            pcm_off[i] = total
            total += int(frames[i]) * channels
        pcm = np.empty(max(total, 1), dtype=np.int16)
        for i, a in enumerate(arrs):
            pcm[int(pcm_off[i]): int(pcm_off[i]) + int(frames[i]) * channels] = a[: int(frames[i]) * channels]
        out_off = np.zeros(len(arrs), dtype=np.uint64)
        cap = 0
        for i in range(len(arrs)):
            out_off[i] = cap
            cap += (self.encode_bound(int(frames[i]), channels, settings) + 15) // 16 * 16
        out = np.empty(cap + 64, dtype=np.uint8)
        lens = np.zeros(len(arrs), dtype=np.uint64)
        st = settings._c()
        self._check(self._L.sea_b200_encode_batch(self._h, len(arrs), pcm.ctypes.data, pcm_off.ctypes.data, frames.ctypes.data,
                                                  sample_rate, channels, C.byref(st), out.ctypes.data, out_off.ctypes.data,
                                                  lens.ctypes.data))
        return [out[int(o): int(o) + int(n)].tobytes() for o, n in zip(out_off, lens)]

    def decode_batch(self, files: Sequence[bytes]) -> List[SeaDecodeInfo]:
        """n independent sea_decode calls in one launch."""
        L = self._L
        hdrs = []
        for f in files:
            h = _Header()
            rc = L.sea_b200_parse_header(np.frombuffer(f, dtype=np.uint8).ctypes.data if len(f) else None, len(f), C.byref(h)) \
                if len(f) else ERR_IO
            if rc:
                raise SeaError(rc, "bad .sea header")
            hdrs.append(h)
        sea_off = np.zeros(len(files), dtype=np.uint64)
        sea_len = np.array([len(f) for f in files], dtype=np.uint64)
        total = 0
        for i, f in enumerate(files):
            sea_off[i] = total
            total += (len(f) + 15) // 16 * 16
        sea = np.zeros(total + 64, dtype=np.uint8)
        for i, f in enumerate(files):
            sea[int(sea_off[i]): int(sea_off[i]) + len(f)] = np.frombuffer(f, dtype=np.uint8)
        caps = np.zeros(len(files), dtype=np.uint64)
        for i, (f, h) in enumerate(zip(files, hdrs)):
            n_chunks = (len(f) - 22 + h.chunk_size - 1) // h.chunk_size
            caps[i] = n_chunks * h.frames_per_chunk * h.channels
        pcm_off = np.zeros(len(files), dtype=np.uint64)
        ptotal = 0
        for i in range(len(files)):
            pcm_off[i] = ptotal
            ptotal += (int(caps[i]) + 15) // 16 * 16
        pcm = np.empty(ptotal + 64, dtype=np.int16)
        n_samples = np.zeros(len(files), dtype=np.uint64)
        self._check(L.sea_b200_decode_batch(self._h, len(files), sea.ctypes.data, sea_off.ctypes.data, sea_len.ctypes.data,
                                            pcm.ctypes.data, pcm_off.ctypes.data, caps.ctypes.data, n_samples.ctypes.data))
        return [SeaDecodeInfo(pcm[int(o): int(o) + int(n)].copy(), h.sample_rate, h.channels)
                for o, n, h in zip(pcm_off, n_samples, hdrs)]

    # ---- batch, caller-owned HOST buffers by raw address (pinned memory recommended) ----------------------------------
    def encode_batch_host(self, pcm_ptr: int, pcm_offsets, n_frames, sample_rate: int, channels: int, settings: EncoderSettings,
                          out_ptr: int, out_offsets) -> np.ndarray:
        po, oo = _u64(pcm_offsets), _u64(out_offsets)
        nf = np.ascontiguousarray(n_frames, dtype=np.uint32)
        lens = np.zeros(nf.size, dtype=np.uint64)
        st = settings._c()
        self._check(self._L.sea_b200_encode_batch(self._h, nf.size, C.c_void_p(pcm_ptr), po.ctypes.data, nf.ctypes.data, sample_rate,
                                                  channels, C.byref(st), C.c_void_p(out_ptr), oo.ctypes.data, lens.ctypes.data))
        return lens

    def decode_batch_host(self, sea_ptr: int, sea_offsets, sea_lens, pcm_ptr: int, pcm_offsets, pcm_caps=None) -> np.ndarray:
        so, sl, po = _u64(sea_offsets), _u64(sea_lens), _u64(pcm_offsets)
        caps = _u64(pcm_caps) if pcm_caps is not None else None
        n = np.zeros(so.size, dtype=np.uint64)
        self._check(self._L.sea_b200_decode_batch(self._h, so.size, C.c_void_p(sea_ptr), so.ctypes.data, sl.ctypes.data,
                                                  C.c_void_p(pcm_ptr), po.ctypes.data, caps.ctypes.data if caps is not None else None,
                                                  n.ctypes.data))
        return n

    # ---- batch, device-resident (raw device pointers; torch tensors expose them as .data_ptr()) -------------------
    def encode_batch_device(self, d_pcm: int, pcm_offsets, n_frames, sample_rate: int, channels: int, settings: EncoderSettings,
                            d_out: int, out_offsets) -> np.ndarray:
        po, oo = _u64(pcm_offsets), _u64(out_offsets)
        nf = np.ascontiguousarray(n_frames, dtype=np.uint32)
        lens = np.zeros(nf.size, dtype=np.uint64)
        st = settings._c()
        self._check(self._L.sea_b200_encode_batch_device(self._h, nf.size, C.c_void_p(d_pcm), po.ctypes.data, nf.ctypes.data, sample_rate,
                                                         channels, C.byref(st), C.c_void_p(d_out), oo.ctypes.data, lens.ctypes.data))
        return lens

    def decode_batch_device(self, d_sea: int, sea_offsets, sea_lens, headers: np.ndarray, d_pcm: int, pcm_offsets,
                            pcm_caps=None) -> np.ndarray:
        so, sl, po = _u64(sea_offsets), _u64(sea_lens), _u64(pcm_offsets)
        hd = np.ascontiguousarray(headers, dtype=np.uint8)
        caps = _u64(pcm_caps) if pcm_caps is not None else None
        n = np.zeros(so.size, dtype=np.uint64)
        self._check(self._L.sea_b200_decode_batch_device(self._h, so.size, C.c_void_p(d_sea), so.ctypes.data, sl.ctypes.data,
                                                         hd.ctypes.data, C.c_void_p(d_pcm), po.ctypes.data,
                                                         caps.ctypes.data if caps is not None else None, n.ctypes.data))
        return n

    def decode_windows_device(self, d_sea: int, sea_offsets, sea_lens, headers: np.ndarray, window_stream, first_frames, n_frames,
                              d_out: int, out_offsets, float32_planar: bool = False, skip_metadata: bool = False) -> np.ndarray:
        """Frame windows [first_frames[w], first_frames[w] + n_frames[w]) of device-resident streams window_stream[w] (described as
        for decode_batch_device) into slots of d_out starting at element out_offsets[w]: int16 [n_frames][channels], or with
        float32_planar float32 [channels][n_frames] = sample / 32768.  Each slot holds what decode_range returns for its window,
        then zeros.  Returns frames_out, the real frames per window."""
        so, sl = _u64(sea_offsets), _u64(sea_lens)
        hd = np.ascontiguousarray(headers, dtype=np.uint8)
        ws = np.ascontiguousarray(window_stream, dtype=np.uint32)
        ff, oo = _u64(first_frames), _u64(out_offsets)
        nf = np.ascontiguousarray(n_frames, dtype=np.uint32)
        if not (ws.size == ff.size == nf.size == oo.size):
            raise SeaError(ERR_INVALID_PARAMETERS, "window arrays differ in length")
        if so.size != sl.size or hd.size < so.size * 22:
            raise SeaError(ERR_INVALID_PARAMETERS, "stream arrays differ in length")
        flags = (WINDOW_F32_PLANAR if float32_planar else 0) | (RANGE_SKIP_METADATA if skip_metadata else 0)
        out = np.zeros(ws.size, dtype=np.uint64)
        self._check(self._L.sea_b200_decode_windows_device(self._h, so.size, C.c_void_p(d_sea), so.ctypes.data, sl.ctypes.data,
                                                           hd.ctypes.data, ws.size, ws.ctypes.data, ff.ctypes.data, nf.ctypes.data, flags,
                                                           C.c_void_p(d_out), oo.ctypes.data, out.ctypes.data))
        return out

    def corpus(self, buf, sea_offsets, sea_lens, headers: np.ndarray, skip_metadata: bool = False) -> "Corpus":
        """Registers the .sea streams held in `buf` (a uint8 CUDA tensor; streams described as for decode_windows_device) for
        Corpus.decode_windows.  Every chunk a window can cover is validated here, once."""
        return Corpus(self, buf, sea_offsets, sea_lens, headers, skip_metadata)


class Corpus:
    """A registered corpus (sea_b200_corpus): fixed-length windows decoded from device-side indices on the current torch stream,
    with no host synchronisation, so the call can sit inside torch.cuda.graph(...).  Keeps `buf` and its Context alive.  A loader
    draws valid starts on the device, e.g. (torch.rand(n, device=dev) * (stream_frames_cuda[s] - W + 1)).long()."""

    def __init__(self, ctx: Context, buf, sea_offsets, sea_lens, headers: np.ndarray, skip_metadata: bool = False):
        import torch

        if not (isinstance(buf, torch.Tensor) and buf.is_cuda and buf.dtype == torch.uint8 and buf.is_contiguous()):
            raise SeaError(ERR_INVALID_PARAMETERS, "buf must be a contiguous uint8 CUDA tensor")
        so, sl = _u64(sea_offsets), _u64(sea_lens)
        hd = np.ascontiguousarray(headers, dtype=np.uint8)
        if so.size != sl.size or hd.size < so.size * 22:
            raise SeaError(ERR_INVALID_PARAMETERS, "stream arrays differ in length")
        if so.size and int(np.max(so + sl)) > buf.numel():
            raise SeaError(ERR_INVALID_PARAMETERS, "a stream runs past the end of buf")
        self._h = C.c_void_p()
        self._ctx, self._L, self._buf = ctx, ctx._L, buf
        self.device = torch.device("cuda", ctx.device)
        # bind the context to torch's stream now: dropping its own stream synchronises, which a later capture must not do
        ctx.set_stream(torch.cuda.current_stream(self.device).cuda_stream)
        ctx._check(self._L.sea_b200_corpus_create(ctx._h, so.size, C.c_void_p(buf.data_ptr()), so.ctypes.data, sl.ctypes.data,
                                                  hd.ctypes.data, RANGE_SKIP_METADATA if skip_metadata else 0, C.byref(self._h)))
        ch, route = C.c_uint32(0), C.c_uint32(0)
        self.stream_frames = np.zeros(so.size, dtype=np.uint64)
        ctx._check(self._L.sea_b200_corpus_info(self._h, C.byref(ch), self.stream_frames.ctypes.data, C.byref(route)))
        self.n_streams = int(so.size)
        self.channels = int(ch.value)
        self.route = "fast" if route.value else "generic"
        self.stream_frames_cuda = torch.from_numpy(self.stream_frames.astype(np.int64)).to(self.device)
        self._status = torch.zeros(1, dtype=torch.int32, device=self.device)
        ctx._corpora.add(self)

    def close(self):
        if getattr(self, "_h", None) and self._h.value:
            # The garbage collector may finalise a context before a corpus that refers to it (a reference cycle, whose weak
            # references it clears first): the corpus's device table is then left to the process, not freed through a
            # destroyed context.
            if self._ctx._h.value:
                self._L.sea_b200_corpus_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    @property
    def status(self):
        """The persistent int32 status tensor decode_windows uses by default (0, or the first error's SeaError code)."""
        return self._status

    def decode_windows(self, stream_idx, first_frames, window_frames: int, *, float32_planar: bool = False, out=None,
                       frames_out=None, status=None):
        """Windows [first_frames[w], + window_frames) of streams stream_idx[w] (int32 or int64 CUDA tensors) into `out`: int16
        [n, window_frames, channels], or with float32_planar float32 [n, channels, window_frames] = sample / 32768 (allocated when
        not given; a given `out` is any contiguous CUDA tensor of that dtype and element count).  Each slot holds what decode_range
        returns for its window, then zeros; frames_out (int32 CUDA tensor of n, optional) gets the real frames per window.  A
        stream index out of range zero-fills its slot and sets `status` (default: the corpus's own, see check()).  Enqueued on
        torch.cuda.current_stream() without host synchronisation or allocation beyond `out`."""
        import torch

        n = stream_idx.numel()
        if first_frames.numel() != n:
            raise SeaError(ERR_INVALID_PARAMETERS, "stream_idx and first_frames differ in length")
        for t in (stream_idx, first_frames):
            if not (t.is_cuda and t.dtype in (torch.int32, torch.int64)):
                raise SeaError(ERR_INVALID_PARAMETERS, "indices must be int32 or int64 CUDA tensors")
        W, ch = int(window_frames), self.channels
        if not 0 <= W < 2**32:
            raise SeaError(ERR_INVALID_PARAMETERS, "window_frames must fit 32 bits")
        # uint32 stream indices: a negative or too large index stays out of range (-1 -> 0xffffffff)
        si = stream_idx.reshape(-1)
        if si.dtype == torch.int64:
            si = si.clamp(-1, 2**31 - 1).to(torch.int32)
        si = si.contiguous()
        ff = first_frames.reshape(-1).to(torch.int64).contiguous()  # read as uint64: negative starts lie past every stream's end
        dtype = torch.float32 if float32_planar else torch.int16
        if out is None:
            out = torch.empty((n, ch, W) if float32_planar else (n, W, ch), dtype=dtype, device=self.device)
        elif not (out.is_cuda and out.dtype == dtype and out.is_contiguous() and out.numel() == n * W * ch):
            raise SeaError(ERR_INVALID_PARAMETERS, f"out must be a contiguous {dtype} CUDA tensor of {n * W * ch} elements")
        fo = 0
        if frames_out is not None:
            if not (frames_out.is_cuda and frames_out.dtype == torch.int32 and frames_out.is_contiguous() and frames_out.numel() == n):
                raise SeaError(ERR_INVALID_PARAMETERS, "frames_out must be a contiguous int32 CUDA tensor of n elements")
            fo = frames_out.data_ptr()
        st = self._status if status is None else status
        if not (st.is_cuda and st.dtype == torch.int32 and st.numel() >= 1):
            raise SeaError(ERR_INVALID_PARAMETERS, "status must be an int32 CUDA tensor")
        self._ctx.set_stream(torch.cuda.current_stream(self.device).cuda_stream)
        flags = WINDOW_F32_PLANAR if float32_planar else 0
        self._ctx._check(self._L.sea_b200_corpus_decode_windows_async(self._h, n, C.c_void_p(si.data_ptr()), C.c_void_p(ff.data_ptr()),
                                                                      W, flags, C.c_void_p(out.data_ptr()), C.c_void_p(fo),
                                                                      C.c_void_p(st.data_ptr())))
        return out

    def check(self):
        """Synchronises with the corpus's status tensor, raises SeaError if a call stored an error there, and clears it."""
        code = int(self._status.item())
        if code:
            self._status.zero_()
            raise SeaError(code, "a window named a stream index out of range")


class MultiContext:
    """One context per GPU of the box (sea_b200_multi): batch calls shard the streams over the GPUs in-process, one host thread
    per GPU, nothing exchanged between them; per-GPU counts come back with the result (SURVEY 8e)."""

    def __init__(self, devices: Sequence[int]):
        self._L = lib()
        self._h = C.c_void_p()
        devs = np.ascontiguousarray(devices, dtype=np.int32)
        rc = self._L.sea_b200_multi_create(devs.ctypes.data, devs.size, C.byref(self._h))
        if rc:
            raise SeaError(rc, "sea_b200_multi_create failed (no CPU fallback)")
        self.devices = list(int(d) for d in devs)

    def close(self):
        if getattr(self, "_h", None) and self._h.value:
            self._L.sea_b200_multi_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _check(self, rc: int):
        if rc < 0:
            raise SeaError(rc, self._L.sea_b200_multi_last_error(self._h).decode(errors="replace"))

    def encode_batch_host(self, pcm_ptr: int, pcm_offsets, n_frames, sample_rate: int, channels: int, settings: EncoderSettings,
                          out_ptr: int, out_offsets):
        """-> (out_lens[n], first_stream_of_device[g], bytes_per_device[g])"""
        po, oo = _u64(pcm_offsets), _u64(out_offsets)
        nf = np.ascontiguousarray(n_frames, dtype=np.uint32)
        lens = np.zeros(nf.size, dtype=np.uint64)
        first = np.zeros(len(self.devices), dtype=np.uint32)
        per = np.zeros(len(self.devices), dtype=np.uint64)
        st = settings._c()
        self._check(self._L.sea_b200_multi_encode_batch(self._h, nf.size, C.c_void_p(pcm_ptr), po.ctypes.data, nf.ctypes.data, sample_rate,
                                                        channels, C.byref(st), C.c_void_p(out_ptr), oo.ctypes.data, lens.ctypes.data,
                                                        first.ctypes.data, per.ctypes.data))
        return lens, first, per

    def decode_batch_host(self, sea_ptr: int, sea_offsets, sea_lens, pcm_ptr: int, pcm_offsets, pcm_caps=None):
        """-> (n_samples[n], first_stream_of_device[g], samples_per_device[g])"""
        so, sl, po = _u64(sea_offsets), _u64(sea_lens), _u64(pcm_offsets)
        caps = _u64(pcm_caps) if pcm_caps is not None else None
        n = np.zeros(so.size, dtype=np.uint64)
        first = np.zeros(len(self.devices), dtype=np.uint32)
        per = np.zeros(len(self.devices), dtype=np.uint64)
        self._check(self._L.sea_b200_multi_decode_batch(self._h, so.size, C.c_void_p(sea_ptr), so.ctypes.data, sl.ctypes.data,
                                                        C.c_void_p(pcm_ptr), po.ctypes.data, caps.ctypes.data if caps is not None else None,
                                                        n.ctypes.data, first.ctypes.data, per.ctypes.data))
        return n, first, per


_default_ctx: Optional[Context] = None


def default_context() -> Context:
    global _default_ctx
    if _default_ctx is None:
        _default_ctx = Context(0)
    return _default_ctx


def sea_encode(input_samples, sample_rate: int, channels: int, settings: EncoderSettings, ctx: Optional[Context] = None) -> bytes:
    """lib.rs:13-36."""
    return (ctx or default_context()).sea_encode(input_samples, sample_rate, channels, settings)


def sea_decode(encoded: bytes, ctx: Optional[Context] = None) -> SeaDecodeInfo:
    """lib.rs:44-63."""
    return (ctx or default_context()).sea_decode(encoded)


def parse_header(data: bytes) -> SeaFileHeader:
    h = _Header()
    buf = np.frombuffer(data[:22], dtype=np.uint8)
    rc = lib().sea_b200_parse_header(buf.ctypes.data if buf.size else None, buf.size, C.byref(h)) if buf.size else ERR_IO
    if rc:
        raise SeaError(rc, "bad .sea header")
    return SeaFileHeader(h.version, h.channels, h.chunk_size, h.frames_per_chunk, h.sample_rate, h.total_frames, h.metadata_size)


def _read_max_or_zero(reader: BinaryIO, n: int) -> bytes:
    """common.rs:103-123."""
    parts, got = [], 0
    while got < n:
        b = reader.read(n - got)
        if not b:
            break
        parts.append(b)
        got += len(b)
    return b"".join(parts)


def _serialize_header(channels, chunk_size, frames_per_chunk, sample_rate, total_frames) -> bytes:
    """file.rs:78-93 with empty metadata."""
    import struct

    return b"seac" + struct.pack("<BBHHIII", 1, channels, chunk_size & 0xFFFF, frames_per_chunk, sample_rate, total_frames, 0)


class SeaEncoder:
    """SeaEncoder<R, W> (encoder.rs:37-159): reader yields little-endian interleaved i16 bytes, writer takes .sea bytes."""

    START, WRITING, FINISHED = 0, 1, 2

    def __init__(self, channels: int, sample_rate: int, total_frames: Optional[int], settings: EncoderSettings, reader: BinaryIO,
                 writer: BinaryIO, ctx: Optional[Context] = None):
        self._ctx = ctx or default_context()
        self._L = self._ctx._L
        self.channels, self.sample_rate = channels, sample_rate
        self.total_frames = total_frames or 0
        self.settings = settings
        self.reader, self.writer = reader, writer
        self.written_frames = 0
        self.state = self.START
        self._h = C.c_void_p()
        st = settings._c()
        self._ctx._check(self._L.sea_b200_encoder_create(self._ctx._h, channels, sample_rate, C.byref(st), C.byref(self._h)))
        if total_frames is not None and total_frames == 0:  # encoder.rs:73-78
            self.writer.write(_serialize_header(channels, 0, settings.frames_per_chunk, sample_rate, 0))
            self.state = self.WRITING

    @property
    def chunk_size(self) -> int:
        return self._L.sea_b200_encoder_chunk_size(self._h)

    def encode_frame(self) -> bool:
        """encoder.rs:106-149; returns True while more input is expected."""
        if self.state == self.FINISHED:
            raise SeaError(ERR_ENCODER_CLOSED)
        fpc = self.settings.frames_per_chunk
        frames = min(fpc, self.total_frames - self.written_frames) if self.total_frames > 0 else fpc
        full = fpc * self.channels
        raw = _read_max_or_zero(self.reader, frames * self.channels * 2)
        if len(raw) % (2 * self.channels) != 0:
            raise SeaError(ERR_IO, "UnexpectedEof (encoder.rs:95-99)")
        samples = np.frombuffer(raw, dtype="<i2")
        eof = samples.size == 0 or samples.size < full
        if samples.size:
            out = np.empty(70000, dtype=np.uint8)
            n = C.c_uint64(0)
            s = np.ascontiguousarray(samples)
            self._ctx._check(self._L.sea_b200_encoder_make_chunk(self._h, s.ctypes.data, s.size, out.ctypes.data, out.size, C.byref(n)))
            chunk = out[: n.value].tobytes()
            if eof:
                assert len(chunk) <= self.chunk_size
            else:
                assert len(chunk) == self.chunk_size
            if self.state == self.START:  # header goes out after the first chunk fixed chunk_size (encoder.rs:134-138)
                self.writer.write(_serialize_header(self.channels, self.chunk_size, fpc, self.sample_rate, self.total_frames))
                self.state = self.WRITING
            self.writer.write(chunk)
            self.written_frames += frames
        if eof:
            self.state = self.FINISHED
        return not eof

    def encode_frames(self, max_chunks: int) -> bool:
        """Up to max_chunks encode_frame() steps in ONE launch (sea_b200_encoder_make_chunks): same bytes, same state machine,
        one H2D / kernel / D2H per call instead of one per chunk.  Returns True while more input is expected."""
        if self.state == self.FINISHED:
            raise SeaError(ERR_ENCODER_CLOSED)
        fpc = self.settings.frames_per_chunk
        want = fpc * max_chunks
        frames = min(want, self.total_frames - self.written_frames) if self.total_frames > 0 else want
        raw = _read_max_or_zero(self.reader, frames * self.channels * 2)
        if len(raw) % (2 * self.channels) != 0:
            raise SeaError(ERR_IO, "UnexpectedEof (encoder.rs:95-99)")
        samples = np.ascontiguousarray(np.frombuffer(raw, dtype="<i2"))
        eof = samples.size == 0 or samples.size < want * self.channels
        if samples.size:
            out = np.empty(70000 * max_chunks, dtype=np.uint8)
            n, nck = C.c_uint64(0), C.c_uint32(0)
            self._ctx._check(self._L.sea_b200_encoder_make_chunks(self._h, samples.ctypes.data, samples.size, out.ctypes.data, out.size,
                                                                  C.byref(n), C.byref(nck)))
            if self.state == self.START:
                self.writer.write(_serialize_header(self.channels, self.chunk_size, fpc, self.sample_rate, self.total_frames))
                self.state = self.WRITING
            self.writer.write(out[: n.value].tobytes())
            self.written_frames += samples.size // self.channels
        if eof:
            self.state = self.FINISHED
        return not eof

    def flush(self):
        if hasattr(self.writer, "flush"):
            self.writer.flush()

    def finalize(self):
        self.flush()
        self.state = self.FINISHED

    def close(self):
        if self._h.value:
            self._L.sea_b200_encoder_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class SeaDecoder:
    """SeaDecoder<R, W> (decoder.rs:10-72)."""

    def __init__(self, reader: BinaryIO, writer: BinaryIO, ctx: Optional[Context] = None):
        self._ctx = ctx or default_context()
        self._L = self._ctx._L
        self.reader, self.writer = reader, writer
        hdr = _read_max_or_zero(reader, 22)
        self._h = C.c_void_p()
        buf = np.frombuffer(hdr, dtype=np.uint8)
        if buf.size < 22:
            raise SeaError(ERR_IO, "short header")
        self._ctx._check(self._L.sea_b200_decoder_create(self._ctx._h, buf.ctypes.data, buf.size, C.byref(self._h)))
        self.header = parse_header(hdr)
        self.frames_read = 0

    def decode_frame(self) -> bool:
        """decoder.rs:33-59 + file.rs:180-209."""
        h = self.header
        if h.total_frames != 0 and h.total_frames <= self.frames_read:
            return False
        remaining = h.total_frames - self.frames_read if h.total_frames > 0 else -1
        encoded = _read_max_or_zero(self.reader, h.chunk_size)
        if not encoded:
            return False
        buf = np.frombuffer(encoded, dtype=np.uint8)
        out = np.empty(h.frames_per_chunk * h.channels, dtype=np.int16)
        n = C.c_uint64(0)
        self._ctx._check(self._L.sea_b200_decoder_decode_chunk(self._h, buf.ctypes.data, buf.size, remaining, out.ctypes.data, out.size,
                                                               C.byref(n)))
        self.frames_read += n.value // h.channels
        self.writer.write(out[: n.value].astype("<i2").tobytes())
        return True

    def decode_frames(self, max_chunks: int) -> bool:
        """Up to max_chunks decode_frame() steps in one chunk-parallel launch (sea_b200_decoder_decode_chunks)."""
        h = self.header
        if h.total_frames != 0 and h.total_frames <= self.frames_read:
            return False
        remaining = h.total_frames - self.frames_read if h.total_frames > 0 else -1
        encoded = _read_max_or_zero(self.reader, h.chunk_size * max_chunks)
        if not encoded:
            return False
        buf = np.frombuffer(encoded, dtype=np.uint8)
        out = np.empty(h.frames_per_chunk * h.channels * max_chunks, dtype=np.int16)
        n = C.c_uint64(0)
        self._ctx._check(self._L.sea_b200_decoder_decode_chunks(self._h, self._ctx._h, buf.ctypes.data, buf.size, remaining,
                                                                out.ctypes.data, out.size, C.byref(n)))
        self.frames_read += n.value // h.channels
        self.writer.write(out[: n.value].astype("<i2").tobytes())
        return True

    def flush(self):
        if hasattr(self.writer, "flush"):
            self.writer.flush()

    def finalize(self):
        self.flush()

    def get_header(self) -> SeaFileHeader:
        return self.header

    def close(self):
        if self._h.value:
            self._L.sea_b200_decoder_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass
