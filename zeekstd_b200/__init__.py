"""zeekstd_b200 -- B200-native seekable-Zstandard codec behind rorosen/zeekstd's API surface.

Python mirror of the reference's public items (lib/src/lib.rs:38-58) over the C ABI in
include/zeekstd_b200.h; every codec byte is produced by the CUDA kernels in csrc/.

    Encoder / RawEncoder / EncodeOptions / FrameSizePolicy     lib/src/encode.rs
    Decoder / DecodeOptions                                     lib/src/decode.rs
    SeekTable / Serializer / Format                             lib/src/seek_table.rs
    BytesWrapper / OffsetFrom / Seekable                        lib/src/seekable.rs
    Error                                                       lib/src/error.rs

There is no CPU fallback: constructing a Context without a usable CUDA device raises Error.
"""
from __future__ import annotations

import ctypes
import io
from ctypes import byref, c_size_t, c_uint32, c_uint64, c_void_p

import numpy as np

from . import _native
from ._native import CompressionProgress, EpilogueProgress

SEEKABLE_MAGIC_NUMBER = 0x8F92EAB1      # lib.rs:52
SEEKABLE_MAX_FRAMES = 0x08000000        # lib.rs:54
SEEK_TABLE_INTEGRITY_SIZE = 9           # lib.rs:56
SEEKABLE_MAX_FRAME_SIZE = 0x40000000    # lib.rs:58

_ERR_NUMBER_CONVERSION = -1001
_ERR_OFFSET_OUT_OF_RANGE = -1002
_ERR_FRAME_INDEX_TOO_LARGE = -1003
_ERR_IO = -1004
_ERR_NO_DEVICE = -1005
_ERR_CUDA = -1007


class Error(Exception):
    """lib/src/error.rs: opaque error with kind predicates; zstd codes keep libzstd's numbering."""

    def __init__(self, rc: int, lib=None):
        self.rc = int(rc)
        lib = lib or _native.default_lib()
        name = lib.zk_error_name(self.rc)
        detail = ""
        if self.rc == _ERR_CUDA:
            msg = lib.zk_last_cuda_error()
            detail = f" [{msg.decode()}]" if msg else ""
        super().__init__(f"{name.decode() if name else 'error'}{detail}; code {self.rc}")

    def is_number_conversion_failed(self) -> bool: return self.rc == _ERR_NUMBER_CONVERSION
    def is_offset_out_of_range(self) -> bool: return self.rc == _ERR_OFFSET_OUT_OF_RANGE
    def is_frame_index_too_large(self) -> bool: return self.rc == _ERR_FRAME_INDEX_TOO_LARGE
    def is_io(self) -> bool: return self.rc == _ERR_IO
    def is_cuda(self) -> bool: return self.rc == _ERR_CUDA
    def is_zstd(self) -> bool: return -1000 < self.rc < 0
    def zstd_code(self) -> int: return -self.rc if self.is_zstd() else 0


def _check(rc: int, lib=None):
    if rc != 0:
        raise Error(rc, lib)


def _buf(b):
    """-> (address, length, keepalive) for bytes-like / numpy input"""
    if isinstance(b, np.ndarray):
        a = np.ascontiguousarray(b).view(np.uint8).reshape(-1)
        return a.ctypes.data, a.size, a
    a = np.frombuffer(b, dtype=np.uint8) if len(b) else np.zeros(0, dtype=np.uint8)
    return a.ctypes.data, a.size, (a, b)


class Format:
    """seek_table::Format (seek_table.rs:228-241)"""
    Head = 0
    Foot = 1


class FrameSizePolicy:
    """encode.rs:21-39"""
    COMPRESSED = 0
    UNCOMPRESSED = 1

    def __init__(self, kind: int, size: int):
        self.kind, self.size = kind, size

    @classmethod
    def Compressed(cls, size: int): return cls(cls.COMPRESSED, size)

    @classmethod
    def Uncompressed(cls, size: int): return cls(cls.UNCOMPRESSED, size)

    @classmethod
    def default(cls): return cls.Uncompressed(0x200000)


class CParameter:
    """Compression parameters of a Context, named as zstd-safe's CParameter (ZSTD_c_* values).  0 restores the default."""
    WINDOW_LOG = 101                      # ZK_C_WINDOW_LOG
    ENABLE_LONG_DISTANCE_MATCHING = 160   # ZK_C_ENABLE_LONG_DISTANCE_MATCHING

    def __init__(self, param: int, value: int):
        self.param, self.value = param, int(value)

    @classmethod
    def WindowLog(cls, log: int): return cls(cls.WINDOW_LOG, log)

    @classmethod
    def EnableLongDistanceMatching(cls, on: bool): return cls(cls.ENABLE_LONG_DISTANCE_MATCHING, int(bool(on)))


class DParameter:
    """Decompression parameters of a Context, named as zstd-safe's DParameter (ZSTD_d_* values).  0 restores the default."""
    WINDOW_LOG_MAX = 100                  # ZK_D_WINDOW_LOG_MAX

    def __init__(self, param: int, value: int):
        self.param, self.value = param, int(value)

    @classmethod
    def WindowLogMax(cls, log: int): return cls(cls.WINDOW_LOG_MAX, log)


class Context:
    """Owns the CUDA streams / HBM scratch (the role CCtx / DCtx play in the reference)."""

    def __init__(self, device: int = 0, lib=None):
        self.lib = lib or _native.default_lib()
        h = c_void_p()
        _check(self.lib.zk_ctx_create(device, 0, byref(h)), self.lib)
        self._h = h
        self.cparams: dict[int, int] = {}     # values set so far (sticky, as on the native context)
        self.dparams: dict[int, int] = {}

    def set_cparameter(self, p: CParameter) -> "Context":
        """CCtx::set_parameter: applies to every later compress call on this context (window log 0 or 10..30, LDM 0/1)"""
        _check(self.lib.zk_ctx_set_cparameter(self._h, p.param, p.value), self.lib)
        self.cparams[p.param] = p.value
        return self

    def set_dparameter(self, p: DParameter) -> "Context":
        """DCtx::set_parameter: applies to every later decompress call on this context (window log max 0 or 10..30)"""
        _check(self.lib.zk_ctx_set_dparameter(self._h, p.param, p.value), self.lib)
        self.dparams[p.param] = p.value
        return self

    def close(self):
        if self._h:
            self.lib.zk_ctx_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    @property
    def kernel_launches(self) -> int: return int(self.lib.zk_ctx_kernel_launches(self._h))

    @property
    def last_device_ms(self) -> float: return float(self.lib.zk_ctx_last_device_ms(self._h))

    # ---- batch codec (the hot path) ------------------------------------------------------------
    def compress_frames(self, data, frame_size: int = 0x200000, level: int = 0, checksum: bool = False, prefix=None):
        """-> (compressed bytes (np.uint8), c_sizes, d_sizes).  Host buffers.  prefix: raw-content prefix of every frame."""
        addr, n, keep = _buf(data)
        lib = self.lib
        cap = lib.zk_compress_bound(n, frame_size)
        dst = np.empty(cap + 64, dtype=np.uint8)
        nfmax = n // max(frame_size, 1) + 2
        cs = np.zeros(nfmax, dtype=np.uint32); ds = np.zeros(nfmax, dtype=np.uint32)
        nf = c_uint32(); dl = c_size_t()
        if prefix is not None:
            paddr, pn, pkeep = _buf(prefix)
            _check(lib.zk_compress_frames_prefix(self._h, addr, n, frame_size, level, int(checksum), paddr, pn, dst.ctypes.data, cap,
                                                 cs.ctypes.data_as(_native.u32p), ds.ctypes.data_as(_native.u32p), nfmax, byref(nf), byref(dl)), lib)
        else:
            _check(lib.zk_compress_frames(self._h, addr, n, frame_size, level, int(checksum), dst.ctypes.data, cap,
                                          cs.ctypes.data_as(_native.u32p), ds.ctypes.data_as(_native.u32p), nfmax, byref(nf),
                                          byref(dl)), lib)
        return dst[: dl.value], cs[: nf.value].copy(), ds[: nf.value].copy()

    def decompress_frames(self, comp, c_off, d_off, verify_checksum: bool = True, out: np.ndarray | None = None, need=None, prefix=None):
        """decode frames given N+1 cumulative offsets -> (np.uint8 output, per-frame status, rc).
        need (optional, one uint32 per frame): only that many leading bytes of each frame are wanted (range reads,
        zk_decompress_frames_upto): the rest of a frame's output range is then unspecified and its checksum is not verified."""
        addr, n, keep = _buf(comp)
        co = np.ascontiguousarray(c_off, dtype=np.uint64); do = np.ascontiguousarray(d_off, dtype=np.uint64)
        nf = len(co) - 1
        total = int(do[-1])
        if out is None:
            out = np.empty(total + 64, dtype=np.uint8)
        elif not (isinstance(out, np.ndarray) and out.dtype == np.uint8 and out.flags["C_CONTIGUOUS"] and out.size >= total):
            raise ValueError(f"out: need a C-contiguous np.uint8 array of at least {total} bytes")
        st = np.zeros(max(nf, 1), dtype=np.int32)
        nd = None if need is None else np.ascontiguousarray(need, dtype=np.uint32)
        if nd is not None and len(nd) != nf:
            raise ValueError("need: one entry per frame")
        paddr, pn, pkeep = _buf(prefix) if prefix is not None else (None, 0, None)
        rc = self.lib.zk_decompress_frames_prefix(self._h, addr, co.ctypes.data_as(_native.u64p), do.ctypes.data_as(_native.u64p), nf,
                                                  out.ctypes.data, None if nd is None else nd.ctypes.data_as(_native.u32p),
                                                  int(verify_checksum), st.ctypes.data_as(_native.i32p), paddr, pn)
        return out[:total], st[:nf], rc


_default_ctx: Context | None = None


def default_context() -> Context:
    global _default_ctx
    if _default_ctx is None:
        _default_ctx = Context(0)
    return _default_ctx


def set_default_context(ctx: Context | None) -> None:
    global _default_ctx
    _default_ctx = ctx


# ---------------------------------------------------------------------------------------------- SeekTable
class SeekTable:
    """lib/src/seek_table.rs:267-935"""

    def __init__(self, _h=None, _owned=True, lib=None, _keep=None):
        self.lib = lib or _native.default_lib()
        self._h = _h if _h is not None else c_void_p(self.lib.zk_seek_table_new())
        self._owned = _owned
        self._keep = _keep

    def __del__(self):
        try:
            if self._owned and self._h:
                self.lib.zk_seek_table_free(self._h)
        except Exception:
            pass

    @classmethod
    def from_bytes(cls, buf, format: int = Format.Foot, lib=None):
        """SeekTable::from_seekable_format(&mut BytesWrapper::new(buf), format), :379-436"""
        lib = lib or _native.default_lib()
        addr, n, keep = _buf(buf)
        h = c_void_p()
        _check(lib.zk_seek_table_from_bytes(addr, n, format, byref(h)), lib)
        return cls(h, True, lib)

    from_seekable = from_bytes

    @classmethod
    def from_reader(cls, reader, lib=None):
        """stand-alone Head-format seek table, :461-493"""
        return cls.from_bytes(reader.read(), Format.Head, lib)

    def clone(self): return SeekTable(c_void_p(self.lib.zk_seek_table_clone(self._h)), True, self.lib)
    def log_frame(self, c_size: int, d_size: int): _check(self.lib.zk_seek_table_log_frame(self._h, c_size, d_size), self.lib)
    def num_frames(self) -> int: return int(self.lib.zk_seek_table_num_frames(self._h))
    def frame_index_comp(self, off: int) -> int: return int(self.lib.zk_seek_table_frame_index_comp(self._h, off))
    def frame_index_decomp(self, off: int) -> int: return int(self.lib.zk_seek_table_frame_index_decomp(self._h, off))

    def _get(self, fn, index):
        v = c_uint64()
        _check(fn(self._h, index, byref(v)), self.lib)
        return int(v.value)

    def frame_start_comp(self, i): return self._get(self.lib.zk_seek_table_frame_start_comp, i)
    def frame_start_decomp(self, i): return self._get(self.lib.zk_seek_table_frame_start_decomp, i)
    def frame_end_comp(self, i): return self._get(self.lib.zk_seek_table_frame_end_comp, i)
    def frame_end_decomp(self, i): return self._get(self.lib.zk_seek_table_frame_end_decomp, i)
    def frame_size_comp(self, i): return self._get(self.lib.zk_seek_table_frame_size_comp, i)
    def frame_size_decomp(self, i): return self._get(self.lib.zk_seek_table_frame_size_decomp, i)
    def max_frame_size_comp(self): return int(self.lib.zk_seek_table_max_frame_size_comp(self._h))
    def max_frame_size_decomp(self): return int(self.lib.zk_seek_table_max_frame_size_decomp(self._h))
    def size_comp(self): return int(self.lib.zk_seek_table_size_comp(self._h))
    def size_decomp(self): return int(self.lib.zk_seek_table_size_decomp(self._h))

    def offsets(self):
        n = self.num_frames() + 1
        c = np.zeros(n, dtype=np.uint64); d = np.zeros(n, dtype=np.uint64)
        self.lib.zk_seek_table_offsets(self._h, c.ctypes.data_as(_native.u64p), d.ctypes.data_as(_native.u64p), n)
        return c, d

    def into_serializer(self): return self.into_format_serializer(Format.Foot)
    def into_format_serializer(self, format: int): return Serializer(c_void_p(self.lib.zk_seek_table_into_serializer(self._h, format)), self.lib)

    def __eq__(self, other):
        a, b = self.offsets(), other.offsets()
        return a[0].tolist() == b[0].tolist() and a[1].tolist() == b[1].tolist()


class Serializer(io.RawIOBase):
    """seek_table.rs:955-1059 (resumable; also readable like `impl Read`)"""

    def __init__(self, h, lib):
        super().__init__()
        self._h, self.lib = h, lib

    def __del__(self):
        try:
            if self._h:
                self.lib.zk_serializer_free(self._h)
        except Exception:
            pass

    def write_into(self, buf) -> int:
        mv = memoryview(buf)
        if len(mv) == 0:
            return 0
        arr = (ctypes.c_uint8 * len(mv)).from_buffer(mv)
        return int(self.lib.zk_serializer_write_into(self._h, arr, len(mv)))

    def reset(self): self.lib.zk_serializer_reset(self._h)
    def encoded_len(self) -> int: return int(self.lib.zk_serializer_encoded_len(self._h))
    def readable(self): return True
    def readinto(self, b): return self.write_into(b)

    def to_bytes(self) -> bytes:
        out = bytearray(self.encoded_len())
        n = self.write_into(out)
        return bytes(out[:n])


# ---------------------------------------------------------------------------------------------- encode
class EncodeOptions:
    """encode.rs:110-207 (builder)"""

    def __init__(self, ctx: Context | None = None):
        self.ctx = ctx or default_context()
        self._policy = FrameSizePolicy.default()
        self._checksum = False
        self._level = 0

    def frame_size_policy(self, policy: FrameSizePolicy): self._policy = policy; return self
    def checksum_flag(self, flag: bool): self._checksum = bool(flag); return self
    def compression_level(self, level: int): self._level = int(level); return self

    def _native_opts(self):
        lib = self.ctx.lib
        o = c_void_p(lib.zk_encode_options_new(self.ctx._h))
        lib.zk_encode_options_frame_size_policy(o, self._policy.kind, self._policy.size)
        lib.zk_encode_options_checksum_flag(o, int(self._checksum))
        lib.zk_encode_options_compression_level(o, self._level)
        return o

    def into_raw_encoder(self): return RawEncoder(self)
    def into_encoder(self, writer): return Encoder(writer, self)


class RawEncoder:
    """encode.rs:266-545"""

    def __init__(self, opts: EncodeOptions | None = None):
        opts = opts or EncodeOptions()
        self.ctx, self.lib = opts.ctx, opts.ctx.lib
        h = c_void_p()
        _check(self.lib.zk_encode_options_into_raw_encoder(opts._native_opts(), byref(h)), self.lib)
        self._h = h

    def __del__(self):
        try:
            if self._h:
                self.lib.zk_raw_encoder_free(self._h)
        except Exception:
            pass

    def compress(self, input, output) -> CompressionProgress:
        """-> progress with .in_progress / .out_progress (encode.rs:398)"""
        addr, n, keep = _buf(input)
        mv = memoryview(output)
        oarr = (ctypes.c_uint8 * len(mv)).from_buffer(mv) if len(mv) else None
        p = CompressionProgress()
        _check(self.lib.zk_raw_encoder_compress(self._h, addr, n, oarr, len(mv), byref(p)), self.lib)
        return p

    def compress_with_prefix(self, input, output, prefix=None) -> CompressionProgress:
        """encode.rs:311-354: `prefix` (bytes-like, or None) becomes the raw-content prefix of a frame when passed on the
        frame's first call; the caller keeps it alive until the frame is closed"""
        if prefix is None:
            return self.compress(input, output)
        addr, n, keep = _buf(input)
        paddr, pn, pkeep = _buf(prefix)
        self._prefix_keep = pkeep
        mv = memoryview(output)
        oarr = (ctypes.c_uint8 * len(mv)).from_buffer(mv) if len(mv) else None
        p = CompressionProgress()
        _check(self.lib.zk_raw_encoder_compress_with_prefix(self._h, addr, n, oarr, len(mv), paddr, pn, byref(p)), self.lib)
        return p

    def end_frame(self, output) -> EpilogueProgress:
        mv = memoryview(output)
        oarr = (ctypes.c_uint8 * len(mv)).from_buffer(mv) if len(mv) else None
        p = EpilogueProgress()
        _check(self.lib.zk_raw_encoder_end_frame(self._h, oarr, len(mv), byref(p)), self.lib)
        return p

    def seek_table(self) -> SeekTable:
        return SeekTable(c_void_p(self.lib.zk_raw_encoder_seek_table(self._h)), False, self.lib, _keep=self)

    def into_seek_table(self) -> SeekTable:
        h = c_void_p(self.lib.zk_raw_encoder_into_seek_table(self._h))
        self._h = None
        return SeekTable(h, True, self.lib)

    def reset_frame(self): self.lib.zk_raw_encoder_reset_frame(self._h)
    def reset_seek_table(self): self.lib.zk_raw_encoder_reset_seek_table(self._h)


class Encoder(io.RawIOBase):
    """encode.rs:568-800: compresses into any object with .write(bytes) (W: std::io::Write)"""

    def __init__(self, writer, opts: EncodeOptions | None = None):
        super().__init__()
        opts = opts or EncodeOptions()
        self.ctx, self.lib = opts.ctx, opts.ctx.lib
        self._writer = writer

        def _write(user, data, n):
            try:
                writer.write(ctypes.string_at(data, n))
                return 0
            except Exception:
                return -1

        def _flush(user):
            try:
                if hasattr(writer, "flush"):
                    writer.flush()
                return 0
            except Exception:
                return -1

        self._wcb = _native.WRITE_FN(_write)
        self._fcb = _native.FLUSH_FN(_flush)
        h = c_void_p()
        _check(self.lib.zk_encode_options_into_encoder(opts._native_opts(), self._wcb, self._fcb, None, byref(h)), self.lib)
        self._h = h

    def __del__(self):
        try:
            if self._h:
                self.lib.zk_encoder_free(self._h)
        except Exception:
            pass

    def compress(self, buf) -> int:
        addr, n, keep = _buf(buf)
        c = c_size_t()
        _check(self.lib.zk_encoder_compress(self._h, addr, n, byref(c)), self.lib)
        return int(c.value)

    def compress_with_prefix(self, buf, prefix=None) -> int:
        """encode.rs:641-665"""
        if prefix is None:
            return self.compress(buf)
        addr, n, keep = _buf(buf)
        paddr, pn, pkeep = _buf(prefix)
        self._prefix_keep = pkeep
        c = c_size_t()
        _check(self.lib.zk_encoder_compress_with_prefix(self._h, addr, n, paddr, pn, byref(c)), self.lib)
        return int(c.value)

    def writable(self): return True
    def write(self, b): return self.compress(b)

    def end_frame(self) -> int:
        w = c_size_t()
        _check(self.lib.zk_encoder_end_frame(self._h, byref(w)), self.lib)
        return int(w.value)

    def flush(self):
        if getattr(self, "_h", None):
            _check(self.lib.zk_encoder_flush(self._h), self.lib)

    def finish(self) -> int: return self.finish_format(Format.Foot)

    def finish_format(self, format: int) -> int:
        t = c_uint64()
        h, self._h = self._h, None
        _check(self.lib.zk_encoder_finish_format(h, format, byref(t)), self.lib)
        return int(t.value)

    def written_compressed(self) -> int: return int(self.lib.zk_encoder_written_compressed(self._h))
    def seek_table(self) -> SeekTable: return SeekTable(c_void_p(self.lib.zk_encoder_seek_table(self._h)), False, self.lib, _keep=self)


# ---------------------------------------------------------------------------------------------- decode
class OffsetFrom:
    """seekable.rs:8-13"""
    START = 0
    END = 1


class BytesWrapper:
    """seekable.rs:43-97: a seekable view over bytes"""

    def __init__(self, src):
        self.src = src


class DecodeOptions:
    """decode.rs:13-114 (builder).  src: BytesWrapper / bytes-like, or a file-like object with read+seek."""

    def __init__(self, src, ctx: Context | None = None):
        self.ctx = ctx or default_context()
        self.src = src
        self._seek_table = None
        self._lower = self._upper = self._offset = self._limit = None

    def seek_table(self, st: SeekTable): self._seek_table = st; return self
    def lower_frame(self, i: int): self._lower = i; return self
    def upper_frame(self, i: int): self._upper = i; return self
    def offset(self, v: int): self._offset = v; return self
    def offset_limit(self, v: int): self._limit = v; return self
    def into_decoder(self): return Decoder(self)


class Decoder(io.RawIOBase):
    """decode.rs:121-579 (incl. impl Read / impl Seek)"""

    def __init__(self, src_or_opts):
        super().__init__()
        opts = src_or_opts if isinstance(src_or_opts, DecodeOptions) else DecodeOptions(src_or_opts)
        self.ctx, self.lib = opts.ctx, opts.ctx.lib
        lib = self.lib
        src = opts.src
        self._keep = None
        if isinstance(src, BytesWrapper):
            src = src.src
        if isinstance(src, (bytes, bytearray, memoryview, np.ndarray)):
            addr, n, keep = _buf(src)
            self._keep = keep
            o = c_void_p(lib.zk_decode_options_new_bytes(self.ctx._h, addr, n))
        else:
            f = src

            def _set_offset(user, whence, off):
                try:
                    return f.seek(off, 0 if whence == 0 else 2)
                except Exception:
                    return -1

            def _read(user, buf, n):
                try:
                    data = f.read(n)
                    ctypes.memmove(buf, data, len(data))
                    return len(data)
                except Exception:
                    return -1

            self._cbs = (_native.SET_OFFSET_FN(_set_offset), _native.READ_FN(_read))
            sk = _native.Seekable(None, self._cbs[0], self._cbs[1])
            o = c_void_p(lib.zk_decode_options_new_seekable(self.ctx._h, sk))
            self._keep = f
        if opts._seek_table is not None: lib.zk_decode_options_seek_table(o, opts._seek_table._h)
        if opts._lower is not None: lib.zk_decode_options_lower_frame(o, opts._lower)
        if opts._upper is not None: lib.zk_decode_options_upper_frame(o, opts._upper)
        if opts._offset is not None: lib.zk_decode_options_offset(o, opts._offset)
        if opts._limit is not None: lib.zk_decode_options_offset_limit(o, opts._limit)
        h = c_void_p()
        _check(lib.zk_decode_options_into_decoder(o, byref(h)), lib)
        self._h = h

    def __del__(self):
        try:
            if self._h:
                self.lib.zk_decoder_free(self._h)
        except Exception:
            pass

    def decompress(self, buf) -> int:
        mv = memoryview(buf)
        if len(mv) == 0:
            return 0
        arr = (ctypes.c_uint8 * len(mv)).from_buffer(mv)
        p = c_size_t()
        _check(self.lib.zk_decoder_decompress(self._h, arr, len(mv), byref(p)), self.lib)
        return int(p.value)

    def decompress_with_prefix(self, buf, prefix=None) -> int:
        """decode.rs:201-270: every frame is decoded against the raw-content prefix"""
        if prefix is None:
            return self.decompress(buf)
        mv = memoryview(buf)
        if len(mv) == 0:
            return 0
        arr = (ctypes.c_uint8 * len(mv)).from_buffer(mv)
        paddr, pn, pkeep = _buf(prefix)
        self._prefix_keep = pkeep
        p = c_size_t()
        _check(self.lib.zk_decoder_decompress_with_prefix(self._h, arr, len(mv), paddr, pn, byref(p)), self.lib)
        return int(p.value)

    def readable(self): return True
    def seekable(self): return True
    def readinto(self, b): return self.decompress(b)

    def read_all(self) -> bytes:
        out = bytearray(self.offset_limit() - self.offset())
        n = 0
        while n < len(out):
            k = self.decompress(memoryview(out)[n:])
            if k == 0:
                break
            n += k
        return bytes(out[:n])

    def reset(self): self.lib.zk_decoder_reset(self._h)

    def set_lower_frame(self, i: int) -> int:
        v = c_uint64(); _check(self.lib.zk_decoder_set_lower_frame(self._h, i, byref(v)), self.lib); return int(v.value)

    def set_upper_frame(self, i: int) -> int:
        v = c_uint64(); _check(self.lib.zk_decoder_set_upper_frame(self._h, i, byref(v)), self.lib); return int(v.value)

    def set_offset(self, off: int): _check(self.lib.zk_decoder_set_offset(self._h, off), self.lib)
    def set_offset_limit(self, lim: int): _check(self.lib.zk_decoder_set_offset_limit(self._h, lim), self.lib)
    def read_compressed(self) -> int: return int(self.lib.zk_decoder_read_compressed(self._h))
    def offset(self) -> int: return int(self.lib.zk_decoder_offset(self._h))
    def offset_limit(self) -> int: return int(self.lib.zk_decoder_offset_limit(self._h))
    def seek_table(self) -> SeekTable: return SeekTable(c_void_p(self.lib.zk_decoder_seek_table(self._h)), False, self.lib, _keep=self)

    def seek(self, pos: int, whence: int = 0) -> int:
        """impl Seek (decode.rs:545-579): whence 0 Start, 1 Current, 2 End (Python convention)"""
        v = c_uint64()
        native_whence = {0: 0, 1: 2, 2: 1}[whence]
        _check(self.lib.zk_decoder_seek(self._h, native_whence, pos, byref(v)), self.lib)
        return int(v.value)


__all__ = ["Context", "CParameter", "DParameter", "default_context", "set_default_context", "Error", "Format", "FrameSizePolicy", "SeekTable", "Serializer",
           "EncodeOptions", "RawEncoder", "Encoder", "CompressionProgress", "EpilogueProgress", "DecodeOptions", "Decoder",
           "BytesWrapper", "OffsetFrom", "SEEKABLE_MAGIC_NUMBER", "SEEKABLE_MAX_FRAMES", "SEEK_TABLE_INTEGRITY_SIZE",
           "SEEKABLE_MAX_FRAME_SIZE"]
