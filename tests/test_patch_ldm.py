"""Patch mode with long-distance matching: the context parameters ZK_C_WINDOW_LOG, ZK_C_ENABLE_LONG_DISTANCE_MATCHING and
ZK_D_WINDOW_LOG_MAX (what the reference's CLI sets for `--patch-from` / `--patch-apply`, cli/src/compress.rs:31-37,
cli/src/decompress.rs:53-62).

The first part runs on the CPU emulation build (`emul_lib`) at emulator sizes, the second on the B200 (`gpu_lib`) at full size.
libzstd is driven directly through ctypes here, because these calls need its advanced parameters (ZSTD_CCtx_setParameter /
ZSTD_DCtx_setParameter), which the oracle's driver does not take.
"""
from __future__ import annotations

import ctypes
import hashlib
import json
import os

import numpy as np
import pytest

import zeekstd_b200 as zk
from oracle import oracle as O
from util import golden_bytes, make_ctx

GOLDEN_LDM = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "ldm_golden.json")


# ----------------------------------------------------------------------------- libzstd with parameters
class _InBuf(ctypes.Structure):
    _fields_ = [("src", ctypes.c_void_p), ("size", ctypes.c_size_t), ("pos", ctypes.c_size_t)]


class _OutBuf(ctypes.Structure):
    _fields_ = [("dst", ctypes.c_void_p), ("size", ctypes.c_size_t), ("pos", ctypes.c_size_t)]


_ZSTD = None
_c_compressionLevel, _c_windowLog, _c_checksumFlag, _c_enableLDM, _d_windowLogMax = 100, 101, 201, 160, 100


def _zstd():
    global _ZSTD
    if _ZSTD is None:
        z = ctypes.CDLL(os.environ.get("ZK_LIBZSTD", O.SYSTEM_LIBZSTD))
        vp, sz = ctypes.c_void_p, ctypes.c_size_t
        for name, res, args in (("ZSTD_createCCtx", vp, []), ("ZSTD_freeCCtx", sz, [vp]), ("ZSTD_createDCtx", vp, []), ("ZSTD_freeDCtx", sz, [vp]),
                                ("ZSTD_CCtx_setParameter", sz, [vp, ctypes.c_int, ctypes.c_int]), ("ZSTD_CCtx_refPrefix", sz, [vp, vp, sz]),
                                ("ZSTD_CCtx_reset", sz, [vp, ctypes.c_int]), ("ZSTD_compress2", sz, [vp, vp, sz, vp, sz]),
                                ("ZSTD_DCtx_setParameter", sz, [vp, ctypes.c_int, ctypes.c_int]), ("ZSTD_DCtx_refPrefix", sz, [vp, vp, sz]),
                                ("ZSTD_DCtx_reset", sz, [vp, ctypes.c_int]),
                                ("ZSTD_decompressStream", sz, [vp, ctypes.POINTER(_OutBuf), ctypes.POINTER(_InBuf)]),
                                ("ZSTD_compressBound", sz, [sz]), ("ZSTD_isError", ctypes.c_uint, [sz]), ("ZSTD_getErrorCode", ctypes.c_int, [sz])):
            f = getattr(z, name); f.restype = res; f.argtypes = args
        _ZSTD = z
    return _ZSTD


def _u8(b) -> np.ndarray:
    return b if isinstance(b, np.ndarray) else np.frombuffer(bytes(b), dtype=np.uint8)


def zstd_compress(data, frame_size: int, level: int, prefix=None, window_log: int = 0, ldm: bool = False, checksum: bool = True):
    """libzstd, one frame per frame_size bytes, the prefix referenced at every frame start -> (frames, d_sizes)"""
    z = _zstd(); src = _u8(data); pf = None if prefix is None else _u8(prefix)
    cc = z.ZSTD_createCCtx()
    try:
        for p, v in ((_c_compressionLevel, level), (_c_checksumFlag, int(checksum)), (_c_windowLog, window_log), (_c_enableLDM, int(ldm))):
            assert not z.ZSTD_isError(z.ZSTD_CCtx_setParameter(cc, p, v))
        frames, ds = [], []
        for lo in range(0, src.size, frame_size):
            part = src[lo: lo + frame_size]
            if pf is not None:
                assert not z.ZSTD_isError(z.ZSTD_CCtx_refPrefix(cc, pf.ctypes.data, pf.size))
            out = np.empty(z.ZSTD_compressBound(part.size) + 64, dtype=np.uint8)
            r = z.ZSTD_compress2(cc, out.ctypes.data, out.size, part.ctypes.data, part.size)
            assert not z.ZSTD_isError(r), z.ZSTD_getErrorCode(r)
            frames.append(out[:r].tobytes()); ds.append(part.size)
        return frames, ds
    finally:
        z.ZSTD_freeCCtx(cc)


def zstd_decompress(frames, d_sizes, prefix=None, window_log_max: int = 0) -> bytes:
    """libzstd streaming decompression (what the reference's Decoder runs), the prefix re-referenced for every frame; raises
    O.ZstdError(code) on an error"""
    z = _zstd(); pf = None if prefix is None else _u8(prefix)
    dc = z.ZSTD_createDCtx()
    try:
        assert not z.ZSTD_isError(z.ZSTD_DCtx_setParameter(dc, _d_windowLogMax, window_log_max))
        res = []
        for fr, d in zip(frames, d_sizes):
            z.ZSTD_DCtx_reset(dc, 1)
            if pf is not None:
                assert not z.ZSTD_isError(z.ZSTD_DCtx_refPrefix(dc, pf.ctypes.data, pf.size))
            src = np.frombuffer(fr, dtype=np.uint8); out = np.empty(max(int(d), 1), dtype=np.uint8)
            ib = _InBuf(src.ctypes.data, src.size, 0); ob = _OutBuf(out.ctypes.data, int(d), 0)
            while True:
                r = z.ZSTD_decompressStream(dc, ctypes.byref(ob), ctypes.byref(ib))
                if z.ZSTD_isError(r):
                    raise O.ZstdError(z.ZSTD_getErrorCode(r))
                if r == 0 or (ib.pos == ib.size and ob.pos == ob.size):
                    break
            assert r == 0 and ob.pos == int(d), (r, ob.pos, d)
            res.append(out[: ob.pos].tobytes())
        return b"".join(res)
    finally:
        z.ZSTD_freeDCtx(dc)


# ----------------------------------------------------------------------------- inputs
def patch_pair(old: np.ndarray, seed: int, edits: int = 40, moved: int = 4096):
    """NEW = OLD rotated by half its length, with `edits` random inserts / deletes / overwrites of 1-64 bytes and one moved range:
    the useful matches lie about half of OLD back, far beyond the 64 KiB reach of the kernels without long-distance matching"""
    rng = np.random.default_rng(seed)
    n = old.size
    new = np.concatenate([old[n // 2:], old[: n // 2]])
    pieces, pos = [], 0
    for at in np.sort(rng.integers(0, n - 64, edits)):
        at = int(at)
        if at < pos:
            continue
        pieces.append(new[pos:at]); k = int(rng.integers(0, 3)); ln = int(rng.integers(1, 65))
        rnd = rng.integers(0, 256, ln, dtype=np.uint8)
        if k == 0:
            pieces.append(rnd); pos = at                 # insert
        elif k == 1:
            pos = at + ln                                # delete
        else:
            pieces.append(rnd); pos = at + ln            # overwrite
    pieces.append(new[pos:])
    new = np.concatenate(pieces)
    a = int(rng.integers(0, new.size // 2)); seg = new[a: a + moved].copy()
    new = np.concatenate([new[:a], new[a + moved:]])
    b = int(rng.integers(0, new.size))
    return np.concatenate([new[:b], seg, new[b:]])


def small_old(n: int = 256 << 10, seed: int = 3) -> np.ndarray:
    text = np.frombuffer(golden_bytes("dickens.txt"), dtype=np.uint8)
    s = int(np.random.default_rng(seed).integers(0, text.size - n))
    return text[s: s + n].copy()


def patch_window_log(n: int) -> int:
    return min(30, max(17, n.bit_length()))


def split(comp: np.ndarray, cs):
    out, pos = [], 0
    for c in cs:
        out.append(comp[pos: pos + int(c)].tobytes()); pos += int(c)
    return out


def restated(frames, ds, prefix):
    """the restated decoder, frame by frame -> (bytes, largest offset).  It keeps the default window limit, so a frame announcing
    more than 2^27 is handed over with its Window_Descriptor lowered to 2^27: nothing else of the frame depends on the descriptor
    (blocks stay at most 128 KiB) and the restatement does not bound offsets by the window"""
    out, mo = [], 0
    for fr, d in zip(frames, ds):
        fr = bytearray(fr)
        if not fr[4] & 0x20 and fr[5] > 0x88:
            fr[5] = 0x88
        o, st = O.oracle_decompress_ex(bytes(fr), int(d), prefix=prefix)
        out.append(o); mo = max(mo, st["max_offset"])
    return b"".join(out), mo


def window_of(frame: bytes) -> int:
    wd = frame[5]
    return (1 << (10 + (wd >> 3))) + ((1 << (10 + (wd >> 3))) >> 3) * (wd & 7)


def ldm_compress(ctx, new, old, frame_size, level, window_log, checksum=True):
    ctx.set_cparameter(zk.CParameter.WindowLog(window_log)).set_cparameter(zk.CParameter.EnableLongDistanceMatching(True))
    try:
        return ctx.compress_frames(new, frame_size, level, checksum, prefix=old)
    finally:
        ctx.set_cparameter(zk.CParameter.WindowLog(0)).set_cparameter(zk.CParameter.EnableLongDistanceMatching(False))


def ours_decompress(ctx, frames, ds, prefix=None, window_log_max=0):
    comp = np.frombuffer(b"".join(frames) + b"\0" * 64, dtype=np.uint8)
    co = np.concatenate([[0], np.cumsum([len(f) for f in frames])]).astype(np.uint64)
    do = np.concatenate([[0], np.cumsum(ds)]).astype(np.uint64)
    ctx.set_dparameter(zk.DParameter.WindowLogMax(window_log_max))
    try:
        out, st, rc = ctx.decompress_frames(comp, co, do, True, prefix=prefix)
    finally:
        ctx.set_dparameter(zk.DParameter.WindowLogMax(0))
    return out.tobytes(), st, rc


def check_ldm_patch(ctx, old, new, frame_size, level, checksum=True):
    """our LDM patch: libzstd and this decoder restore it; offsets reach past 64 KiB and stay within the announced window"""
    wl = patch_window_log(old.size)
    comp, cs, ds = ldm_compress(ctx, new, old, frame_size, level, wl, checksum)
    frames = split(comp, cs)
    assert all(f[5] == (wl - 10) << 3 for f in frames), [hex(f[5]) for f in frames[:3]]
    assert zstd_decompress(frames, ds, prefix=old, window_log_max=wl) == new.tobytes()
    back, st, rc = ours_decompress(ctx, frames, ds, prefix=old, window_log_max=wl)
    assert rc == 0 and not st.any() and back == new.tobytes(), (rc, st[:4])
    return comp.size, frames, ds


# ============================================================================= CPU (emulation build)
@pytest.fixture(scope="module")
def ectx(emul_lib):
    return make_ctx(emul_lib)


@pytest.fixture(scope="module")
def pair():
    old = small_old()
    return old, patch_pair(old, seed=11)


def test_parameter_api(ectx):
    lib = ectx.lib
    for p in (zk.CParameter.WINDOW_LOG, zk.CParameter.ENABLE_LONG_DISTANCE_MATCHING):
        assert lib.zk_ctx_set_cparameter(ectx._h, p, 0) == 0
    assert lib.zk_ctx_set_dparameter(ectx._h, zk.DParameter.WINDOW_LOG_MAX, 0) == 0
    assert lib.zk_ctx_set_cparameter(ectx._h, 999, 1) == -40 and lib.zk_ctx_set_dparameter(ectx._h, 101, 20) == -40
    for bad in (1, 9, 31, -1):
        assert lib.zk_ctx_set_cparameter(ectx._h, zk.CParameter.WINDOW_LOG, bad) == -42
        assert lib.zk_ctx_set_dparameter(ectx._h, zk.DParameter.WINDOW_LOG_MAX, bad) == -42
    assert lib.zk_ctx_set_cparameter(ectx._h, zk.CParameter.ENABLE_LONG_DISTANCE_MATCHING, 2) == -42
    for ok in (10, 30):
        assert lib.zk_ctx_set_cparameter(ectx._h, zk.CParameter.WINDOW_LOG, ok) == 0
        assert lib.zk_ctx_set_dparameter(ectx._h, zk.DParameter.WINDOW_LOG_MAX, ok) == 0
    with pytest.raises(zk.Error) as e:
        ectx.set_cparameter(zk.CParameter.WindowLog(31))
    assert e.value.zstd_code() == 42
    # back to the defaults: the prefix-mode golden bytes of the encoder are reproduced
    ectx.set_cparameter(zk.CParameter.WindowLog(0)).set_cparameter(zk.CParameter.EnableLongDistanceMatching(False))
    ectx.set_dparameter(zk.DParameter.WindowLogMax(0))
    d = np.frombuffer(golden_bytes("dickens_96k.txt"), dtype=np.uint8)
    comp, _, _ = ectx.compress_frames(d[20_000:], 40_000, 3, True, prefix=d[:30_000])
    g = json.load(open(os.path.join(os.path.dirname(GOLDEN_LDM), "encoder_golden.json")))["3+prefix"]
    assert comp.size == g["size"] and hashlib.sha256(comp.tobytes()).hexdigest() == g["sha256"]


def test_ldm_without_prefix_is_a_noop(ectx):
    d = np.frombuffer(golden_bytes("dickens_96k.txt"), dtype=np.uint8)
    plain, _, _ = ectx.compress_frames(d, 40_000, 3, True)
    ectx.set_cparameter(zk.CParameter.EnableLongDistanceMatching(True))
    try:
        ldm, _, _ = ectx.compress_frames(d, 40_000, 3, True)
    finally:
        ectx.set_cparameter(zk.CParameter.EnableLongDistanceMatching(False))
    assert ldm.tobytes() == plain.tobytes()
    # a raised window log alone only changes the Window_Descriptor
    ectx.set_cparameter(zk.CParameter.WindowLog(22))
    try:
        wide, cs, ds = ectx.compress_frames(d, 40_000, 3, True)
    finally:
        ectx.set_cparameter(zk.CParameter.WindowLog(0))
    frames = split(wide, cs)
    assert all(f[5] == (22 - 10) << 3 for f in frames)
    assert b"".join(bytes(f[:5]) + bytes([0x38]) + bytes(f[6:]) for f in frames) == plain.tobytes()
    assert zstd_decompress(frames, ds) == d.tobytes()


@pytest.mark.parametrize("level", [1, 3, 4, 13])
@pytest.mark.parametrize("frame_size", [64 << 10, 160 << 10, 1 << 20])
def test_ldm_patch(ectx, pair, level, frame_size):
    old, new = pair
    size, frames, ds = check_ldm_patch(ectx, old, new, frame_size, level)
    back, max_off = restated(frames, ds, old)
    assert back == new.tobytes()
    assert (64 << 10) < max_off <= window_of(frames[0]), max_off
    plain, _, _ = ectx.compress_frames(new, frame_size, level, True, prefix=old)
    assert size * 10 <= plain.size, (size, plain.size)
    if level == 3:
        ref, _ = zstd_compress(new, frame_size, 3, prefix=old, window_log=patch_window_log(old.size), ldm=True)
        assert size <= 2 * sum(len(f) for f in ref), (size, sum(len(f) for f in ref))


@pytest.mark.parametrize("level", [1, 3])
def test_window_smaller_than_prefix(ectx, pair, level):
    old, new = pair
    comp, cs, ds = ldm_compress(ectx, new, old, 1 << 20, level, 17)
    frames = split(comp, cs)
    assert frames[0][5] == 0x38
    back, max_off = restated(frames, ds, old)
    assert back == new.tobytes() and max_off <= 1 << 17, max_off
    assert zstd_decompress(frames, ds, prefix=old, window_log_max=17) == new.tobytes()


def test_libzstd_ldm_patch_decodes_here(ectx, pair):
    old, new = pair
    frames, ds = zstd_compress(new, 96 << 10, 3, prefix=old, window_log=patch_window_log(old.size), ldm=True)
    back, st, rc = ours_decompress(ectx, frames, ds, prefix=old)
    assert rc == 0 and back == new.tobytes()


def test_window_log_max(ectx):
    body = (len(b"hello") << 3 | 1).to_bytes(3, "little") + b"hello"
    fr = b"\x28\xb5\x2f\xfd\x00" + bytes([0x90]) + body             # Window_Descriptor 2^28
    for wlm, code in ((0, 16), (27, 16), (28, 0), (30, 0)):
        try:
            assert zstd_decompress([fr], [5], window_log_max=wlm) == b"hello"
            ref = 0
        except O.ZstdError as e:
            ref = e.code
        got, st, rc = ours_decompress(ectx, [fr], [5], window_log_max=wlm)
        assert ref == code and rc == -code and (code or got == b"hello"), (wlm, ref, rc)
    # the limit is exactly 2^L: 2^27 * 1.125 passes at 28, not at 27
    fr = b"\x28\xb5\x2f\xfd\x00" + bytes([0x89]) + body
    assert ours_decompress(ectx, [fr], [5], window_log_max=27)[2] == -16
    assert ours_decompress(ectx, [fr], [5], window_log_max=28)[2] == 0


def test_cli_patch(ectx, pair, tmp_path):
    from cases import _cli
    old, new = pair
    pf, nf = str(tmp_path / "old"), str(tmp_path / "new")
    open(pf, "wb").write(old.tobytes()); open(nf, "wb").write(new.tobytes())
    zp, zn = str(tmp_path / "patch.zst"), str(tmp_path / "full.zst")
    before = (dict(ectx.cparams), dict(ectx.dparams))
    assert _cli(ectx, ["compress", nf, "-o", zp, "--patch-from", pf, "-s", 128 << 10])[0] == 0
    rc, out, err = _cli(ectx, ["decompress", zp, "-c", "--patch-apply", pf])
    assert rc == 0 and out == new.tobytes(), err
    assert (dict(ectx.cparams), dict(ectx.dparams)) == before or all(v == 0 for v in {**ectx.cparams, **ectx.dparams}.values())
    # the same prefix call without long-distance matching
    plain, _, _ = ectx.compress_frames(new, 128 << 10, 3, True, prefix=old)
    assert os.path.getsize(zp) * 10 <= plain.size, (os.path.getsize(zp), plain.size)


def ldm_golden_cases():
    """(key, OLD, NEW, frame size, level, window log): the inputs of tests/golden/ldm_golden.json"""
    old = small_old(192 << 10, seed=5)
    new = patch_pair(old, seed=21)
    return [(f"{lvl}+ldm", old, new, 64 << 10, lvl, patch_window_log(old.size)) for lvl in (1, 3, 4, 7, 10, 13)] + \
           [("3+ldm+w17", old, new, 64 << 10, 3, 17)]


def ldm_golden(ctx) -> dict:
    out = {}
    for key, old, new, fs, lvl, wl in ldm_golden_cases():
        comp, _, _ = ldm_compress(ctx, new, old, fs, lvl, wl)
        out[key] = {"size": int(comp.size), "sha256": hashlib.sha256(comp.tobytes()).hexdigest()}
    return out


def test_ldm_golden_deterministic(emul_lib):
    import subprocess
    import sys
    want = json.load(open(GOLDEN_LDM))
    here = os.path.dirname(os.path.abspath(__file__))
    code = ("import json, sys; sys.path[:0] = [%r, %r]; from zeekstd_b200 import _native; from zeekstd_b200.build import build_emul; "
            "from util import make_ctx; import test_patch_ldm as t; print(json.dumps(t.ldm_golden(make_ctx(_native.load(build_emul())))))"
            % (os.path.dirname(here), here))
    for seed in ("1", "987654321"):
        r = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, env={**os.environ, "ZK_EMUL_SEED": seed})
        assert r.returncode == 0, r.stderr[-2000:]
        assert json.loads(r.stdout.strip().splitlines()[-1]) == want, seed


# ============================================================================= GPU (B200), full size
@pytest.fixture(scope="module")
def gctx(gpu_lib):
    return make_ctx(gpu_lib)


def big_old(n: int, seed: int) -> np.ndarray:
    from zeekstd_b200 import corpus
    return corpus.make_mix(n, seed=seed).numpy()


@pytest.fixture(scope="module")
def big_pair():
    old = big_old(256 << 20, seed=7)
    return old, patch_pair(old, seed=13)


@pytest.mark.gpu
@pytest.mark.parametrize("level", [1, 3, 13])
def test_gpu_ldm_patch_full_size(gctx, big_pair, level):
    old, new = big_pair
    size, frames, ds = check_ldm_patch(gctx, old, new, 2 << 20, level)
    plain, _, _ = gctx.compress_frames(new, 2 << 20, level, True, prefix=old)
    assert size * 10 <= plain.size, (size, plain.size)


@pytest.mark.gpu
def test_gpu_libzstd_ldm_patch_decodes_here(gctx, big_pair):
    old, new = big_pair
    wl = patch_window_log(old.size)
    frames, ds = zstd_compress(new[: 32 << 20], 2 << 20, 3, prefix=old, window_log=wl, ldm=True)
    back, st, rc = ours_decompress(gctx, frames, ds, prefix=old, window_log_max=wl)
    assert rc == 0 and back == new[: 32 << 20].tobytes()


@pytest.mark.gpu
def test_gpu_cli_patch_full_size(gctx, big_pair, tmp_path):
    from cases import _cli
    old, new = big_pair
    pf, nf, zp = str(tmp_path / "old"), str(tmp_path / "new"), str(tmp_path / "patch.zst")
    old.tofile(pf); new.tofile(nf)
    assert _cli(gctx, ["compress", nf, "-o", zp, "--patch-from", pf])[0] == 0
    rc, out, err = _cli(gctx, ["decompress", zp, "-c", "--patch-apply", pf])
    assert rc == 0 and out == new.tobytes(), err
    assert os.path.getsize(zp) * 10 <= new.size, os.path.getsize(zp)


@pytest.mark.gpu
def test_gpu_window_log_30_offset_codes(gctx):
    """offsets of 2^28 .. 2^30: Offset codes 28, 29 and 30.  A random 1 GiB + 3 prefix (no matches but the planted ones); NEW is 8 MiB cut
    from its 4th byte on (offsets 2^30 in the first frame, 2^30 - k * 2 MiB after) and 2 MiB cut from 3 * 2^27 before its end"""
    plen = (1 << 30) + 3
    old = np.random.default_rng(9).integers(0, 256, plen, dtype=np.uint8)
    new = np.concatenate([old[3: 3 + (8 << 20)], old[plen - 3 * (1 << 27): plen - 3 * (1 << 27) + (2 << 20)]])
    comp, cs, ds = ldm_compress(gctx, new, old, 2 << 20, 3, 30)
    frames = split(comp, cs)
    assert all(f[5] == 0xA0 for f in frames)
    offs = []
    for fr, d in zip(frames, ds):
        back, mo = restated([fr], [d], old)
        assert back == new[sum(ds[: len(offs)]): sum(ds[: len(offs)]) + d].tobytes()
        offs.append(mo)
    codes = {(o + 3).bit_length() - 1 for o in offs}
    assert {28, 29, 30} <= codes, offs
    assert zstd_decompress(frames, ds, prefix=old, window_log_max=30) == new.tobytes()
    back, st, rc = ours_decompress(gctx, frames, ds, prefix=old, window_log_max=30)
    assert rc == 0 and back == new.tobytes()


@pytest.mark.gpu
def test_gpu_window_log_30_without_prefix(gctx):
    """one frame of 600 MiB from libzstd (window log 30, LDM) whose second half repeats the first, 300 MiB back: zk_exec_kernel
    resolves the offsets with WindowLogMax(30) and the frame is refused by default"""
    half = np.random.default_rng(17).integers(0, 256, 300 << 20, dtype=np.uint8)
    data = np.concatenate([half, half])
    frames, ds = zstd_compress(data, data.size, 1, window_log=30, ldm=True)
    assert len(frames) == 1 and frames[0][4] & 0x20            # Single_Segment: the window is the content size, 600 MiB
    got, st, rc = ours_decompress(gctx, frames, ds)
    assert rc == -16
    got, st, rc = ours_decompress(gctx, frames, ds, window_log_max=30)
    assert rc == 0 and got == data.tobytes()


@pytest.mark.gpu
def test_gpu_ldm_golden(gctx):
    assert ldm_golden(gctx) == json.load(open(GOLDEN_LDM))
