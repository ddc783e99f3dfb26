"""Command-line front end with the reference CLI's arguments and behaviour (SURVEY.md 8f.4), over the GPU codec.

    python -m zeekstd_b200 [compress] [-l N] [-s 2M] [--frame-size-policy ..] [--patch-from F] [INPUT] [-o OUT]
    python -m zeekstd_b200 decompress [--from N | --from-frame I] [--to N|end | --to-frame I|end] [--patch-apply F] INPUT [-o OUT]
    python -m zeekstd_b200 list [--from-frame I] [--to-frame I|end | --num-frames N] [-d] [--seek-table-format head|foot] INPUT

What each piece follows in the reference: argument set and value parsers cli/src/args.rs:10-329; sub-commands, output
path derivation, overwrite checks and the list tables cli/src/command.rs:33-473; the compress loop (Encoder fed from a
reader, optional stand-alone Head-format seek table) cli/src/compress.rs:55-106; the decompress loop
cli/src/decompress.rs:21-117.  The codec underneath is this package's Encoder / Decoder, i.e. the CUDA path: there is no
CPU route.  Patch files get the parameters the reference sets (compress.rs:31-37, decompress.rs:53-62): `--patch-from`
sets window log clamp(ilog2(len) + 1, 17, 30) and long-distance matching, so matches reach anywhere in the window's part of
the prefix; `--patch-apply` raises the decoder's window limit to 2^max(27, ilog2(len) + 1) (at most 2^30) -- never below
the default, since this encoder's frames announce at least 128 KiB.  `--mmap-prefix` / `--no-mmap-prefix` choose between
np.memmap and a read.
"""
from __future__ import annotations

import argparse
import os
import stat
import sys
import time

import numpy as np

IN_CHUNK = 1 << 17            # CCtx::in_size() of the reference's read loop (compress.rs:60)
OUT_CHUNK = 8 << 20           # the reference uses DCtx::out_size(); larger here so one call spans whole frames
MMAP_THRESHOLD = 0x0010_0000  # args.rs:10 (the reference's comment says 128 MiB; the constant is 1 MiB)


class CliError(Exception):
    pass


# ------------------------------------------------------------------------------------------- value parsers (args.rs:12-112)
def byte_value(s: str) -> int:
    digits = ""
    for ch in s:
        if ch.isascii() and ch.isdigit():
            digits += ch
        else:
            break
    unit = "".join(ch for ch in s[len(digits):] if not ch.isspace())
    if not digits:
        raise argparse.ArgumentTypeError(f"invalid byte value: {s!r}")
    v = int(digits)
    mul = {"B": 1, "": 1, "K": 1 << 10, "kib": 1 << 10, "M": 1 << 20, "mib": 1 << 20, "G": 1 << 30, "gib": 1 << 30}.get(unit)
    if mul is None:
        raise argparse.ArgumentTypeError(f"Unknown unit: {unit!r}")
    v *= mul
    if v >= 1 << 64:
        raise argparse.ArgumentTypeError("Byte value too large")
    return v


def offset_limit(s: str):
    return None if s.lower() == "end" else byte_value(s)


def last_frame(s: str):
    if s.lower() == "end":
        return "end"
    try:
        v = int(s)
    except ValueError:
        raise argparse.ArgumentTypeError(f"invalid frame index: {s!r}")
    if not 0 <= v < 1 << 32:
        raise argparse.ArgumentTypeError(f"invalid frame index: {s!r}")
    return v


def num_frames(s: str) -> int:
    try:
        v = int(s)
    except ValueError:
        raise argparse.ArgumentTypeError(f"invalid frame number: {s!r}")
    if v <= 0:
        raise argparse.ArgumentTypeError("frame number must be greater than 0")
    return v


def u32(s: str) -> int:
    v = int(s)
    if not 0 <= v < 1 << 32:
        raise argparse.ArgumentTypeError(f"out of range: {s!r}")
    return v


def human_bytes(n: int) -> str:
    """indicatif::HumanBytes: binary prefixes, two decimals, plain integer below 1 KiB"""
    if n < 1024:
        return f"{n} B"
    v = float(n)
    for p in ("Ki", "Mi", "Gi", "Ti", "Pi", "Ei"):
        v /= 1024.0
        if v < 1024.0 or p == "Ei":
            return f"{v:.2f} {p}B"
    return f"{n} B"


def raw_bytes(n: int) -> str:
    return str(n)


# ------------------------------------------------------------------------------------------------------------ parser
def _add_flags(p, top: bool):
    d = {} if top else {"default": argparse.SUPPRESS}
    p.add_argument("-q", "--quiet", action="store_true", help="Suppress output. Ignored in list mode.", **d)
    p.add_argument("-r", "--raw-bytes", action="store_true", help="Disable human-readable formatting for all byte numbers.", **d)


def _add_common(p):
    p.add_argument("-f", "--force", action="store_true", help="Disable input and output checks.")
    p.add_argument("-c", "--stdout", action="store_true", help="Write to STDOUT.")
    p.add_argument("--no-progress", action="store_true", help="Do not show the progress counter.")
    p.add_argument("--mmap-prefix", action="store_true", help="Force memory-mapping prefix (patch) files.")
    p.add_argument("--no-mmap-prefix", action="store_true", help="Force disable memory-mapping prefix (patch) files.")
    p.add_argument("--seek-table-file", default=None, help='Path to the seek table file. If specified, implies the "Head" seek table format.')


def _level(s: str) -> int:
    v = int(s)
    if not 1 <= v <= 19:
        raise argparse.ArgumentTypeError("compression level must be between 1 and 19")
    return v


def build_parser() -> argparse.ArgumentParser:
    ap = argparse.ArgumentParser(prog="zeekstd_b200", description="Compress and decompress data using the Zstandard Seekable Format (B200 codec).")
    _add_flags(ap, True)
    sub = ap.add_subparsers(dest="command")

    c = sub.add_parser("compress", aliases=["c"], help="Compress INPUT_FILE (default); reads from STDIN if INPUT_FILE is `-` or not provided")
    _add_flags(c, False); _add_common(c)
    c.add_argument("-l", "--compression-level", type=_level, default=3)
    c.add_argument("--no-checksum", action="store_true", help="Don't include frame checksums.")
    c.add_argument("-s", "--frame-size", type=byte_value, default=byte_value("2M"))
    c.add_argument("--frame-size-policy", choices=["compressed", "uncompressed"], default="uncompressed")
    c.add_argument("--patch-from", default=None, help="Provide a reference point for Zstandard's diff engine.")
    c.add_argument("input_file", nargs="?", default="-")
    c.add_argument("-o", "--output-file", default=None)

    d = sub.add_parser("decompress", aliases=["d"], help="Decompress INPUT_FILE")
    _add_flags(d, False); _add_common(d)
    g0 = d.add_mutually_exclusive_group()
    g0.add_argument("--from", dest="from_", type=int, default=None, help="The offset (of the uncompressed data) where decompression starts.")
    g0.add_argument("--from-frame", type=u32, default=None)
    g1 = d.add_mutually_exclusive_group()
    g1.add_argument("--to", type=offset_limit, default="end", help="Accepts the special value 'end'.")
    g1.add_argument("--to-frame", type=last_frame, default=None)
    d.add_argument("--patch-apply", default=None)
    d.add_argument("input_file")
    d.add_argument("-o", "--output-file", default=None)

    li = sub.add_parser("list", aliases=["l"], help="Print information about seekable Zstandard-compressed files")
    _add_flags(li, False)
    li.add_argument("--from-frame", type=u32, default=None)
    g2 = li.add_mutually_exclusive_group()
    g2.add_argument("--to-frame", type=last_frame, default=None)
    g2.add_argument("--num-frames", type=num_frames, default=None)
    li.add_argument("-d", "--detail", action="store_true")
    li.add_argument("--seek-table-format", choices=["head", "foot"], default="foot")
    li.add_argument("input_file")
    return ap


_COMMANDS = {"compress": "compress", "c": "compress", "decompress": "decompress", "d": "decompress", "list": "list", "l": "list"}
_TOP_FLAGS = {"-q", "--quiet", "-r", "--raw-bytes", "-h", "--help"}


def parse_args(argv):
    """main.rs:12-31: without a sub-command the arguments are those of `compress`"""
    argv = list(argv)
    i = 0
    while i < len(argv) and argv[i] in _TOP_FLAGS:
        i += 1
    if i == len(argv) or argv[i] not in _COMMANDS:
        if i == len(argv) and not argv:
            build_parser().print_help(sys.stderr)
            raise SystemExit(2)
        argv.insert(i, "compress")
    ns = build_parser().parse_args(argv)
    ns.command = _COMMANDS[ns.command]
    return ns


# ------------------------------------------------------------------------------------------------------ file checks
def _checked_out_file(path: str, in_path, quiet: bool, force: bool):
    """command.rs:45-78"""
    exists = os.path.exists(path)
    is_chr = exists and stat.S_ISCHR(os.stat(path).st_mode)
    if not force and exists and not is_chr:
        if quiet or in_path is None:
            raise CliError(f"{path} already exists; not overwritten")
        sys.stderr.write(f"{path} already exists; overwrite (y/n) ? ")
        sys.stderr.flush()
        if sys.stdin.readline().rstrip("\r\n") != "y":
            raise CliError(f"{path} already exists")
    try:
        return open(path, "wb")
    except OSError as e:
        raise CliError(f"Failed to open output file: {e}")


def _out_path(ns, in_path):
    """command.rs:93-126"""
    if ns.command == "list" or ns.stdout:
        return None
    if ns.output_file is not None:
        return ns.output_file
    if in_path is None:
        return None
    if ns.command == "compress":
        return in_path + ".zst"
    root, ext = os.path.splitext(in_path)
    if ext != ".zst":
        raise CliError(f"{in_path}: unknown extension (.zst expected); cannot derive the output file name")
    return root


def _new_writer(out_path, in_path, quiet: bool, force: bool):
    if out_path is not None:
        return _checked_out_file(out_path, in_path, quiet, force)
    if not force and sys.stdout.isatty():
        raise CliError("stdout is a terminal, aborting")
    return sys.stdout.buffer


def _load_prefix(path, use_mmap: bool):
    """command.rs:349-384"""
    if path is None:
        return None
    try:
        if use_mmap and os.path.getsize(path) > 0:
            return np.memmap(path, dtype=np.uint8, mode="r")
        return np.fromfile(path, dtype=np.uint8)
    except OSError as e:
        raise CliError(f"Failed to load prefix (patch) file: {e}")


def _use_mmap(ns, prefix_len) -> bool:
    """args.rs:162-172"""
    if ns.mmap_prefix:
        return True
    if ns.no_mmap_prefix:
        return False
    return prefix_len is not None and prefix_len >= MMAP_THRESHOLD


class _Progress:
    """the reference's indicatif counter ("{pos} of {len}" on stderr, 5 Hz), shown on a terminal only"""

    def __init__(self, total, fmt, enabled: bool, pos: int = 0):
        self.total, self.fmt, self.pos, self.last = total, fmt, pos, 0.0
        self.on = enabled and sys.stderr.isatty()

    def inc(self, n: int):
        self.pos += n
        if self.on and time.monotonic() - self.last >= 0.2:
            self.last = time.monotonic()
            tot = self.fmt(self.total) if self.total is not None else "?"
            sys.stderr.write(f"\r{self.fmt(self.pos)} of {tot}")
            sys.stderr.flush()

    def finish(self):
        if self.on:
            sys.stderr.write("\r" + " " * 48 + "\r")
            sys.stderr.flush()


# --------------------------------------------------------------------------------------------------------- commands
def _read_seek_table(zk, path: str, fmt: int):
    """SeekTable::from_seekable_format over a file without reading the archive: only the table's bytes are fetched
    (Foot: the integrity field gives the frame count, seek_table.rs:379-436; Head: the skippable header gives the size)"""
    size = os.path.getsize(path)
    with open(path, "rb") as f:
        if fmt == zk.Format.Head:
            head = f.read(8)
            n = int.from_bytes(head[4:8], "little") + 8 if len(head) == 8 else 8
            f.seek(0)
            return zk.SeekTable.from_bytes(f.read(min(n, size)), zk.Format.Head)
        tail_n = min(size, zk.SEEK_TABLE_INTEGRITY_SIZE)
        f.seek(size - tail_n)
        tail = f.read(tail_n)
        want = size
        if tail_n == zk.SEEK_TABLE_INTEGRITY_SIZE:
            frames = int.from_bytes(tail[0:4], "little")
            per = 12 if tail[4] & 0x80 else 8
            want = min(size, 8 + frames * per + zk.SEEK_TABLE_INTEGRITY_SIZE)
        f.seek(size - want)
        return zk.SeekTable.from_bytes(f.read(want), zk.Format.Foot)


def _run_compress(zk, ns, fmt_bytes) -> int:
    in_path = None if ns.input_file == "-" else ns.input_file
    out_path = _out_path(ns, in_path)
    if in_path is not None:
        try:
            reader = open(in_path, "rb")
        except OSError as e:
            raise CliError(f"Failed to open input file: {e}")
    else:
        if not ns.force and sys.stdin.isatty():
            raise CliError("stdin is a terminal, aborting")
        reader = sys.stdin.buffer
    if ns.frame_size >= 1 << 32:
        raise CliError("Frame size too big")
    prefix_len = os.path.getsize(ns.patch_from) if ns.patch_from and os.path.exists(ns.patch_from) else None
    st_file = None
    if ns.seek_table_file is not None:
        try:
            st_file = _checked_out_file(ns.seek_table_file, in_path, ns.quiet, ns.force)
        except CliError as e:
            raise CliError(f"Failed to create seek table file: {e}")
    in_len = os.path.getsize(in_path) if in_path is not None and os.path.isfile(in_path) else None
    bar = _Progress(in_len, fmt_bytes, not ns.quiet and not ns.no_progress)
    writer = _new_writer(out_path, in_path, ns.quiet, ns.force)

    policy = (zk.FrameSizePolicy.Compressed if ns.frame_size_policy == "compressed" else zk.FrameSizePolicy.Uncompressed)(ns.frame_size)
    enc = (zk.EncodeOptions().frame_size_policy(policy).checksum_flag(not ns.no_checksum)
           .compression_level(ns.compression_level).into_encoder(writer))
    prefix = _load_prefix(ns.patch_from, _use_mmap(ns, prefix_len))

    read = 0
    while True:
        buf = reader.read(IN_CHUNK)
        if not buf:
            break
        read += len(buf)
        bar.inc(len(buf))
        mv, pos = memoryview(buf), 0
        while pos < len(mv):
            pos += enc.compress_with_prefix(mv[pos:], prefix)
    if st_file is not None:
        enc.end_frame()
        enc.flush()
        written = enc.written_compressed()
        ser = enc.seek_table().clone().into_format_serializer(zk.Format.Head)
        blob = ser.to_bytes()
        st_file.write(blob)
        st_file.close()
        written += len(blob)
    else:
        written = enc.finish()
    bar.finish()
    if writer is not sys.stdout.buffer:
        writer.close()
    else:
        writer.flush()
    if not ns.quiet:
        ratio = 100.0 / read * written if read else float("nan")
        sys.stderr.write(f"{in_path or 'STDIN'} : {ratio:.2f}% ( {fmt_bytes(read)} => {fmt_bytes(written)}, {out_path or 'STDOUT'})\n")
    return 0


def _patch_window_log(prefix_len: int, floor: int) -> int:
    """ilog2(len) + 1 (cli/src/compress.rs:31-37), between `floor` and 30 (the largest window log of this codec)"""
    return min(30, max(floor, max(prefix_len, 1).bit_length()))


class _ContextParams:
    """sets context parameters for one command and restores the previous values afterwards (the context outlives the command)"""

    def __init__(self, ctx, cparams=(), dparams=()):
        self.ctx, self.cparams, self.dparams = ctx, list(cparams), list(dparams)

    def __enter__(self):
        self.saved = (dict(self.ctx.cparams), dict(self.ctx.dparams))
        for p in self.cparams:
            self.ctx.set_cparameter(p)
        for p in self.dparams:
            self.ctx.set_dparameter(p)
        return self

    def __exit__(self, *exc):
        import zeekstd_b200 as zk
        for p in self.cparams:
            self.ctx.set_cparameter(zk.CParameter(p.param, self.saved[0].get(p.param, 0)))
        for p in self.dparams:
            self.ctx.set_dparameter(zk.DParameter(p.param, self.saved[1].get(p.param, 0)))
        return False


def _run_decompress(zk, ns, fmt_bytes) -> int:
    in_path = ns.input_file
    out_path = _out_path(ns, in_path)
    prefix_len = os.path.getsize(ns.patch_apply) if ns.patch_apply and os.path.exists(ns.patch_apply) else None
    writer = _new_writer(out_path, in_path, ns.quiet, ns.force)
    try:
        src = open(in_path, "rb")
    except OSError as e:
        raise CliError(f"Failed to open input file: {e}")
    try:
        if ns.seek_table_file is not None:
            try:
                with open(ns.seek_table_file, "rb") as f:
                    table = zk.SeekTable.from_reader(f)
            except OSError as e:
                raise CliError(f"Failed to open seek table file: {e}")
        else:
            table = _read_seek_table(zk, in_path, zk.Format.Foot)
    except zk.Error as e:
        raise CliError(f"Failed to parse seek table: {e}")
    try:
        offset = table.frame_start_decomp(ns.from_frame) if ns.from_frame is not None else (ns.from_ or 0)
    except zk.Error as e:
        raise CliError(f"Failed to get decompression offset: {e}")
    try:
        if ns.to_frame is not None:
            limit = table.size_decomp() if ns.to_frame == "end" else table.frame_end_decomp(ns.to_frame)
        else:
            limit = table.size_decomp() if ns.to is None else ns.to
    except zk.Error as e:
        raise CliError(f"Failed to get decompression offset limit: {e}")
    bar = _Progress(limit, fmt_bytes, not ns.quiet and not ns.no_progress, pos=offset)
    try:
        dec = zk.DecodeOptions(src).seek_table(table).offset(offset).offset_limit(limit).into_decoder()
    except zk.Error as e:
        raise CliError(f"Failed to create decoder: {e}")
    prefix = _load_prefix(ns.patch_apply, _use_mmap(ns, prefix_len))

    buf = bytearray(OUT_CHUNK)
    view = memoryview(buf)
    written = 0
    while True:
        try:
            n = dec.decompress_with_prefix(view, prefix)
        except zk.Error as e:
            raise CliError(f"Failed to decompress data: {e}")
        if n == 0:
            break
        bar.inc(n)
        writer.write(view[:n])
        written += n
    bar.finish()
    if writer is not sys.stdout.buffer:
        writer.close()
    else:
        writer.flush()
    src.close()
    if not ns.quiet:
        sys.stderr.write(f"{in_path} : {fmt_bytes(written)}\n")
    return 0


def _run_list(zk, ns, fmt_bytes) -> int:
    if not os.path.exists(ns.input_file):
        raise CliError("Failed to open input file")
    try:
        st = _read_seek_table(zk, ns.input_file, zk.Format.Head if ns.seek_table_format == "head" else zk.Format.Foot)
    except zk.Error as e:
        raise CliError(f"Failed to read seek table: {e}")
    if ns.num_frames is not None:
        end = (ns.from_frame or 0) + ns.num_frames - 1
    elif ns.to_frame is not None:
        end = st.num_frames() - 1 if ns.to_frame == "end" else ns.to_frame
    else:
        end = None
    out = sys.stdout
    if ns.from_frame is None and end is None and not ns.detail:
        n = st.num_frames()
        comp, unc = st.frame_end_comp(n - 1), st.frame_end_decomp(n - 1)
        ratio = unc / comp if comp else float("nan")
        out.write(f"{'Frames': <15} {'Compressed': <15} {'Uncompressed': <15} {'Max Frame Size': <15} {'Ratio': <10} {'Filename': <15}\n")
        out.write(f"{n: <15} {fmt_bytes(comp): <15} {fmt_bytes(unc): <15} {fmt_bytes(st.max_frame_size_decomp()): <15} {ratio: <10.3f} {ns.input_file: <15}\n")
        return 0
    start = ns.from_frame or 0
    if end is None:
        end = st.num_frames() - 1
    if start > end:
        raise CliError(f"Start frame ({start}) cannot be greater than end frame ({end})")
    out.write(f"{'Frame Index': <15} {'Compressed': <15} {'Uncompressed': <15} {'Compressed Offset': <20} {'Uncompressed Offset': <20}\n")
    lines = []
    for i in range(start, end + 1):
        try:
            row = (fmt_bytes(st.frame_size_comp(i)), fmt_bytes(st.frame_size_decomp(i)), fmt_bytes(st.frame_start_comp(i)), fmt_bytes(st.frame_start_decomp(i)))
        except zk.Error as e:
            out.write("".join(lines))
            raise CliError(str(e))
        lines.append(f"{i: <15} {row[0]: <15} {row[1]: <15} {row[2]: <20} {row[3]: <20}\n")
        if len(lines) == 100:
            out.write("".join(lines)); lines = []
    out.write("".join(lines))
    return 0


def main(argv=None) -> int:
    ns = parse_args(sys.argv[1:] if argv is None else argv)
    import zeekstd_b200 as zk
    fmt_bytes = raw_bytes if ns.raw_bytes else human_bytes
    try:
        if ns.command == "compress":
            n = os.path.getsize(ns.patch_from) if ns.patch_from and os.path.exists(ns.patch_from) else None
            cp = [] if n is None else [zk.CParameter.WindowLog(_patch_window_log(n, 17)), zk.CParameter.EnableLongDistanceMatching(True)]
            with _ContextParams(zk.default_context(), cparams=cp):
                return _run_compress(zk, ns, fmt_bytes)
        if ns.command == "decompress":
            n = os.path.getsize(ns.patch_apply) if ns.patch_apply and os.path.exists(ns.patch_apply) else None
            dp = [] if n is None else [zk.DParameter.WindowLogMax(_patch_window_log(n, 27))]
            with _ContextParams(zk.default_context(), dparams=dp):
                return _run_decompress(zk, ns, fmt_bytes)
        return _run_list(zk, ns, fmt_bytes)
    except CliError as e:
        sys.stderr.write(f"Error: {e}\n")
        return 1
    except zk.Error as e:
        sys.stderr.write(f"Error: {e}\n")
        return 1


if __name__ == "__main__":
    sys.exit(main())
