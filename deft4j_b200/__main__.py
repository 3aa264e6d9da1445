"""`python -m deft4j_b200 optimise|optimise-folder|gzip-compress ...` — mirror of deft4j-cmd (SURVEY.md §8f row 4).

cmd/Main.java:8-25 (subcommands), cmd/Optimise.java:15-54, cmd/OptimiseFolder.java:33-67 and
cmd/CMDUtil.java:57-181: same positional arguments, option names, stdout/stderr lines, temp-file overwrite protocol
and exit codes.  Only `--mode NONE` exists here (the recompress modes call third-party compressors, DESIGN.md §5).
"""
import argparse
import os
import shutil
import sys
import tempfile

from .container import getContainerForBytes, getContainerForExt, RawDeflateFile


def _stream_cls():
    from .deflate_stream import DeflateStream   # the CUDA engine; raises when the library or a device is missing
    return DeflateStream


def optimise_bytes(data, container, merge_blocks, out=None, err=None):
    """CMDUtil.optimise (CMDUtil.java:57-116): returns the rewritten bytes or None."""
    out, err = out or sys.stdout, err or sys.stderr
    if container is None:
        print("Invalid file container", file=err)
        return None
    if container.read(data):
        print("File type recognised as " + container.fileType(), file=out)
        saved = container.optimise(merge_blocks, out)
        if saved != 0:
            print("Saved %d bits with optimisation" % saved, file=out)
        try:
            return container.write()   # always re-serialised, even when nothing was saved (SURVEY.md H11)
        except IOError:
            print("Failed to write output", file=err)
    print("Invalid %s file" % container.fileType(), file=err)
    return None


def optimise_file(inp, outp, fmt, raw, merge_blocks, stream_cls, out=None, err=None):
    """CMDUtil.optimiseFile (CMDUtil.java:119-181)."""
    out, err = out or sys.stdout, err or sys.stderr
    if not os.path.isfile(inp):
        print("Error: Input file does not exist", file=err)
        return False
    if os.path.isdir(outp):
        print("Error: Output file is a directory", file=err)
        return False
    with open(inp, "rb") as f:
        data = f.read()
    if raw:
        container = RawDeflateFile(stream_cls)
    elif fmt is not None:
        container = getContainerForExt(fmt, stream_cls)
    else:
        container = getContainerForBytes(data, os.path.basename(inp), stream_cls)
    result = optimise_bytes(data, container, merge_blocks, out, err)
    if result is None:
        print("Failed to optimise input file", file=err)
        return False
    if os.path.isfile(outp):       # overwrite through a temp file, only on success (:137-176)
        ext = os.path.splitext(inp)[1] or None
        fd, tmp = tempfile.mkstemp(prefix="deft-temp-", suffix=ext)
        try:
            with os.fdopen(fd, "wb") as f:
                f.write(result)
            shutil.copyfile(tmp, outp)
        finally:
            try:
                os.unlink(tmp)
            except OSError:
                print("Issue deleting temporary file " + tmp, file=err)
    else:
        with open(outp, "wb") as f:
            f.write(result)
    return True


def _write_back(path, result, inp, err):
    """the overwrite-through-a-temp-file protocol of CMDUtil.optimiseFile (:137-176)"""
    if os.path.isfile(path):
        ext = os.path.splitext(inp)[1] or None
        fd, tmp = tempfile.mkstemp(prefix="deft-temp-", suffix=ext)
        try:
            with os.fdopen(fd, "wb") as f:
                f.write(result)
            shutil.copyfile(tmp, path)
        finally:
            try:
                os.unlink(tmp)
            except OSError:
                print("Issue deleting temporary file " + tmp, file=err)
    else:
        with open(path, "wb") as f:
            f.write(result)


def optimise_files_batched(paths, merge_blocks, stream_cls, out, err, max_bytes=256 << 20):
    """`optimise-folder` over many files: the deflate streams of a whole group of files (up to max_bytes of input) go to
    the device as ONE list (DeflateFilesContainer.optimise's batch point, DeflateFilesContainer.java:18-43, widened
    to the folder); every file then prints and is written back exactly as CMDUtil.optimiseFile would have done."""
    import io
    from .container.deflate_files_container import optimise_containers
    ok = True
    group, size = [], 0
    native_png = stream_cls is None or getattr(stream_cls, "__module__", "") == "deft4j_b200.deflate_stream"

    def flush():
        nonlocal ok
        conts = [g for g in group if g[2] is not None]
        sinks = [io.StringIO() for _ in conts]
        try:
            totals = optimise_containers([g[2] for g in conts], merge_blocks, sinks)
        except Exception as e:  # noqa: BLE001
            print("Error when optimising files %s ..: %r" % (conts[0][0] if conts else "", e), file=err)
            totals, ok = None, False
        k = 0
        for path, data, cont in group:
            print("Optimising file " + path, file=out)
            if cont is None:
                print("Invalid file container" if data is None else "Invalid file", file=err)
                print("Failed to optimise input file", file=err)
                print("Error when optimising file " + path, file=err)
                ok = False
                continue
            print("File type recognised as " + cont.fileType(), file=out)
            if totals is None:
                k += 1
                continue
            out.write(sinks[k].getvalue())
            if totals[k] != 0:
                print("Saved %d bits with optimisation" % totals[k], file=out)
            k += 1
            try:
                _write_back(path, cont.write(), path, err)
            except IOError:
                print("Failed to write output", file=err)
                print("Error when optimising file " + path, file=err)
                ok = False
        group.clear()

    pending = []   # (path, data) of the group being collected

    def native_group(fmt):
        """A group made of files of ONE kind (PNG, ZIP, gzip or zlib by magic) goes through that kind's native front-end
        (deft4cu_{png,zip,gz,zlib}_optimise_batch): same lines, same files, the container work in C++ instead of in this
        interpreter."""
        nonlocal ok
        from .container import optimise_png_files, optimise_zip_files, optimise_gz_files, optimise_zlib_files
        fn, label = {"png": (optimise_png_files, "PNG"), "zip": (optimise_zip_files, "Zip"),
                     "gzip": (optimise_gz_files, "GZip"), "zlib": (optimise_zlib_files, "ZLib")}[fmt]
        res = fn([d for _, d in pending], merge_blocks)
        for (path, _), r in zip(pending, res):
            print("Optimising file " + path, file=out)
            if r["status"] == 1:
                print("Invalid file", file=err)
                print("Failed to optimise input file", file=err)
                print("Error when optimising file " + path, file=err)
                ok = False
                continue
            print("File type recognised as " + label, file=out)
            if r["status"] == 3:
                print("Error when optimising file " + path, file=err)
                ok = False
                continue
            for i, (name, saved) in enumerate(r["streams"]):
                if saved > 0:
                    print("%d bits saved in stream %d (%s)" % (saved, i, name), file=out)
            if r["saved_bits"] > 0:
                print("Total bits saved %d" % r["saved_bits"], file=out)
            if r["saved_bits"] != 0:
                print("Saved %d bits with optimisation" % r["saved_bits"], file=out)
            if r["status"] == 2:
                print("Failed to write output", file=err)
                print("Error when optimising file " + path, file=err)
                ok = False
                continue
            _write_back(path, r["out"], path, err)
        pending.clear()

    def read_group():
        from .container.deflate_files_container import read_containers
        from .container.container_util import detectFormat
        if native_png and pending:
            kinds = {detectFormat(d) for _, d in pending}
            if len(kinds) == 1 and next(iter(kinds)) in ("png", "zip", "gzip", "zlib"):
                if group:
                    flush()
                native_group(kinds.pop())
                return
        conts = read_containers([d for _, d in pending], [os.path.basename(p) for p, _ in pending], stream_cls)
        for (path, data), cont in zip(pending, conts):
            group.append((path, data, cont))
        pending.clear()

    for path in paths:
        with open(path, "rb") as f:
            data = f.read()
        pending.append((path, data))
        size += len(data)
        if size >= max_bytes or len(pending) >= 4096:
            read_group()
            flush()
            size = 0
    if pending:
        read_group()
    if group:
        flush()
    return ok


def gzip_compress_file(inp, outp, merge_blocks, block_bytes, stream_cls, out=None, err=None):
    """`gzip-compress`: the input's bytes compressed and optimised on the device, wrapped in a gzip member with GZFile's
    default header."""
    from .container.gz_file import GZFile
    out, err = out or sys.stdout, err or sys.stderr
    if not os.path.isfile(inp):
        print("Error: Input file does not exist", file=err)
        return False
    if os.path.isdir(outp):
        print("Error: Output file is a directory", file=err)
        return False
    with open(inp, "rb") as f:
        data = f.read()
    stream = stream_cls.compress_batch([data], block_bytes=block_bytes)[0]
    if stream is None:
        print("Failed to compress input file", file=err)
        return False
    saved = stream.optimise(merge_blocks)
    if saved != 0:
        print("Saved %d bits with optimisation" % saved, file=out)
    gz = GZFile(stream_cls)
    gz.setData(stream)
    _write_back(outp, gz.write(), inp, err)
    return True


def main(argv=None, out=None, err=None, stream_cls=None):
    """`stream_cls` lets a caller supply another implementation of the DeflateStream interface (the CPU-only tests
    pass their checker); the command line always uses the CUDA engine."""
    out, err = out or sys.stdout, err or sys.stderr
    ap = argparse.ArgumentParser(prog="deft4j", description="Deflate stream optimiser")
    sub = ap.add_subparsers(dest="cmd", required=True)

    def common(p):
        p.add_argument("--recompress-mode", "--mode", "-m", default="NONE", choices=["NONE"], dest="mode",
                       help="only NONE is available in this build")
        p.add_argument("--zopfli-iter", "--iter", "-I", type=int, default=20, help="(unused with --mode NONE)")
        p.add_argument("--merge-blocks", "-b", dest="merge_blocks", action="store_true", default=True,
                       help="Try merging deflate blocks (default)")
        p.add_argument("--no-merge-blocks", dest="merge_blocks", action="store_false")

    p = sub.add_parser("optimise", help="Deflate stream optimiser")
    p.add_argument("inputFile", help="The file to optimise")
    p.add_argument("outputFile", help="The optimised file")
    p.add_argument("--format", "-f", default=None, help="File format")
    p.add_argument("--raw", "-r", action="store_true", help="Ignore file format, treat input as a raw deflate stream")
    common(p)
    p = sub.add_parser("optimise-folder", help="Optimise every recognised file below a folder, in place")
    p.add_argument("inputFolder")
    common(p)
    p = sub.add_parser("gzip-compress", help="Compress a file to gzip with this library's own device compressor",
                       description="Compress inputFile into a gzip file on the GPU: LZ77 matching and a lazy parse into "
                       "fixed-coded blocks, then this optimiser's block rewriting.  The compressor is this library's own; "
                       "its bytes are not those of the reference's gzip-compress, whose compressors are not available here.")
    p.add_argument("inputFile", help="The file to compress")
    p.add_argument("outputFile", help="The gzip file to write")
    p.add_argument("--merge-blocks", "-b", dest="merge_blocks", action="store_true", default=False,
                   help="Also try merging deflate blocks (off by default: on large stationary inputs it is slow)")
    p.add_argument("--block-bytes", type=int, default=0,
                   help="Input bytes per deflate block, 256..65535 (default 32768)")
    a = ap.parse_args(argv)
    cls = stream_cls or _stream_cls()
    if a.cmd == "gzip-compress":
        ok = gzip_compress_file(a.inputFile, a.outputFile, a.merge_blocks, a.block_bytes, cls, out, err)
        if not ok:
            print("Failed to compress " + a.inputFile, file=err)
        return 0 if ok else 1
    if a.cmd == "optimise":
        try:
            ok = optimise_file(a.inputFile, a.outputFile, a.format, a.raw, a.merge_blocks, cls, out, err)
        except Exception:
            print("Error when optimising file " + a.inputFile, file=err)
            raise
        if not ok:
            print("Failed to optimise " + a.inputFile, file=err)
        return 0 if ok else 1
    # optimise-folder (OptimiseFolder.java:33-67): regular files whose format is recognised by magic or extension
    ok = True
    paths = []
    if os.path.isdir(a.inputFolder):
        for root, _, files in os.walk(a.inputFolder):
            paths += [os.path.join(root, f) for f in sorted(files)]
    else:
        paths = [a.inputFolder]
    todo = []
    for path in paths:
        if not os.path.isfile(path):
            continue
        with open(path, "rb") as f:
            head = f.read(16)
        cont = getContainerForBytes(head, os.path.basename(path), cls)
        if cont is None or isinstance(cont, RawDeflateFile):
            continue
        todo.append(path)
    ok = optimise_files_batched(todo, a.merge_blocks, cls, out, err)
    if not ok:
        print("Failed to optimise " + a.inputFolder, file=err)
    return 0 if ok else 1


if __name__ == "__main__":
    sys.exit(main())
