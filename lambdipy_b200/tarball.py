"""Release tarballs compressed on the GPU.

Reference: PackageBuild.create_compressed_tarball (/root/reference/lambdipy/package_build.py:165-172)
writes `tarfile.open(path, "w:gz")` -- zlib level 9 on one core -- over every top-level entry of the
build directory.  Here the tar stream is laid out by `tarfile`'s own header code (so PAX headers, long
and non-ASCII names, links, directories and the end-of-archive blocks are what `tarfile` writes), but
file bodies are only recorded as (path, size); liblambdipy_b200 reads them, DEFLATE-compresses the
stream on the B200 (lb2_gzip_segments) and writes the .tar.gz.

`gzip.decompress` of the result equals the tar `tarfile.open(path, "w")` writes for the same tree; the
compressed bytes differ from zlib's.
"""
import ctypes as C
import glob
import os
import struct
import tarfile
import time

from . import _native as N


class _Recorder:
    """File object for TarFile: literal writes are kept, file bodies are added as (path, size)."""

    def __init__(self):
        self.segments = []   # bytes | (path, size)
        self.size = 0

    def write(self, b):
        b = bytes(b)
        if not b:
            return 0
        if self.segments and isinstance(self.segments[-1], bytearray):
            self.segments[-1] += b
        else:
            self.segments.append(bytearray(b))
        self.size += len(b)
        return len(b)

    def add_file(self, path, size):
        if size:
            self.segments.append((path, size))
            self.size += size

    def tell(self):
        return self.size


class _RecordingTarFile(tarfile.TarFile):
    """`tarfile` in "w" mode whose regular-file bodies are recorded instead of copied."""

    def addfile(self, tarinfo, fileobj=None):
        if fileobj is None or not tarinfo.isreg():
            return super().addfile(tarinfo, fileobj)
        # TarFile.addfile with the body replaced by a (path, size) record (3.13 refuses addfile(ti, None))
        self._check("awx")
        buf = tarinfo.tobuf(self.format, self.encoding, self.errors)
        self.fileobj.write(buf)
        self.offset += len(buf)
        self.fileobj.add_file(fileobj.name, tarinfo.size)
        blocks, remainder = divmod(tarinfo.size, tarfile.BLOCKSIZE)
        if remainder > 0:
            self.fileobj.write(tarfile.NUL * (tarfile.BLOCKSIZE - remainder))
            blocks += 1
        self.offset += blocks * tarfile.BLOCKSIZE
        self.members.append(tarinfo)


def record_tar(build_directory):
    """The tar stream of the reference's selection as segments: bytes (headers, padding, end of archive)
    and (path, size) for file bodies."""
    rec = _Recorder()
    with _RecordingTarFile(fileobj=rec, mode="w") as tar:
        for path in glob.glob(f'{build_directory}/*'):   # package_build.py:169, unsorted, no dotfiles
            tar.add(path, arcname=os.path.basename(path))
    return [bytes(s) if isinstance(s, bytearray) else s for s in rec.segments]


def materialize(segments):
    """The tar bytes the segments stand for (tests)."""
    out = bytearray()
    for s in segments:
        if isinstance(s, bytes):
            out += s
        else:
            with open(s[0], "rb") as f:
                out += f.read(s[1])
    return bytes(out)


def gzip_header(tarball_path, mtime=None):
    """The member header `tarfile.open(tarball_path, "w:gz")` writes (gzip.GzipFile), except XFL = 0: the
    stream is not zlib level 9."""
    fname = os.path.basename(tarball_path)
    try:
        fname = fname.encode("latin-1")
    except UnicodeEncodeError:
        fname = b""
    if fname.endswith(b".gz"):
        fname = fname[:-3]
    mtime = int(time.time()) if mtime is None else int(mtime)
    flags = 0x08 if fname else 0
    return b"\x1f\x8b\x08" + bytes([flags]) + struct.pack("<L", mtime) + b"\x00\xff" + (fname + b"\x00" if fname else b"")


def create_tarball(build_directory, tarball_path, ctx=None):
    """Write tarball_path as the reference does (tar of the top-level entries of build_directory, gzip),
    compressed on the GPU.  Returns the library's stats as a dict.  Raises NativeError (LB2_E_IO when a
    file changed size after it was recorded; no output file is left then)."""
    segments = record_tar(build_directory)
    if ctx is None:
        from .project_build import _context
        ctx = _context()
    keep = []
    arr = (N.GzSegment * max(1, len(segments)))()
    for i, s in enumerate(segments):
        if isinstance(s, bytes):
            buf = C.create_string_buffer(s, len(s))
            keep.append(buf)
            arr[i] = N.GzSegment(C.cast(buf, C.c_void_p), None, len(s))
        else:
            arr[i] = N.GzSegment(None, os.fsencode(s[0]), s[1])
    hdr = gzip_header(tarball_path)
    st = N.GzipStats()
    ctx.check(ctx.lib.lb2_gzip_segments(ctx.h, arr, len(segments), os.fsencode(tarball_path), hdr, len(hdr), C.byref(st)))
    return st.as_dict()


def deflate_device(ctx, d_in, n, hist=0, final=True, stream=None):
    """Raw DEFLATE of n device bytes at d_in (the `hist` bytes before it are history).  Returns
    (stream bytes, crc32, stats dict)."""
    cap = max(1, (n + 65535) // 65536) * 66560
    d_out = ctx.dev_alloc(cap)
    try:
        out_len, crc, st = C.c_uint64(), C.c_uint32(), N.GzipStats()
        ctx.check(ctx.lib.lb2_deflate_device(ctx.h, d_in, n, hist, 1 if final else 0, d_out, cap, C.byref(out_len),
                                             C.byref(crc), C.byref(st), stream))
        out = (C.c_char * max(1, out_len.value))()
        if out_len.value:
            ctx.d2h(out, d_out, out_len.value)
        return out.raw[:out_len.value], crc.value, st.as_dict()
    finally:
        ctx.dev_free(d_out)


def deflate_bytes(ctx, data, history=b"", final=True):
    """Raw DEFLATE of host bytes `data`, back-references allowed into `history` (at most its last 32 KiB)."""
    history = history[-32768:]
    blob = history + data
    d = ctx.dev_alloc(len(blob))
    try:
        if blob:
            ctx.h2d(d, C.c_char_p(blob), len(blob))
        return deflate_device(ctx, (d or 0) + len(history), len(data), len(history), final)
    finally:
        ctx.dev_free(d)


def gzip_bytes(ctx, data, name="data"):
    """A single-member gzip file of `data`, compressed on the GPU."""
    raw, crc, _ = deflate_bytes(ctx, data)
    return gzip_header(name + ".gz", mtime=0) + raw + struct.pack("<LL", crc, len(data) & 0xFFFFFFFF)
