"""Shared helpers for the test-suite (test infrastructure; not part of the product)."""
import ctypes
import json
import os
import subprocess
import zlib

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLDEN = os.path.join(ROOT, "tests", "golden")
REF_BIN = os.path.join(ROOT, "oracle", "_ref", "fastq_info")


def read_stream(path):
    """Bytes a gzFile reader would deliver: gzip members are inflated and concatenated, anything else is passed through."""
    with open(path, "rb") as fh:
        raw = fh.read()
    if raw[:2] != b"\x1f\x8b":
        return raw
    out = []
    while raw[:2] == b"\x1f\x8b":
        d = zlib.decompressobj(wbits=31)
        out.append(d.decompress(raw))
        out.append(d.flush())
        raw = d.unused_data
    return b"".join(out)


def golden_transcripts():
    with open(os.path.join(GOLDEN, "transcripts.json")) as fh:
        return json.load(fh)


def positional_files(argv):
    """The (up to two) file operands of a fastq_info argv (options may appear anywhere: GNU getopt permutes)."""
    pos = []
    stop = False
    for w in argv:
        if not stop and w == "--":
            stop = True
            continue
        if not stop and w.startswith("-") and len(w) > 1:
            continue
        pos.append(w)
    return pos


class _OracleResult(ctypes.Structure):
    _fields_ = [("rc", ctypes.c_int), ("out", ctypes.c_void_p), ("out_len", ctypes.c_size_t),
                ("err", ctypes.c_void_p), ("err_len", ctypes.c_size_t)]


_oracle = None


def oracle_lib():
    """Build (if needed) and load oracle/liboracle.so — the CPU restatement used as the checker."""
    global _oracle
    if _oracle is None:
        so = os.path.join(ROOT, "oracle", "liboracle.so")
        src = os.path.join(ROOT, "oracle", "fastq_oracle.c")
        if not os.path.exists(so) or os.path.getmtime(so) < os.path.getmtime(src):
            subprocess.check_call(["make", "-C", os.path.join(ROOT, "oracle"), "liboracle.so"], stdout=subprocess.DEVNULL)
        lib = ctypes.CDLL(so)
        lib.oracle_fastq_info.restype = ctypes.c_int
        lib.oracle_fastq_info.argtypes = [ctypes.c_int, ctypes.POINTER(ctypes.c_char_p), ctypes.c_char_p, ctypes.c_size_t,
                                          ctypes.c_char_p, ctypes.c_size_t, ctypes.POINTER(_OracleResult)]
        lib.oracle_free.argtypes = [ctypes.POINTER(_OracleResult)]
        lib.oracle_qual_range2enc.restype = ctypes.c_char_p
        lib.oracle_qual_range2enc.argtypes = [ctypes.c_uint, ctypes.c_uint]
        lib.oracle_sniff_format.argtypes = [ctypes.c_char_p]
        lib.oracle_sniff_colorspace.argtypes = [ctypes.c_char_p]
        lib.oracle_readname.restype = ctypes.c_long
        lib.oracle_readname.argtypes = [ctypes.c_char_p, ctypes.c_int, ctypes.c_int, ctypes.c_char_p, ctypes.POINTER(ctypes.c_ulong)]
        _oracle = lib
    return _oracle


def oracle_run(argv, data1=None, data2=None):
    """Run the oracle's fastq_info on in-memory streams → (rc, stdout, stderr) as latin-1 text."""
    lib = oracle_lib()
    full = [b"fastq_info"] + [a.encode("latin-1") for a in argv]
    arr = (ctypes.c_char_p * (len(full) + 1))(*full, None)
    res = _OracleResult()
    unopenable = ctypes.c_size_t(-1).value  # "could not open" marker
    lib.oracle_fastq_info(len(full), arr, data1, len(data1) if data1 is not None else unopenable,
                          data2, len(data2) if data2 is not None else unopenable, ctypes.byref(res))
    out = ctypes.string_at(res.out, res.out_len).decode("latin-1")
    err = ctypes.string_at(res.err, res.err_len).decode("latin-1")
    rc = res.rc
    lib.oracle_free(ctypes.byref(res))
    return rc, out, err


def oracle_run_files(argv, cwd=GOLDEN):
    """Like the CLI: open the positional files (relative to cwd), inflate, and run the oracle."""
    pos = positional_files(argv)
    datas = []
    for p in pos[:2]:
        path = os.path.join(cwd, p)
        datas.append(read_stream(path) if os.path.isfile(path) else None)
    while len(datas) < 2:
        datas.append(None)
    return oracle_run(argv, datas[0], datas[1])


def have_ref(tool="fastq_info"):
    return os.path.exists(os.path.join(ROOT, "oracle", "_ref", tool))


def fuzz_golden(name):
    """What the reference binaries returned on the seeded fuzz inputs of one test (tests/golden/fuzz/<name>.json, written by
    tests/golden/make_fuzz_golden.py): the fuzz tests compare with it where the binaries are not built."""
    path = os.path.join(GOLDEN, "fuzz", name + ".json")
    if not os.path.exists(path):
        import pytest
        pytest.skip(f"neither the reference binaries (oracle/_ref) nor tests/golden/fuzz/{name}.json: run tests/golden/make_fuzz_golden.py where they are built")
    with open(path) as fh:
        return json.load(fh)


def ref_run(argv, cwd=GOLDEN):
    """Run the unmodified reference binary (oracle/_ref) → (rc, stdout, stderr)."""
    p = subprocess.run([REF_BIN] + list(argv), cwd=cwd, capture_output=True)
    return p.returncode, p.stdout.decode("latin-1"), p.stderr.decode("latin-1")


# ---------------------------------------------------------------------------------------------- libfastq_gpu
class _Transcript(ctypes.Structure):
    _fields_ = [("rc", ctypes.c_int), ("out", ctypes.c_void_p), ("out_len", ctypes.c_size_t),
                ("err", ctypes.c_void_p), ("err_len", ctypes.c_size_t)]


_fqg = {}


def fqg_lib(kind="gpu"):
    """kind='gpu': the product, fastq_utils_b200/libfastq_gpu.so (needs a CUDA device to create a context).
    kind='sim': tests/sim/libfastq_sim.so — same host code over a sequential stand-in device (host-logic tests only)."""
    if kind not in _fqg:
        if kind == "sim":
            d = os.path.join(ROOT, "tests", "sim")
            subprocess.check_call(["make", "-C", d], stdout=subprocess.DEVNULL)
            so = os.path.join(d, "libfastq_sim.so")
        else:
            so = os.path.join(ROOT, "fastq_utils_b200", "libfastq_gpu.so")
        lib = ctypes.CDLL(so)
        lib.fqg_fastq_info_mem.restype = ctypes.c_int
        lib.fqg_fastq_info_mem.argtypes = [ctypes.c_int, ctypes.POINTER(ctypes.c_char_p), ctypes.c_char_p, ctypes.c_size_t,
                                           ctypes.c_char_p, ctypes.c_size_t, ctypes.c_int, ctypes.c_size_t,
                                           ctypes.POINTER(_Transcript)]
        lib.fqg_transcript_free.argtypes = [ctypes.POINTER(_Transcript)]
        lib.fqg_reader_tool_mem.restype = ctypes.c_int
        lib.fqg_reader_tool_mem.argtypes = [ctypes.c_int, ctypes.POINTER(ctypes.c_char_p), ctypes.c_char_p, ctypes.c_size_t,
                                            ctypes.c_int, ctypes.c_size_t, ctypes.POINTER(_Transcript)]
        _fqg[kind] = lib
    return _fqg[kind]


def fqg_run(argv, data1=None, data2=None, chunk=0, kind="gpu"):
    """fastq_info through the C ABI on in-memory streams → (rc, stdout, stderr) as latin-1 text."""
    lib = fqg_lib(kind)
    full = [b"fastq_info"] + [a.encode("latin-1") for a in argv]
    arr = (ctypes.c_char_p * (len(full) + 1))(*full, None)
    tr = _Transcript()
    unopenable = ctypes.c_size_t(-1).value
    st = lib.fqg_fastq_info_mem(len(full), arr, data1, len(data1) if data1 is not None else unopenable,
                                data2, len(data2) if data2 is not None else unopenable, 0, chunk, ctypes.byref(tr))
    if st != 0:
        raise RuntimeError(f"fqg_fastq_info_mem failed with status {st}")
    out = ctypes.string_at(tr.out, tr.out_len).decode("latin-1")
    err = ctypes.string_at(tr.err, tr.err_len).decode("latin-1")
    rc = tr.rc
    lib.fqg_transcript_free(ctypes.byref(tr))
    return rc, out, err


def fqg_run_files(argv, cwd=GOLDEN, chunk=0, kind="gpu"):
    pos = positional_files(argv)
    datas = []
    for p in pos[:2]:
        path = os.path.join(cwd, p)
        datas.append(read_stream(path) if os.path.isfile(path) else None)
    while len(datas) < 2:
        datas.append(None)
    return fqg_run(argv, datas[0], datas[1], chunk=chunk, kind=kind)


def fqg_reader_tool(tool, argv, data1=None, chunk=0, kind="gpu"):
    """fastq_num_reads / fastq_not_empty through the C ABI on an in-memory stream → (rc, stdout, stderr) as latin-1 text."""
    lib = fqg_lib(kind)
    full = [tool.encode("latin-1")] + [a.encode("latin-1") for a in argv]
    arr = (ctypes.c_char_p * (len(full) + 1))(*full, None)
    tr = _Transcript()
    st = lib.fqg_reader_tool_mem(len(full), arr, data1, len(data1) if data1 is not None else ctypes.c_size_t(-1).value, 0, chunk, ctypes.byref(tr))
    if st != 0:
        raise RuntimeError(f"fqg_reader_tool_mem failed with status {st}")
    out = ctypes.string_at(tr.out, tr.out_len).decode("latin-1")
    err = ctypes.string_at(tr.err, tr.err_len).decode("latin-1")
    rc = tr.rc
    lib.fqg_transcript_free(ctypes.byref(tr))
    return rc, out, err


def fqg_reader_tool_files(tool, argv, cwd=GOLDEN, chunk=0, kind="gpu"):
    data = None
    if len(argv) >= 1:
        path = os.path.join(cwd, argv[0])
        data = read_stream(path) if os.path.isfile(path) else None
    return fqg_reader_tool(tool, argv, data, chunk=chunk, kind=kind)


def reader_golden():
    with open(os.path.join(GOLDEN, "reader_transcripts.json")) as fh:
        return json.load(fh)


def ref_reader_tool(tool, data, name="a.fq"):
    """The unmodified reference tool (oracle/_ref/<tool>) on a temporary plain-text file → (rc, stdout, stderr)."""
    import tempfile
    with tempfile.TemporaryDirectory() as d:
        with open(os.path.join(d, name), "wb") as fh:
            fh.write(data)
        p = subprocess.run([os.path.join(ROOT, "oracle", "_ref", tool), name], cwd=d, capture_output=True)
    return p.returncode, p.stdout.decode("latin-1"), p.stderr.decode("latin-1")


# ---------------------------------------------------------------------------------------------- streamed entry point
class _StreamIO(ctypes.Structure):
    _fields_ = [("user", ctypes.c_void_p),
                ("open", ctypes.CFUNCTYPE(ctypes.c_void_p, ctypes.c_void_p, ctypes.c_char_p)),
                ("read", ctypes.CFUNCTYPE(ctypes.c_long, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_size_t)),
                ("close", ctypes.CFUNCTYPE(None, ctypes.c_void_p, ctypes.c_void_p))]


def fqg_run_stream(argv, files, piece=0, kind="gpu", max_read=None):
    """fastq_info through fqg_fastq_info_stream: `files` maps operand names to inflated bytes (a missing name cannot be opened); the
    library asks for the operands it wants → (rc, stdout, stderr, names opened in order)."""
    lib = fqg_lib(kind)
    lib.fqg_fastq_info_stream.restype = ctypes.c_int
    lib.fqg_fastq_info_stream.argtypes = [ctypes.c_int, ctypes.POINTER(ctypes.c_char_p), ctypes.POINTER(_StreamIO), ctypes.c_int, ctypes.c_size_t, ctypes.POINTER(_Transcript)]
    opened, state = [], {}

    def _open(user, name):
        nm = name.decode("latin-1")
        opened.append(nm)
        if nm not in files:
            return None
        h = len(state) + 1
        state[h] = [files[nm], 0]
        return h

    def _read(user, h, buf, cap):
        data, pos = state[h]
        k = min(cap, len(data) - pos, max_read or cap)
        ctypes.memmove(buf, data[pos:pos + k], k)
        state[h][1] = pos + k
        return k

    def _close(user, h):
        state.pop(h, None)
    io = _StreamIO(None, _StreamIO._fields_[1][1](_open), _StreamIO._fields_[2][1](_read), _StreamIO._fields_[3][1](_close))
    full = [b"fastq_info"] + [a.encode("latin-1") for a in argv]
    arr = (ctypes.c_char_p * (len(full) + 1))(*full, None)
    tr = _Transcript()
    st = lib.fqg_fastq_info_stream(len(full), arr, ctypes.byref(io), 0, piece, ctypes.byref(tr))
    if st != 0:
        raise RuntimeError(f"fqg_fastq_info_stream failed with status {st}")
    out = ctypes.string_at(tr.out, tr.out_len).decode("latin-1")
    err = ctypes.string_at(tr.err, tr.err_len).decode("latin-1")
    rc = tr.rc
    lib.fqg_transcript_free(ctypes.byref(tr))
    return rc, out, err, opened
