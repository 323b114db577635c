"""fastq_trim_poly_at (src/fastq_trim_poly_at.c) behind fqg_trim_poly_at_stream: records delimited on the device by the reader loop, the
poly-A / poly-T scans evaluated there, the reference's line-buffer edits replayed on the host.  Against the committed transcripts of the
reference's own binary (exit status, stdout, stderr, inflated output file) and, fuzzed, against the binary (where it is not built,
against its stored results for the same seeds)."""
import ctypes
import gzip
import hashlib
import json
import os
import random
import subprocess
import sys
import tempfile

import pytest

from _util import GOLDEN, ROOT, fuzz_golden, read_stream

sys.path.insert(0, GOLDEN)
from make_trim_golden import poly_100k  # noqa: E402

CASES = json.load(open(os.path.join(GOLDEN, "trim_transcripts.json")))
REF = os.path.join(ROOT, "oracle", "_ref", "fastq_trim_poly_at")
_libs = {}


def _lib(kind):
    """None = the product library (needs a GPU); 'sim' = the same host code over the tests' stand-in device"""
    if kind == "gpu":
        return None
    if "sim" not in _libs:
        from fastq_utils_b200 import api
        d = os.path.join(ROOT, "tests", "sim")
        subprocess.check_call(["make", "-C", d], stdout=subprocess.DEVNULL)
        _libs["sim"] = api.bind(ctypes.CDLL(os.path.join(d, "libfastq_sim.so")))
    return _libs["sim"]


_big = {}


def _files(argv):
    files = {}
    for w in argv:
        w = w.split("=", 1)[-1]
        if w == "trim_inputs/poly_100k.fq":
            if "b" not in _big:
                _big["b"] = poly_100k().encode("latin-1")
            files[w] = _big["b"]
        elif (w.startswith("inputs/") or w.startswith("trim_inputs/")) and os.path.isfile(os.path.join(GOLDEN, w)):
            files[w] = read_stream(os.path.join(GOLDEN, w))
    return files


def _run(c, kind):
    from fastq_utils_b200 import api
    return api.trim_poly_at(c["argv"], files=_files(c["argv"]), _lib=_lib(kind))


def _check(c, got):
    rc, out, err, oname, data = got
    assert rc == c["rc"] and err == c["stderr"] and out == c["stdout"], (c["argv"], rc, err[-300:], c["stderr"][-300:])
    assert (oname is not None) == c["created"], c["argv"]
    if "outfile" in c:
        assert data.decode("latin-1") == c["outfile"], c["argv"]
    elif "outfile_len" in c:
        assert (len(data), hashlib.sha256(data).hexdigest()) == (c["outfile_len"], c["outfile_sha256"]), c["argv"]


# (the hand-made files and option cases all; every second run over the validation corpus, whose files have little to trim)
@pytest.mark.parametrize("idx", [i for i, c in enumerate(CASES) if i % 2 == 0 or not any(w.startswith("inputs/") for w in c["argv"])])
def test_sim_trim_matches_reference(idx):
    _check(CASES[idx], _run(CASES[idx], "sim"))


@pytest.mark.parametrize("idx", [i for i, c in enumerate(CASES) if "trim_inputs/" in " ".join(c["argv"]) and "poly_100k" not in " ".join(c["argv"])][::2])
def test_sim_trim_in_small_windows(idx, monkeypatch):
    """the stream in windows of 256 bytes: the line buffers' history (poly_shortqual.fq) must survive the window boundaries"""
    monkeypatch.setenv("FQG_TOOL_WINDOW_BYTES", "256")
    _check(CASES[idx], _run(CASES[idx], "sim"))


@pytest.mark.gpu
@pytest.mark.parametrize("idx", range(0, len(CASES), 3))
def test_gpu_trim_matches_reference(idx):
    _check(CASES[idx], _run(CASES[idx], "gpu"))


def _fuzz_file(rng):
    recs = []
    for i in range(rng.choice([0, 1, 2, 7, 30])):
        L = rng.choice([1, 4, 20, 60])
        k = rng.choice([0, 2, 9, 10, 15])
        core = "".join(rng.choice("ACGTNn") for _ in range(L))
        m = rng.random()
        seq = core + "".join(rng.choice("AaNn") for _ in range(k)) if m < 0.4 else "".join(rng.choice("TtNn") for _ in range(k)) + core if m < 0.8 else core
        ql = len(seq) if rng.random() < 0.85 else rng.randrange(0, len(seq) + 5)
        eol = "\r\n" if rng.random() < 0.05 else "\n"
        recs.append(f"@r{i} x{eol}{seq}{eol}+{eol}{'I' * ql}{eol}")
    data = "".join(recs).encode()
    m = rng.random()
    if m < 0.2 and data:
        data = data[:rng.randrange(len(data))]           # cut anywhere: a truncated record, or a last line without LF
    elif m < 0.3 and data:
        b = bytearray(data)
        b[rng.randrange(len(b))] = 0                     # a NUL byte: gzgets keeps it, strlen stops there
        data = bytes(b)
    return data


def fuzz_runs(seed):
    """seed -> 40 (argv, contents of f.fq)"""
    rng = random.Random(seed)
    runs = []
    for _ in range(40):
        data = _fuzz_file(rng)
        opts = rng.choice([[], ["--min_poly_at_len", "2"], ["--min_poly_at_len", "9", "--min_len", "0"], ["--min_len", "30"], ["--min_poly_at_len", "1", "--min_len", "3"]])
        runs.append((opts + ["--file", "f.fq", "--outfile", "o.gz"], data))
    return runs


def _digest(b):
    return [len(b), hashlib.sha256(b).hexdigest()]


def reference_result(seed):
    """the reference binary on fuzz_runs(seed) -> per run [rc, stdout, stderr, (length, sha256) of the inflated output or None]"""
    out = []
    with tempfile.TemporaryDirectory() as d:
        o = os.path.join(d, "o.gz")
        for argv, data in fuzz_runs(seed):
            with open(os.path.join(d, "f.fq"), "wb") as fh:
                fh.write(data)
            if os.path.exists(o):
                os.unlink(o)
            pr = subprocess.run([REF] + argv, cwd=d, capture_output=True)
            out.append([pr.returncode, pr.stdout.decode("latin-1"), pr.stderr.decode("latin-1"), _digest(gzip.open(o, "rb").read()) if pr.returncode == 0 else None])
    return out


def _against_binary(seed, kind):
    """against the reference binary where it is built, else against its stored results for the same seed"""
    from fastq_utils_b200 import api
    wants = reference_result(seed) if os.path.exists(REF) else fuzz_golden("trim_fuzz")[str(seed)]
    for (argv, data), want in zip(fuzz_runs(seed), wants):
        got = api.trim_poly_at(argv, files={"f.fq": data}, _lib=_lib(kind))
        assert [got[0], got[1], got[2]] == want[:3], (argv, data)
        if want[0] == 0:
            assert _digest(got[4]) == want[3], (argv, data)


SEEDS_SIM, SEEDS_GPU = range(12), range(100, 104)


@pytest.mark.parametrize("seed", SEEDS_SIM)
def test_sim_trim_fuzz_against_binary(seed):
    _against_binary(seed, "sim")


@pytest.mark.gpu
@pytest.mark.parametrize("seed", SEEDS_GPU)
def test_gpu_trim_fuzz_against_binary(seed):
    _against_binary(seed, "gpu")
