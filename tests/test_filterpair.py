"""fastq_filterpair (src/fastq_filterpair.c) behind fqg_filterpair_mem: file 1 through the index loop (validation, duplicate check), the
records of both files delimited by the reader loop, names hashed and looked up in the index on the device, the reference's sequential
bookkeeping (lookup-then-delete, seek counters, where its last loop starts) replayed on the host.  Against the committed transcripts of the
reference's own binary (exit status, stdout, stderr, the three inflated output files) and, fuzzed, against the binary (where it is
not built, against its stored results for the same seeds)."""
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
from make_filterpair_golden import big_pair  # noqa: E402

CASES = json.load(open(os.path.join(GOLDEN, "filterpair_transcripts.json")))
REF = os.path.join(ROOT, "oracle", "_ref", "fastq_filterpair")
_libs, _big = {}, {}


def _lib(kind):
    if kind == "gpu":
        return None
    if "sim" not in _libs:
        from fastq_utils_b200 import api
        d = os.path.join(ROOT, "tests", "sim")
        subprocess.check_call(["make", "-C", d], stdout=subprocess.DEVNULL)
        _libs["sim"] = api.bind(ctypes.CDLL(os.path.join(d, "libfastq_sim.so")))
    return _libs["sim"]


def _data(w):
    if w in ("pair_inputs/big_1.fq", "pair_inputs/big_2.fq"):
        if not _big:
            a, b = big_pair()
            _big["pair_inputs/big_1.fq"], _big["pair_inputs/big_2.fq"] = a.encode("latin-1"), b.encode("latin-1")
        return _big[w]
    p = os.path.join(GOLDEN, w)
    return read_stream(p) if os.path.isfile(p) else None


def _same(text, c, key):
    if key in c:
        return text.decode("latin-1") == c[key]
    return (len(text), hashlib.sha256(text).hexdigest()) == (c[key + "_len"], c[key + "_sha256"])


def _check(c, kind):
    from fastq_utils_b200 import api
    argv = c["argv"]
    d1 = _data(argv[0]) if len(argv) >= 1 else None
    d2 = _data(argv[1]) if len(argv) >= 2 else None
    rc, out, err, created, bufs = api.filterpair(argv, d1, d2, _lib=_lib(kind))
    assert rc == c["rc"] and out == c["stdout"], (argv, rc, err[-300:])
    assert _same(err.encode("latin-1"), c, "stderr"), (argv, err[-400:], c.get("stderr", "")[-400:])
    assert created == c["created"], argv
    if "\nPaired: " in err and ("out0" in c or "out0_len" in c):  # the reference closed its three files
        for k in range(3):
            assert _same(bufs[k], c, f"out{k}"), (argv, k)


# (every pair of different files; of the runs of a corpus file against itself every second one)
@pytest.mark.parametrize("idx", [i for i, c in enumerate(CASES) if len(c["argv"]) < 2 or c["argv"][0] != c["argv"][1] or (i // 2) % 2 == 0])
def test_sim_filterpair_matches_reference(idx):
    _check(CASES[idx], "sim")


@pytest.mark.gpu
@pytest.mark.parametrize("idx", range(0, len(CASES), 2))
def test_gpu_filterpair_matches_reference(idx):
    _check(CASES[idx], "gpu")


def _fuzz_pair(rng):
    n = rng.choice([0, 1, 3, 12, 40])
    fmt = rng.choice(["slash", "casava", "plain"])

    def name(i, mate):
        return f"q{i}/{mate}" if fmt == "slash" else f"q{i} {mate}:N:0:AC" if fmt == "casava" else f"q{i}_{mate}"
    rec = lambda nm, L: f"@{nm}\n{''.join(rng.choice('ACGTN') for _ in range(L))}\n+\n{'I' * L}\n"  # noqa: E731
    f1 = [rec(name(i, 1), rng.choice([1, 8, 30])) for i in range(n) if rng.random() < 0.9]
    ids = [i for i in range(n) if rng.random() < 0.85] + [rng.randrange(n + 3) for _ in range(rng.choice([0, 0, 2]))]
    if rng.random() < 0.5:
        rng.shuffle(ids)
    f2 = [rec(name(i, 2), rng.choice([1, 8, 30])) for i in ids]
    a, b = "".join(f1).encode(), "".join(f2).encode()
    m = rng.random()
    if m < 0.15 and b:
        b = b[:rng.randrange(len(b))]
    elif m < 0.25 and b:
        x = bytearray(b)
        x[rng.randrange(len(x))] = rng.choice([0, ord("X"), ord("\n")])
        b = bytes(x)
    elif m < 0.32 and a:
        x = bytearray(a)
        x[rng.randrange(len(x))] = rng.choice([0, ord("X"), ord("\n")])
        a = bytes(x)
    return a, b


def fuzz_runs(seed):
    """seed -> 8 (argv, contents of a.fq, contents of b.fq)"""
    rng = random.Random(seed)
    runs = []
    for _ in range(8):  # (the reference takes 1.5 s per run: it clears a table of 100 000 001 buckets)
        a, b = _fuzz_pair(rng)
        runs.append((["a.fq", "b.fq", "p1.gz", "p2.gz", "up.gz"] + rng.choice([[], [], ["sorted"]]), a, b))
    return runs


def _digest(b):
    return [len(b), hashlib.sha256(b).hexdigest()]


def reference_result(seed):
    """the reference binary on fuzz_runs(seed) -> per run [rc, stdout, stderr, created, (length, sha256) of the three inflated outputs
    when it reported its counts, else None]"""
    out = []
    with tempfile.TemporaryDirectory() as d:
        for argv, a, b in fuzz_runs(seed):
            for nm, dta in (("a.fq", a), ("b.fq", b)):
                with open(os.path.join(d, nm), "wb") as fh:
                    fh.write(dta)
            for o in argv[2:5]:
                if os.path.exists(os.path.join(d, o)):
                    os.unlink(os.path.join(d, o))
            pr = subprocess.run([REF] + argv, cwd=d, capture_output=True)
            err = pr.stderr.decode("latin-1")
            outs = [_digest(gzip.open(os.path.join(d, o), "rb").read()) for o in argv[2:5]] if "\nPaired: " in err else None
            out.append([pr.returncode, pr.stdout.decode("latin-1"), err, all(os.path.exists(os.path.join(d, o)) for o in argv[2:5]), outs])
    return out


def _against_binary(seed, kind):
    """against the reference binary where it is built, else against its stored results for the same seed"""
    from fastq_utils_b200 import api
    wants = reference_result(seed) if os.path.exists(REF) else fuzz_golden("filterpair_fuzz")[str(seed)]
    for (argv, a, b), want in zip(fuzz_runs(seed), wants):
        rc, out, err, created, bufs = api.filterpair(argv, a, b, _lib=_lib(kind))
        assert [rc, out, err] == want[:3], (argv, a, b)
        assert created == want[3]
        if want[4] is not None:
            assert [_digest(x) for x in bufs] == want[4], (argv, a, b)


SEEDS_SIM, SEEDS_GPU = range(3), range(100, 102)


@pytest.mark.parametrize("seed", SEEDS_SIM)
def test_sim_filterpair_fuzz_against_binary(seed):
    _against_binary(seed, "sim")


@pytest.mark.gpu
@pytest.mark.parametrize("seed", SEEDS_GPU)
def test_gpu_filterpair_fuzz_against_binary(seed):
    _against_binary(seed, "gpu")
