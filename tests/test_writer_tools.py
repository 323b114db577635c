"""fastq_truncate and fastq_filter_n (src/fastq_truncate.c, src/fastq_filter_n.c) behind fqg_reader_tool_mem: records delimited on the
device by the reader loop, fastq_filter_n's N count evaluated there, the chosen records written as the reference writes them (`%s` of
the four line buffers).  Against the committed transcripts of the reference's own binaries and, fuzzed, against the binaries."""
import hashlib
import json
import os
import random
import subprocess
import tempfile

import pytest

from _util import GOLDEN, ROOT, fqg_reader_tool, fuzz_golden, have_ref, read_stream

CASES = json.load(open(os.path.join(GOLDEN, "writer_transcripts.json")))


def _run(c, kind):
    data = None
    if c["tool"] == "fastq_filter_n" and "--" in c["argv"]:  # the reference takes argv[1 + nopt] for the file: "--" itself, which cannot be opened
        return fqg_reader_tool(c["tool"], c["argv"], None, kind=kind)
    for w in c["argv"]:
        p = os.path.join(GOLDEN, w)
        if w.startswith("inputs/") and os.path.isfile(p):
            data = read_stream(p)
            break
    return fqg_reader_tool(c["tool"], c["argv"], data, kind=kind)


def _check(c, got):
    assert got[0] == c["rc"] and got[2] == c["stderr"], (c["tool"], c["argv"], got[0], got[2][-300:], c["stderr"][-300:])
    if "stdout" in c:
        assert got[1] == c["stdout"], (c["tool"], c["argv"])
    else:
        b = got[1].encode("latin-1")
        assert (len(b), hashlib.sha256(b).hexdigest()) == (c["stdout_len"], c["stdout_sha256"]), (c["tool"], c["argv"])


@pytest.mark.parametrize("idx", range(len(CASES)))
def test_sim_writer_tool_matches_reference(idx):
    _check(CASES[idx], _run(CASES[idx], "sim"))


@pytest.mark.parametrize("window", [300, 4096])
@pytest.mark.parametrize("idx", range(0, len(CASES), 37))
def test_sim_writer_tool_in_small_windows(idx, window, monkeypatch):
    """streams above the size of a chunk are taken in windows that start at record starts (FQG_TOOL_WINDOW_BYTES shrinks them): a
    record cut by a window, a window without a whole record, a broken record in the middle of the stream"""
    monkeypatch.setenv("FQG_TOOL_WINDOW_BYTES", str(window))
    _check(CASES[idx], _run(CASES[idx], "sim"))


@pytest.mark.gpu
@pytest.mark.parametrize("idx", range(0, len(CASES), 2))
def test_gpu_writer_tool_matches_reference(idx):
    _check(CASES[idx], _run(CASES[idx], "gpu"))


def _fuzz_file(rng):
    recs = []
    for i in range(rng.choice([0, 1, 2, 7, 30])):
        L = rng.choice([1, 4, 20, 60])
        seq = "".join(rng.choice("ACGTNn" if rng.random() < 0.5 else "ACGT") for _ in range(L))
        recs.append(f"@r{i} x\n{seq}\n+\n{'I' * L}\n")
    data = "".join(recs).encode()
    m = rng.random()
    if m < 0.2 and data:
        data = data[:rng.randrange(len(data))]           # cut anywhere: a truncated record, or a last line without LF
    elif m < 0.3 and data:
        k = rng.randrange(len(data)); data = data[:k] + b"\x00" + data[k + 1:]  # a NUL: `%s` stops there; a NUL-led header ends the file
    elif m < 0.35:
        data += b"@long " + b"x" * 1200 + b"\nACGT\n+\nIIII\n"   # a header line gzgets splits
    return data


def fuzz_case(seed):
    """seed -> (tool, argv, contents of a.fq)"""
    rng = random.Random(4200 + seed)
    data = _fuzz_file(rng)
    tool, argv = ("fastq_truncate", ["a.fq", str(rng.choice([0, 1, 2, 5, 100, -3]))]) if seed % 2 else ("fastq_filter_n", rng.choice([[], ["-n", "0"], ["-n", "20"], ["-n", "60"]]) + ["a.fq"])
    return tool, argv, data


def reference_result(seed):
    """the reference tool on fuzz_case(seed) -> (rc, stdout, stderr)"""
    tool, argv, data = fuzz_case(seed)
    with tempfile.TemporaryDirectory() as d:
        open(os.path.join(d, "a.fq"), "wb").write(data)
        p = subprocess.run([os.path.join(ROOT, "oracle", "_ref", tool)] + argv, cwd=d, capture_output=True)
    return p.returncode, p.stdout.decode("latin-1"), p.stderr.decode("latin-1")


SEEDS = range(120)


@pytest.mark.parametrize("seed", SEEDS)
def test_sim_writer_tools_fuzz_against_reference(seed):
    """against the reference tools where they are built, else against their stored transcripts"""
    tool, argv, data = fuzz_case(seed)
    want = reference_result(seed) if have_ref("fastq_truncate") else tuple(fuzz_golden("writer_fuzz")[str(seed)])
    assert fqg_reader_tool(tool, argv, data, kind="sim") == want, (tool, argv, data)
