"""The reader-style tools of SURVEY.md §8f-2 (fastq_num_reads, fastq_not_empty) through FQG_MODE_READER: transcripts of the
UNMODIFIED reference tools (tests/golden/reader_transcripts.json, made by tests/golden/make_reader_golden.py from oracle/_ref/)
against the C ABI — on the stand-in device here, on the real kernels in the -m gpu cases."""
import os
import random

import pytest

from _util import ROOT, fqg_reader_tool, fqg_reader_tool_files, fuzz_golden, have_ref, reader_golden, ref_reader_tool
from test_oracle_fuzz import NAMES, make_file, mutate, render

CASES = reader_golden()


def _check(c, kind, chunk):
    got = fqg_reader_tool_files(c["tool"], c["argv"], chunk=chunk, kind=kind)
    assert got == (c["rc"], c["stdout"], c["stderr"]), (c["tool"], c["argv"], chunk)


@pytest.mark.parametrize("idx", range(len(CASES)))
def test_sim_reader_tools_match_reference(idx):
    _check(CASES[idx], "sim", [0, 64, 1000, 4096][idx % 4] if idx % 2 == 0 else 0)


def _fuzz_file(seed):
    rng = random.Random(77_000 + seed)
    recs = make_file(rng, rng.choice([0, 1, 2, 3, 5, 8, 13, 40]), rng.randrange(len(NAMES)), 1)
    for _ in range(rng.choice([0, 0, 1, 1, 2, 3])):
        mutate(rng, recs)
    data = render(rng, recs, rng.choice(["lf", "lf", "lf", "crlf"]))
    if rng.random() < 0.15 and data:  # a NUL-led line somewhere: the reader stops there quietly when it is a header line
        k = rng.randrange(len(data))
        k = data.rfind(b"\n", 0, k) + 1
        data = data[:k] + b"\x00" + data[k:]
    return data


FUZZ_TOOLS = ("fastq_num_reads", "fastq_not_empty")


def reference_result(seed):
    """the reference tools on _fuzz_file(seed) -> [(rc, stdout, stderr) of each of FUZZ_TOOLS]"""
    data = _fuzz_file(seed)
    return [ref_reader_tool(tool, data) for tool in FUZZ_TOOLS]


SEEDS = range(150)


@pytest.mark.parametrize("seed", SEEDS)
def test_sim_reader_tools_fuzz_against_reference(seed):
    """against the reference tools where they are built (make -C oracle ref-tools), else against their stored transcripts"""
    data = _fuzz_file(seed)
    wants = reference_result(seed) if have_ref("fastq_num_reads") else [tuple(w) for w in fuzz_golden("reader_fuzz")[str(seed)]]
    for tool, want in zip(FUZZ_TOOLS, wants):
        got = fqg_reader_tool(tool, ["a.fq"], data, chunk=[0, 0, 37, 512][seed % 4], kind="sim")
        assert got == want, (tool, seed, data[:200])


@pytest.mark.gpu
@pytest.mark.parametrize("idx", range(0, len(CASES), 2))
def test_gpu_reader_tools_match_reference(idx):
    _check(CASES[idx], "gpu", [0, 4096][idx % 4 == 0])


@pytest.mark.gpu
def test_gpu_reader_tools_count_large_streams():
    """A stream large enough for the clean-data pass (several chunks), clean and with contents no validator would accept: the
    count is the number of four-line records either way."""
    import torch
    import fastq_utils_b200 as fq
    rb = fq.illumina_record_bytes()
    n = 300_000
    t = torch.zeros(n * rb + 64, dtype=torch.uint8, device="cuda")
    fq.synth_illumina(t, 0, n, seed=42, mate=1, stream=torch.cuda.current_stream().cuda_stream)
    torch.cuda.synchronize()
    data = bytearray(t[:n * rb].cpu().numpy().tobytes())
    assert fqg_reader_tool("fastq_num_reads", ["a.fq"], bytes(data), chunk=32 << 20) == (0, f"{n}\n", "fastq_utils 0.25.3\n")
    data[123_456 * rb + 80] = ord("*")       # an invalid base
    data[200_000 * rb] = ord("X")            # a header that does not start with '@'
    assert fqg_reader_tool("fastq_num_reads", ["a.fq"], bytes(data), chunk=32 << 20) == (0, f"{n}\n", "fastq_utils 0.25.3\n")
    assert fqg_reader_tool("fastq_not_empty", ["a.fq"], bytes(data)) == (0, "", "")
    cut = bytes(data[:250_000 * rb + 100])   # the last record is cut inside its sequence line
    assert fqg_reader_tool("fastq_num_reads", ["a.fq"], cut) == (1, "", f"fastq_utils 0.25.3\n\nERROR: Error in file a.fq: line {4 * 250_000}: file truncated\n")


def test_python_binding_of_the_reader_tools(tmp_path):
    """fastq_utils_b200.reader_tool and FastqInfo(MODE_READER) (api.py) over the stand-in device, in a process of its own (the
    stand-in is put behind the binding by tests/sim_lib.py)."""
    import subprocess
    import sys
    code = (
        "import fastq_utils_b200 as fq\n"
        "from sim_lib import use_sim_library; use_sim_library()\n"
        "d = b''.join(b'@r%d\\nACGT\\n+\\nIIII\\n' % i for i in range(7)) + b'@x\\nAC*T\\n+\\nII\\n'\n"  # the last record would not validate
        "assert fq.reader_tool('fastq_num_reads', ['a.fq'], d) == (0, '8\\n', 'fastq_utils 0.25.3\\n')\n"
        "assert fq.reader_tool('fastq_not_empty', ['a.fq'], d) == (0, '', '')\n"
        "assert fq.reader_tool('fastq_not_empty', ['a.fq'], b'') == (1, '', '')\n"
        "assert fq.reader_tool('fastq_num_reads', ['a.fq'], None)[0] == 1\n"
        "h = fq.FastqInfo(fq.MODE_READER); h.feed(0, d[:40], last=False); h.feed(0, d[40:], last=True); r = h.finish()\n"
        "assert r.error.code == 0 and r.file[0].n_records == 8, (r.error.code, r.file[0].n_records)\n"
        "n, starts = h.index_records(d, cap=16)\n"  # fqg_index_records: where the four-line records start
        "want = [i for i in range(len(d)) if (i == 0 or d[i - 1] == 10) and d[:i].count(b'\\n') % 4 == 0]\n"
        "assert n == 8 and starts == want[:8], (n, starts, want)\n"
        "assert h.index_records(d[:-1], cap=4) == (8, want[:4]) and h.index_records(d[:-3], cap=0) == (7, [])\n"  # a last line without LF counts
        "print('ok')\n")
    env = dict(os.environ, PYTHONPATH=ROOT + os.pathsep + os.path.join(ROOT, "tests"))
    out = subprocess.run([sys.executable, "-c", code], env=env, capture_output=True, text=True, timeout=120)
    assert out.returncode == 0 and out.stdout.strip() == "ok", out.stderr[-2000:]


@pytest.mark.gpu
def test_gpu_index_records():
    """fqg_index_records on the real scan kernel: record starts of a 50 000-record stream (what fastq_truncate would cut at)."""
    import fastq_utils_b200 as fq
    recs = [b"@r%d\n%s\n+\n%s\n" % (i, b"ACGTN" * (1 + i % 37), b"I" * (5 * (1 + i % 37))) for i in range(50_000)]
    data = b"".join(recs)
    want, off = [], 0
    for r in recs:
        want.append(off)
        off += len(r)
    h = fq.FastqInfo(fq.MODE_SINGLE)
    assert h.index_records(data, cap=len(recs)) == (len(recs), want)
    assert h.index_records(data[:want[40_000] + 5], cap=3) == (40_000, want[:3])  # 160 001 lines: the cut record is not complete
    h.close()
