"""fqg_fastq_info_stream (what the CLI calls): the library picks the file operands the way the reference's main() does, opens them
through the caller's callback in the reference's order and reads them piece by piece on a helper thread.  Checked against the
committed transcripts of the reference binary and, for the operand quirks, against the binary itself."""
import os
import random
import tempfile

import pytest

from _util import GOLDEN, fqg_run_stream, fuzz_golden, golden_transcripts, have_ref, positional_files, read_stream, ref_run

CASES = golden_transcripts()


def _files_of(argv):
    files = {}
    for w in argv:
        p = os.path.join(GOLDEN, w)
        if os.path.isfile(p):
            files[w] = read_stream(p)
    return files


@pytest.mark.parametrize("idx", range(0, len(CASES), 3))
def test_sim_stream_matches_reference_transcript(idx):
    c = CASES[idx]
    piece = [0, 4096, 1 << 16, 300][idx % 4]
    got = fqg_run_stream(c["argv"], _files_of(c["argv"]), piece=piece, kind="sim", max_read=[None, 1000, 17][idx % 3])
    assert got[:3] == (c["rc"], c["stdout"], c["stderr"]), (c["argv"], piece)


OPERAND_ARGVS = [["-rs", "a.fq", "b.fq"], ["--", "a.fq"], ["-r", "--", "a.fq"], ["a.fq", "-r"], ["-s", "a.fq", "b.fq"], ["-e", "a.fq", "b.fq", "pe"],
                 ["-r", "-s", "a.fq", "nope.fq"], ["nope.fq", "b.fq"], ["a.fq", "nope.fq"], ["-q", "-e", "b.fq"]]
OPERAND_A = "".join(f"@r{i}/1\nACGT\n+\nIIII\n" for i in range(3)).encode()
OPERAND_B = "".join(f"@r{i}/2\nTTTT\n+\nFFFF\n" for i in range(2)).encode()


def reference_result(argv):
    """the reference binary with files a.fq and b.fq of OPERAND_A / OPERAND_B -> (rc, stdout, stderr)"""
    with tempfile.TemporaryDirectory() as d:
        open(os.path.join(d, "a.fq"), "wb").write(OPERAND_A)
        open(os.path.join(d, "b.fq"), "wb").write(OPERAND_B)
        return ref_run(argv, cwd=d)


@pytest.mark.parametrize("argv", OPERAND_ARGVS)
def test_sim_operands_like_the_reference(argv):
    """which words the reference treats as file 1 / file 2 (argv[1 + nopt], src/fastq_info.c:258-266): clustered options shift them;
    against the binary where it is built, else against its stored transcripts"""
    want = reference_result(argv) if have_ref() else tuple(fuzz_golden("stream_operands")[" ".join(argv)])
    got = fqg_run_stream(argv, {"a.fq": OPERAND_A, "b.fq": OPERAND_B}, piece=64, kind="sim")
    assert got[:3] == want, (argv, got, want)


@pytest.mark.gpu
@pytest.mark.parametrize("idx", range(0, len(CASES), 9))
def test_gpu_stream_matches_reference_transcript(idx):
    c = CASES[idx]
    got = fqg_run_stream(c["argv"], _files_of(c["argv"]), piece=[0, 1 << 20][idx % 2], kind="gpu")
    assert got[:3] == (c["rc"], c["stdout"], c["stderr"]), c["argv"]
