"""Differential fuzz: oracle (CPU restatement) vs the unmodified reference binary (oracle/_ref/fastq_info).

Seeded mutations of small FASTQ streams in all five modes; transcripts must be byte-identical.  Where the reference binary is not
built, the oracle is compared with the reference's transcripts of the same seeds (tests/golden/fuzz/oracle_fuzz.json).
"""
import os
import random
import tempfile

import pytest

from _util import fuzz_golden, have_ref, oracle_run, ref_run

NAMES = [
    lambda i, m: f"r{i}/{m}",
    lambda i, m: f"M01:5:FC:1:1101:{1000 + i}:{2000 + i} {m}:N:0:ACGT",
    lambda i, m: f"{i + 1}",
    lambda i, m: f"read{i}_x extra words",
    lambda i, m: f"S4_01:4:1:{i}:16/{m} {m}:Y:0:0",
    lambda i, m: f"ab{i}:{m}",
]


def make_file(rng, n, style, mate, seqlen=(1, 40), qual=(35, 74)):
    recs = []
    for i in range(n):
        L = rng.randint(*seqlen)
        seq = "".join(rng.choice("ACGTN") for _ in range(L))
        q = "".join(chr(rng.randint(*qual)) for _ in range(L))
        recs.append([f"@{NAMES[style](i, mate)}", seq, "+", q])
    return recs


def mutate(rng, recs):
    if not recs:
        return
    k = rng.randrange(len(recs))
    r = recs[k]
    op = rng.randrange(22)
    if op == 0: r[1] = r[1][:len(r[1]) // 2] + rng.choice("XxZ-*+@ \t") + r[1][len(r[1]) // 2 + 1:]
    elif op == 1: r[3] = r[3] + "I"
    elif op == 2: r[3] = r[3][:-1]
    elif op == 3: r[0] = r[0][1:]
    elif op == 4: r[2] = "+" + r[0][1:]
    elif op == 5: r[2] = "+" + r[0][1:] + "x"
    elif op == 6: r[2] = "-"
    elif op == 7: recs.append(list(recs[rng.randrange(len(recs))]))
    elif op == 8: r[1] = r[1].replace("T", "U")
    elif op == 9: r[1] = r[1] + "TU"
    elif op == 10: r[1] = r[1] + "UT"
    elif op == 11: r[1] = ""
    elif op == 12: r[0] = "@"
    elif op == 13: r[3] = r[3][:1] + "\x00" + r[3][2:]
    elif op == 14: r[1] = r[1][:1] + "\x00" + r[1][2:]
    elif op == 15: r[1] = r[1][:1] + "\r" + r[1][2:]
    elif op == 16: r[3] = "".join(chr(min(255, ord(c) + rng.choice([0, 30, 60, 100]))) for c in r[3])
    elif op == 17: r[1] = r[1].lower()
    elif op == 18: r[1] = "".join(rng.choice("0123.") for _ in r[1]); r[3] = r[3][:max(0, len(r[1]) - rng.randint(0, 1))]
    elif op == 19: recs[0][1] = "T" + "".join(rng.choice("0123") for _ in recs[0][1]); recs[0][3] = "I" * (len(recs[0][1]) - 1)
    elif op == 20: recs.pop(k)
    elif op == 21: r[0] = r[0] + " "


def render(rng, recs, style):
    nl = "\r\n" if style == "crlf" else "\n"
    s = "".join(l + nl for r in recs for l in r)
    t = rng.randrange(12)
    if t == 0: s = s[:-1]
    elif t == 1: s = s[:rng.randrange(len(s) + 1)]
    elif t == 2: s = s + "\n"
    elif t == 3 and recs: s = s + recs[0][0] + "\n"
    return s.encode("latin-1")


def fuzz_case(seed):
    """seed -> (argv, file a.fq, file b.fq or None)"""
    rng = random.Random(seed)
    style = rng.randrange(len(NAMES))
    n = rng.choice([0, 1, 2, 3, 5, 8, 13])
    mode = rng.choice(["single", "single_r", "pe", "pair", "pair_rs", "pair_s", "pair_r"])
    r1 = make_file(rng, n, style, 1)
    two = mode.startswith("pair")
    r2 = make_file(rng, n, style, 2) if two else None
    if mode == "pe":
        inter = []
        for a, b in zip(r1, make_file(rng, n, style, 2)):
            inter += [a, b]
        r1 = inter
    if two and rng.random() < 0.5:
        rng.shuffle(r2)
    for _ in range(rng.choice([0, 0, 1, 1, 2])):
        mutate(rng, r1 if (not two or rng.random() < 0.5) else r2)
    nlstyle = "crlf" if rng.random() < 0.08 else "lf"
    d1 = render(rng, r1, nlstyle)
    d2 = render(rng, r2, nlstyle) if two else None
    argv = {"single": [], "single_r": ["-r"], "pe": [], "pair": [], "pair_rs": ["-r", "-s"], "pair_s": ["-s"], "pair_r": ["-r"]}[mode]
    if rng.random() < 0.2: argv = ["-q"] + argv
    if rng.random() < 0.2: argv = ["-e"] + argv
    argv = argv + ["a.fq"]
    if two:
        argv.append("b.fq")
    if mode == "pe":
        argv.append("pe")
    return argv, d1, d2


def reference_result(seed):
    """the reference binary on the files of fuzz_case(seed) -> (rc, stdout, stderr)"""
    argv, d1, d2 = fuzz_case(seed)
    with tempfile.TemporaryDirectory() as d:
        open(os.path.join(d, "a.fq"), "wb").write(d1)
        if d2 is not None:
            open(os.path.join(d, "b.fq"), "wb").write(d2)
        return ref_run(argv, cwd=d)


SEEDS = range(240)


@pytest.mark.parametrize("seed", SEEDS)
def test_fuzz_against_reference_binary(seed):
    argv, d1, d2 = fuzz_case(seed)
    want = reference_result(seed) if have_ref() else tuple(fuzz_golden("oracle_fuzz")[str(seed)])
    got = oracle_run(argv, d1, d2)
    assert got == want, (argv, d1, d2)
