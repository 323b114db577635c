"""Multi-rank orchestration (fastq_utils_b200/dist.py) on CPU: world_size 2 and 3 under gloo, with the stand-in device.
Byte ranges are cut at arbitrary positions (inside headers, sequences, qualities); the rank-0 transcript must equal the
CPU oracle's for the whole file."""
import json
import os
import random
import subprocess
import sys

import pytest

from _util import GOLDEN, ROOT, oracle_run, read_stream


def _cases():
    rng = random.Random(5)
    files = ["c18_10000_1.fastq.gz", "test_1.fastq.gz", "test_e9.fastq.gz", "test_e3.fastq.gz", "test_21_1.fastq.gz", "test_e5.fastq.gz",
             "casava.1.8_readname_trunc_1.err2.fastq.gz", "edge_dup3.fastq", "edge_crlf.fastq", "edge_lens.fastq", "edge_tail2.fastq", "edge_no_trailing_nl.fastq"]
    cases = []
    for f in files:
        data = read_stream(os.path.join(GOLDEN, "inputs", f))
        for mode in ("index", "single"):
            cases.append({"file": f, "mode": mode, "hex": data.hex(), "cuts": sorted([rng.random(), rng.random()])})
    # synthetic: a duplicate far apart, split anywhere
    recs = [f"@M0:1:FC:1:11:{i}:{i * 7} 1:N:0:AC\n{'ACGTN' * (3 + i % 5)}\n+\n{'F' * (5 * (3 + i % 5))}\n" for i in range(400)]
    recs[390] = recs[17]
    data = "".join(recs).encode()
    for cuts in ([0.1, 0.5], [0.5, 0.97], [0.045, 0.046]):
        cases.append({"file": "synthetic_dup", "mode": "index", "hex": data.hex(), "cuts": cuts})
        cases.append({"file": "synthetic_dup", "mode": "single", "hex": data.hex(), "cuts": cuts})
    # large enough for every rank to guess its line phase from its own plus lines (the speculative feed of dist.py): a clean file, a
    # duplicate (seen only at the owner), an error on one rank only, a file whose ranks all guess wrong-footed ('+name' lines)
    big = [f"@M0:1:FC:1:11:{i}:{i * 7} 1:N:0:AC\n{'ACGTN' * (3 + i % 5)}\n+\n{'F' * (5 * (3 + i % 5))}\n" for i in range(4000)]
    dupb = list(big); dupb[3900] = dupb[17]
    badb = list(big); badb[3000] = badb[3000].replace("ACGTN", "ACXTN", 1)
    plusb = [r.replace("\n+\n", "\n+" + r.split("\n")[0][1:] + "\n") if i % 7 else r for i, r in enumerate(big)]
    for nm, rr in (("big_clean", big), ("big_dup", dupb), ("big_bad", badb), ("big_plusnames", plusb)):
        for mode in ("index", "single"):
            cases.append({"file": nm, "mode": mode, "hex": "".join(rr).encode().hex(), "cuts": [0.31, 0.64]})
    # a NUL-led header line ends the file quietly (src/fastq.c:248): whatever follows — here a broken record, on a later rank — does
    # not exist for the reference; small (exact path) and large enough for the speculative feed
    for nm, rr, at in (("nul_stop_small", recs[:300], 120), ("nul_stop_big", big, 1500)):
        rr = list(rr)
        rr[at] = "\x00" + rr[at]
        rr[at + (len(rr) - at) // 2] = rr[at + (len(rr) - at) // 2].replace("ACGTN", "AC*TN", 1)
        for mode in ("index", "single"):
            cases.append({"file": nm, "mode": mode, "hex": "".join(rr).encode("latin-1").hex(), "cuts": [0.2, 0.55]})
    # ... and with nothing wrong behind it: no rank has an error to report, the count must still end at the NUL
    quiet = list(big)
    quiet[1500] = "\x00" + quiet[1500]
    for mode in ("index", "single"):
        cases.append({"file": "nul_stop_quiet", "mode": mode, "hex": "".join(quiet).encode("latin-1").hex(), "cuts": [0.2, 0.55]})
    # pairs: default two-file mode (index loop + mate loop)
    def pair_case(f1, f2, c1, c2):
        d1, d2 = read_stream(os.path.join(GOLDEN, "inputs", f1)), read_stream(os.path.join(GOLDEN, "inputs", f2))
        return {"file": f1 + "+" + f2, "mode": "pair", "hex": d1.hex(), "hex2": d2.hex(), "cuts": c1, "cuts2": c2}
    for f1, f2 in [("c18_10000_1.fastq.gz", "c18_10000_2.fastq.gz"), ("a_1.fastq.gz", "a_2.fastq.gz"), ("test_21_1.fastq.gz", "test_21_2.fastq.gz"),
                   ("edge_pair_1.fastq", "edge_pair_2_perm.fastq"), ("edge_pair_1.fastq", "edge_pair_2_rep.fastq"), ("edge_pair_1.fastq", "edge_pair_2_short.fastq"),
                   ("edge_pair_1.fastq", "edge_pair_2_bad.fastq"), ("edge_pair_1.fastq", "edge_pair_2_trunc.fastq"), ("casava.1.8_1.fastq.gz", "casava.1.8_2.fastq.gz"),
                   ("test_solid_1.fastq.gz", "test_solid_2.fastq.gz"), ("test_e19_1.fastq.gz", "test_empty.fastq.gz"), ("test_empty.fastq.gz", "test_1.fastq.gz")]:
        cases.append(pair_case(f1, f2, sorted([rng.random(), rng.random()]), sorted([rng.random(), rng.random()])))
    # interleaved files: ranges cut at pair boundaries (eight lines); sorted-pair files: not sharded, gathered on rank 0 (dist.py)
    for f in ("inter.fastq.gz", "edge_il_ok.fastq", "edge_il_odd.fastq", "edge_il_mismatch.fastq", "edge_il_bad_m2.fastq", "edge_il_trunc_m2.fastq",
              "edge_il_bad_m1_mm.fastq", "edge_il_m2_noat.fastq", "c18_10000_1.fastq.gz"):
        data = read_stream(os.path.join(GOLDEN, "inputs", f))
        cases.append({"file": f, "mode": "interleaved", "hex": data.hex(), "cuts": sorted([rng.random(), rng.random()])})
    il = []
    for i in range(3000):
        for m in (1, 2):
            il.append(f"@M0:1:FC:1:11:{i}:{i * 7} {m}:N:0:AC\n{'ACGTN' * (3 + i % 5)}\n+\n{'F' * (5 * (3 + i % 5))}\n")
    mism = list(il); mism[4001] = mism[4001].replace(":2000:", ":2001:", 1)
    badm2 = list(il); badm2[5001] = badm2[5001].replace("ACGTN", "AC*TN", 1)
    badm1 = list(il); badm1[1000] = badm1[1000].replace("ACGTN", "AC*TN", 1); badm1[301] = badm1[301].replace(":150:", ":151:", 1)
    nulm1 = list(il); nulm1[3000] = "\x00" + nulm1[3000]; nulm1[5000] = nulm1[5000].replace("ACGTN", "AC*TN", 1)
    nulm2 = list(il); nulm2[3001] = "\x00" + nulm2[3001]
    for nm, rr in (("il_clean", il), ("il_odd", il[:-1]), ("il_mismatch", mism), ("il_bad_m2", badm2), ("il_bad_m1_after_mismatch", badm1), ("il_nul_m1", nulm1),
                   ("il_nul_m2", nulm2), ("il_cut_tail", ["".join(il)[:-30]])):
        for cuts in ([0.31, 0.64], [0.5003, 0.5004]):
            cases.append({"file": nm, "mode": "interleaved", "hex": "".join(rr).encode("latin-1").hex(), "cuts": cuts})
    for f1, f2 in [("a_1.fastq.gz", "a_2.fastq.gz"), ("edge_pair_1.fastq", "edge_pair_2_perm.fastq"), ("edge_pair_1.fastq", "edge_pair_2_short.fastq"),
                   ("c18_10000_1.fastq.gz", "c18_10000_2.fastq.gz"), ("edge_pair_1.fastq", "edge_pair_2_bad.fastq")]:
        cases.append(dict(pair_case(f1, f2, sorted([rng.random(), rng.random()]), sorted([rng.random(), rng.random()])), mode="sorted"))
    mates = [r.replace(" 1:N", " 2:N") for r in recs]
    mates[17] = recs[17].replace(" 1:N", " 2:N")
    rng.shuffle(mates)
    cases.append({"file": "synthetic_pair_dup", "mode": "pair", "hex": data.hex(), "hex2": "".join(mates).encode().hex(), "cuts": [0.3, 0.6], "cuts2": [0.2, 0.7]})
    clean = [f"@M0:1:FC:1:11:{i}:{i * 7} 1:N:0:AC\n{'ACGTN' * (3 + i % 5)}\n+\n{'F' * (5 * (3 + i % 5))}\n" for i in range(400)]
    m2 = [x.replace(" 1:N", " 2:N") for x in clean]
    rng.shuffle(m2)
    cases.append({"file": "synthetic_pair_ok", "mode": "pair", "hex": "".join(clean).encode().hex(), "hex2": "".join(m2).encode().hex(), "cuts": [0.3, 0.6], "cuts2": [0.2, 0.7]})
    cases.append({"file": "synthetic_pair_missing", "mode": "pair", "hex": "".join(clean).encode().hex(), "hex2": "".join(m2[:-3]).encode().hex(), "cuts": [0.3, 0.6], "cuts2": [0.2, 0.7]})
    cases.append({"file": "synthetic_pair_extra", "mode": "pair", "hex": "".join(clean[:-5]).encode().hex(), "hex2": "".join(m2).encode().hex(), "cuts": [0.5, 0.6], "cuts2": [0.1, 0.7]})
    return cases


# variants of the name routing: pipelined (chunk by chunk through the chunk hook; the default) and the same with tiny chunks so that
# every range takes several routing rounds
VARIANTS = {"pipelined": {}, "small_chunks": {"FQG_MAX_CHUNK_BYTES": "8192"},
            "overflow": {"FQG_TEST_SLOT_CAP": "7", "FQG_MAX_CHUNK_BYTES": "16384"},  # regions of 7 tuples: every big job overflows and is redone exactly
            # the rounds over peer memory as on the GPUs (the stand-in device maps POSIX shared memory between the ranks): copies of
            # packed regions and an overflowing arena
            "peer_copies": {"FQG_P2P": "1", "FQG_MAX_CHUNK_BYTES": "8192"},
            "peer_overflow": {"FQG_P2P": "1", "FQG_TEST_SLOT_CAP": "7", "FQG_MAX_CHUNK_BYTES": "16384"},
            # 12-bit name hashes: different names with EQUAL hashes everywhere.  One-file jobs (tuples only) fall back to the exact path,
            # whose owners compare the bytes and walk on; two-file jobs route the bytes and judge at once
            "weak_hash": {"FQG_TEST_WEAK_HASH": "1"},
            # one runner for all jobs of a mode (a bench loop, a service): the arena of a small job is regrown for a larger one
            "peer_reuse": {"FQG_P2P": "1", "FQG_MAX_CHUNK_BYTES": "8192", "FQG_TEST_REUSE_RUNNER": "1"}}


@pytest.mark.parametrize("world,variant", [(2, "pipelined"), (3, "small_chunks"), (3, "overflow"),
                                           (3, "peer_copies"), (2, "peer_overflow"), (2, "weak_hash"), (2, "peer_reuse")])
def test_sharded_transcripts_match_oracle(tmp_path, world, variant):
    subprocess.check_call(["make", "-C", os.path.join(ROOT, "tests", "sim")], stdout=subprocess.DEVNULL)
    cases = _cases()
    if variant not in ("pipelined", "small_chunks"):  # the variants of the name routing: only the jobs that route names
        cases = [c for c in cases if c["mode"] in ("index", "pair")]
    cin, cout = tmp_path / "cases.json", tmp_path / "out.json"
    json.dump(cases, open(cin, "w"))
    port = 29600 + world + 10 * list(VARIANTS).index(variant)
    env = dict(os.environ, MASTER_ADDR="127.0.0.1", **VARIANTS[variant])
    subprocess.check_call([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={world}", "--master-addr", "127.0.0.1",
                           "--master-port", str(port), os.path.join(ROOT, "tests", "dist_worker.py"), str(cin), str(cout)], env=env, timeout=600)
    res = json.load(open(cout))
    got, rounds = res["transcripts"], res["rounds"]
    assert len(got) == len(cases)
    for c, g in zip(cases, got):
        argv = {"single": ["-r", "a.fq"], "index": ["a.fq"], "pair": ["a.fq", "b.fq"], "interleaved": ["a.fq", "pe"], "sorted": ["-r", "-s", "a.fq", "b.fq"]}[c["mode"]]
        want = oracle_run(argv, bytes.fromhex(c["hex"]), bytes.fromhex(c["hex2"]) if c["mode"] in ("pair", "sorted") else None)
        assert tuple(g) == want, (c["file"], c["mode"], c["cuts"], g)
    # interleaved files were sharded (ranges cut at pair boundaries), sorted pairs gathered on rank 0
    if variant in ("pipelined", "small_chunks"):
        gath = {(c["file"], c["mode"], tuple(c["cuts"])): g for c, g in zip(cases, res["gathered"])}
        assert gath[("il_clean", "interleaved", (0.31, 0.64))] == 0 and gath[("il_mismatch", "interleaved", (0.31, 0.64))] == 0
        assert gath[("il_nul_m1", "interleaved", (0.31, 0.64))] == 1  # (a NUL-led header line: redone on rank 0)
        assert all(g >= 1 for c, g in zip(cases, res["gathered"]) if c["mode"] == "sorted")
    if variant == "peer_reuse":
        assert res["arena_regrown"] >= 2  # the reused runner replaced its arena by a larger one (unmap, free, allocate, map again)
    # the routing under test was really taken: the clean big file goes through the chunk hook, in several rounds when chunks are small
    by_name = {(c["file"], c["mode"]): r for c, r in zip(cases, rounds)}
    peer = {(c["file"], c["mode"]): p for c, p in zip(cases, res["peer"])}
    assert peer[("big_clean", "index")] == variant.startswith("peer")  # the rounds went through mapped peer memory / through exchanges
    if variant == "weak_hash":
        assert by_name[("synthetic_pair_ok", "pair")] >= 1  # (the one-file jobs were redone exactly; the two-file job went round by round)
    elif variant == "pipelined":
        assert by_name[("big_clean", "index")] >= 1 and by_name[("synthetic_pair_ok", "pair")] >= 2  # (one round per file at least)
    elif variant in ("small_chunks", "peer_copies", "peer_reuse"):
        assert by_name[("big_clean", "index")] >= 3
    elif variant in ("overflow", "peer_overflow"):
        assert by_name[("big_clean", "index")] == 1  # (the worker reports the exact reruns here)


def test_world_of_one():
    """The same orchestration without a process group (what the one-GPU tests of the routing run on the device)."""
    subprocess.check_call(["make", "-C", os.path.join(ROOT, "tests", "sim")], stdout=subprocess.DEVNULL)
    out = subprocess.run([sys.executable, os.path.join(ROOT, "tests", "dist_world1_worker.py")], capture_output=True, text=True, timeout=600)
    assert out.returncode == 0 and out.stdout.strip().startswith("ok 40"), (out.stdout[-500:], out.stderr[-2000:])


@pytest.mark.parametrize("world,variant", [(3, "peer_copies"), (2, "small_chunks")])
def test_random_cuts_through_the_routing_rounds(tmp_path, world, variant):
    """Byte ranges cut at random positions (inside names, at line feeds, one byte apart) and chunks of 8 KiB: many different
    phases of chunk and range boundaries through the chunk-by-chunk routing, clean files and files with one late duplicate."""
    subprocess.check_call(["make", "-C", os.path.join(ROOT, "tests", "sim")], stdout=subprocess.DEVNULL)
    rng = random.Random(2024 + world)
    cases = []
    for k in range(24):
        nrec = rng.choice([900, 1500, 2500, 4000])
        recs = [f"@M{k}:1:FC:1:11:{i}:{i * 7} 1:N:0:AC\n{'ACGTN' * (3 + (i * 7 + k) % 9)}\n+\n{'F' * (5 * (3 + (i * 7 + k) % 9))}\n" for i in range(nrec)]
        if k % 3 == 2:
            recs[nrec - 1 - rng.randrange(50)] = recs[rng.randrange(50)]
        data = "".join(recs).encode()
        cuts = sorted(rng.random() for _ in range(world - 1))
        if k % 5 == 0:  # two cuts right next to each other / at the very start of a line
            p = data.find(b"\n@", int(len(data) * cuts[0])) + 1
            cuts = sorted([p / len(data)] + [(p + 1) / len(data)] * (world - 2))
        cases.append({"file": f"rand{k}", "mode": "index" if k % 4 else "single", "hex": data.hex(), "cuts": cuts})
    cin, cout = tmp_path / "cases.json", tmp_path / "out.json"
    json.dump(cases, open(cin, "w"))
    env = dict(os.environ, MASTER_ADDR="127.0.0.1", **VARIANTS[variant])
    subprocess.check_call([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={world}", "--master-addr", "127.0.0.1",
                           "--master-port", str(29680 + world), os.path.join(ROOT, "tests", "dist_worker.py"), str(cin), str(cout)], env=env, timeout=600)
    res = json.load(open(cout))
    for c, g in zip(cases, res["transcripts"]):
        argv = (["-r"] if c["mode"] == "single" else []) + ["a.fq"]
        assert tuple(g) == oracle_run(argv, bytes.fromhex(c["hex"]), None), (c["file"], c["mode"], c["cuts"], g)
    assert sum(1 for r in res["rounds"] if r >= 3) >= 8  # most index jobs really went round by round
