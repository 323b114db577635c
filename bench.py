#!/usr/bin/env python
"""bench.py — fastq_info hot path throughput on B200 (BASELINE.json metric: FASTQ GB/s and reads/s validated).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--workload illumina_pe|illumina_se|longread] [--dump-outputs DIR]

One step = one complete fastq_info job over synthetic input already resident in HBM.  Workloads (SURVEY.md §8d):

  illumina_pe  (default) BASELINE configs[3]: paired 2x150 bp files, default mode (index loop over file 1, mate loop over file 2),
               50.3 M pairs per GPU — weak scaling, 8 GPUs hold the 400 M pairs the config names; mates permuted inside windows of 1024
  illumina_se  BASELINE configs[2]: 100 M single-end 150 bp reads per GPU, default mode (read-name uniqueness on)
  longread     BASELINE configs[4]: ONT/PacBio-like reads, 1-100 kb log-normal, -r mode, about 30 GB per GPU

`value` is GB/s of decompressed FASTQ over the whole job; `e2e` is the same job fed from pinned HOST memory through fqg_feed (H2D
copy inside the timed region) with the report read back.  Before the timed region the workload's negative twins run once and every
transcript (clean run included, at full size) is compared with the text the reference prints, known by construction: `parity`.
At N=1 the line also carries `also`: the 400 M-pair job streamed through one GPU (`illumina_pe_streamed`) and the command line on gzip
operands against the reference binary, host inflate included (`gz_cli`).
The reference arm times the unmodified reference binary (oracle/_ref/fastq_info, 1 thread — it has none) on a bounded sample.
`--dump-outputs DIR` writes what the last timed step returned (the report and the transcript rendered from it) as DIR/<name>.npy,
so that two builds can be compared output for output: the inputs are generated from fixed seeds.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

HBM_FALLBACK_GBS = 6650.0  # /opt/skills/guides/B200_PROFILING.md fallback when MEASURED_PEAKS.json is absent
KEY_NONE = (1 << 64) - 1
PAIRS_PER_GPU = 49152 * 1024  # 50.3 M: a multiple of the mate file's permutation window; x8 = 402.7 M pairs


def measured_peak():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            d = json.load(open(p))
            v = d.get("hbm_gbs") or d.get("hbm_gb_s")
            if v:
                return float(v), "measured"
        except Exception:
            pass
    return HBM_FALLBACK_GBS, "fallback"


class ClockSampler(threading.Thread):
    """nvidia-smi clocks and throttle reasons during the timed region."""
    Q = "clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, indices, period=0.05):
        super().__init__(daemon=True)
        self.indices, self.rows, self.stop_flag, self.period = indices, [], False, period

    def run(self):
        while not self.stop_flag:
            try:
                out = subprocess.run(["nvidia-smi", "-i", ",".join(str(i) for i in self.indices), f"--query-gpu={self.Q}", "--format=csv,noheader,nounits"],
                                     capture_output=True, text=True, timeout=5).stdout.strip()
                for line in out.splitlines():
                    if line.strip():
                        self.rows.append([x.strip() for x in line.split(",")])
            except Exception:
                pass
            time.sleep(self.period)

    def summary(self):
        sm = sorted(int(r[0]) for r in self.rows if r[0].isdigit())
        mx = [int(r[1]) for r in self.rows if r[1].isdigit()]
        reasons = []
        for i, name in enumerate(["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]):
            if any(len(r) > 2 + i and r[2 + i].lower().startswith("active") for r in self.rows):
                reasons.append(name)
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None, "reasons": reasons, "samples": len(self.rows)}


# ---------------------------------------------------------------------------------------------- the reference's CPU implementation
def reference_binary():
    p = os.path.join(ROOT, "oracle", "_ref", "fastq_info")
    return p if os.path.exists(p) else None


def time_reference(files, argv_head):
    """Wall time of the reference's own fastq_info on plain-text files (inflate excluded on both sides) → (seconds, rc, kind)."""
    shm = "/dev/shm" if os.path.isdir("/dev/shm") else "/tmp"
    paths = []
    for i, data in enumerate(files):
        path = os.path.join(shm, f"fqg_bench_{os.getpid()}_{i + 1}.fastq")
        with open(path, "wb") as fh:
            fh.write(data)
        paths.append(path)
    try:
        ref = reference_binary()
        t0 = time.perf_counter()
        if ref:
            p = subprocess.run([ref] + argv_head + paths, capture_output=True)
            rc, kind = p.returncode, "reference"
        else:  # the reference did not compile here: the oracle's restatement of it (test infrastructure, timed as the CPU baseline only)
            sys.path.insert(0, os.path.join(ROOT, "tests"))
            from _util import oracle_run
            rc, kind = oracle_run(argv_head + ["a.fq", "b.fq"][:len(files)], files[0], files[1] if len(files) > 1 else None)[0], "port"
        return time.perf_counter() - t0, rc, kind
    finally:
        for p in paths:
            os.unlink(p)


def time_gz_cli(files, argv_head):
    """The whole command line on gzip files, host inflate included (north_star: reported separately): `fastq_info_gpu` (zlib on a helper
    thread into pinned pieces, copied and validated while the next piece inflates) against the reference binary on the same files.
    Wall clock of each process — for ours that includes loading CUDA and creating the context.  The two transcripts must be equal."""
    import zlib
    shm = "/dev/shm" if os.path.isdir("/dev/shm") else "/tmp"
    cli = os.path.join(ROOT, "fastq_utils_b200", "fastq_info_gpu")
    ref = reference_binary()
    paths, gz_bytes = [], 0
    try:
        for i, data in enumerate(files):
            path = os.path.join(shm, f"fqg_bench_{os.getpid()}_{i + 1}.fastq.gz")
            co = zlib.compressobj(1, zlib.DEFLATED, 31)
            with open(path, "wb") as fh:
                fh.write(co.compress(bytes(data)))
                fh.write(co.flush())
            gz_bytes += os.path.getsize(path)
            paths.append(path)
        env = dict(os.environ, LD_LIBRARY_PATH=os.path.join(ROOT, "fastq_utils_b200") + ":" + os.environ.get("LD_LIBRARY_PATH", ""))
        t0 = time.perf_counter()
        ours = subprocess.run([cli] + argv_head + paths, capture_output=True, env=env, timeout=300)
        t_ours = time.perf_counter() - t0
        res = {"ours_wall_s": t_ours, "ours_exit_status": ours.returncode, "gz_bytes": gz_bytes}
        # what of that is start-up (loading CUDA, creating the context, page-locked buffers): the same command on an empty file
        empty = os.path.join(shm, f"fqg_bench_{os.getpid()}_empty.fastq")
        open(empty, "wb").close()
        try:
            t0 = time.perf_counter()
            subprocess.run([cli, "-e", empty], capture_output=True, env=env, timeout=300)
            res["ours_startup_wall_s"] = time.perf_counter() - t0
        finally:
            os.unlink(empty)
        if ref:
            t0 = time.perf_counter()
            r = subprocess.run([ref] + argv_head + paths, capture_output=True, timeout=300)
            res.update({"reference_wall_s": time.perf_counter() - t0, "reference_exit_status": r.returncode,
                        "transcripts_equal": (r.returncode, r.stdout, r.stderr) == (ours.returncode, ours.stdout, ours.stderr)})
        return res
    finally:
        for p in paths:
            if os.path.exists(p):
                os.unlink(p)


def host_sample(workload, n):
    """The first n records (pairs) of the workload as host bytes, from the numpy twin of the device generator: libfastq_gpu.so is not
    loaded by the reference arm."""
    from fastq_utils_b200 import synth
    if workload == "illumina_pe":
        n = n // 1024 * 1024
        return [synth.illumina(0, n, seed=43, mate=1), synth.illumina(0, n, seed=43, mate=2, perm_window=1024)], [], n
    if workload == "illumina_se":
        return [synth.illumina(0, n, seed=42, mate=1)], [], n
    raise ValueError(workload)


def longread_layout(nbytes_target, torch, hdr):
    g = torch.Generator().manual_seed(7)
    nrec = int(nbytes_target / (2 * 13_000 + hdr))  # the mean of the clipped log-normal is about 13 kb
    lens = torch.exp(torch.randn(nrec, generator=g) + 8.987).clamp(1000, 100000).to(torch.int64)  # ln 8000 = 8.987
    off = torch.zeros(nrec + 1, dtype=torch.int64)
    off[1:] = torch.cumsum(hdr + 2 * lens + 4, 0)
    return nrec, lens, off


def longread_sample_bytes(nrec, lens, seed=7):
    """host twin of fq_synth_long_kernel for a small sample (reference arm): same shape, numpy"""
    import numpy as np
    out = []
    rng = np.random.default_rng(seed)
    for i in range(nrec):
        L = int(lens[i])
        h = "@%016x runid=%08x read=%010d ch=%03d start_time=2024-01-01T00:00:00Z\n" % (rng.integers(0, 1 << 63), seed, i, 1 + i % 512)
        sq = np.frombuffer(b"ACGT", dtype=np.uint8)[rng.integers(0, 4, L)].tobytes()
        ql = (35 + rng.integers(0, 59, L)).astype(np.uint8).tobytes()
        out.append(h.encode() + sq + b"\n+\n" + ql + b"\n")
    return b"".join(out)


# ---------------------------------------------------------------------------------------------- parity helpers
def _same(got, want, what, parity):
    ok = tuple(got) == tuple(want)
    parity[what] = "ok" if ok else {"got": [got[0], got[1][-200:], got[2][-300:]], "want": [want[0], want[1][-200:], want[2][-300:]]}
    return ok


def dump_outputs(d, rep, transcript):
    """The report of one job (include/fastq_gpu.h: fqg_report) and its rendered transcript as float64 .npy files under d.  Report
    fields are 64-bit integers, which float64 holds exactly only below 2**53: each field is stored as the pair (high 32 bits, low 32
    bits) along the last axis.  The transcript's text is stored as byte codes.  The error's header and name strings are left out (the
    timed job raises no error)."""
    import numpy as np
    os.makedirs(d, exist_ok=True)
    u64 = lambda xs: np.array([[(int(x) & KEY_NONE) >> 32, int(x) & 0xFFFFFFFF] for x in xs], dtype=np.float64)  # noqa: E731
    e = rep.error
    arrays = {"report_files": np.stack([u64([f.n_records, f.num_rds, f.min_rl, f.max_rl, f.min_qual, f.max_qual, f.sniff_format, f.color_space])
                                        for f in rep.file]),  # per file: n_records num_rds min_rl max_rl min_qual max_qual sniff_format color_space
              "report_index": u64([rep.mode, rep.n_index_entries, rep.n_index_left, rep.index_mem, rep.median_rl, *rep.reads_before_error]),
              "report_error": u64([e.code, e.file, e.msg_file, e.chr, e.record, e.line, e.a, e.b, e.event_key]),
              "exit_status": np.array([transcript[0]], dtype=np.float64),
              "stdout": np.frombuffer(transcript[1].encode("latin-1"), dtype=np.uint8).astype(np.float64),
              "stderr": np.frombuffer(transcript[2].encode("latin-1"), dtype=np.uint8).astype(np.float64)}
    for name, arr in arrays.items():
        np.save(os.path.join(d, name + ".npy"), arr)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours")
    ap.add_argument("--workload", default="illumina_pe", choices=["illumina_pe", "illumina_se", "longread"])
    ap.add_argument("--reads", type=int, default=0, help="records (illumina_pe: pairs) per GPU; 0 = the workload's default")
    ap.add_argument("--gb", type=float, default=30.0, help="longread: GB per GPU")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-extras", action="store_true", help="N=1: skip the `also` runs (other configurations, the streamed 400 M-pair job)")
    ap.add_argument("--cpu-sample-reads", type=int, default=1_000_000, help="records (pairs) of the CPU baseline's sample")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the report and transcript of the last timed step as DIR/<name>.npy")
    a = ap.parse_args()
    if a.steps < 1:
        ap.error("--steps must be at least 1")
    if a.dump_outputs and a.impl == "reference":
        ap.error("--dump-outputs writes what our timed job computed: not available with --impl reference")

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
    from fastq_utils_b200 import synth
    rb = synth.ILL_REC
    wl = a.workload
    n = a.reads or {"illumina_pe": PAIRS_PER_GPU, "illumina_se": 100_000_000, "longread": 0}[wl]
    if wl == "illumina_pe":
        n = max(1024, n // 1024 * 1024)

    # ------------------------------------------------------------------ reference arm: the reference's own CPU implementation
    if a.impl == "reference":
        if rank != 0:
            return
        ns = a.cpu_sample_reads
        if wl == "longread":
            import torch
            nrec, lens, off = longread_layout(0.5e9, torch, 82)
            files, head, ns = [longread_sample_bytes(nrec, lens)], ["-r"], nrec
            name = f"longread_skew_seed7_{a.gb:.0f}GB_-r"
        else:
            files, head, ns = host_sample(wl, ns)
            name = f"illumina_pe_{n * world // 1_000_000}M_pairs_2x150" if wl == "illumina_pe" else f"illumina_se_{n // 1_000_000}M_150bp_uniqueness_on"
        nbytes = sum(len(f) for f in files)
        times = []
        for i in range(a.warmup + a.steps):
            dt, rc, kind = time_reference(files, head)
            assert rc == 0, rc
            if i >= a.warmup:
                times.append(dt)
        per = sum(times) / len(times)
        gbs = nbytes / per / 1e9
        reads = ns * (2 if wl == "illumina_pe" else 1)
        print(json.dumps({"impl": "reference", "metric": "fastq_info_validated_GBps", "value": gbs, "unit": "GB/s", "n_gpus": a.gpus, "steps": a.steps,
                          "warmup": a.warmup, "ms_per_step": per * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
                          "dtype": "u8", "data": "synthetic", "config": {"workload": name, "mode": "fastq_info " + (" ".join(head) or "default")}, "reads_per_s": reads / per,
                          "cpu_baseline": {"value": gbs, "unit": "GB/s", "cores": 1, "kind": kind,
                                           "sample": f"first {ns} {'pairs' if wl == 'illumina_pe' else 'records'} ({nbytes / 1e6:.0f} MB plain text) of the workload, generated on the host (numpy twin of the device generator; libfastq_gpu.so not loaded), wall clock, reference is single-threaded, host nproc={os.cpu_count()}"},
                          "e2e": {"value": gbs, "unit": "GB/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}))
        return

    # ------------------------------------------------------------------ our arm
    import torch
    import torch.distributed as dist
    import fastq_utils_b200 as fq
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    stream = torch.cuda.current_stream().cuda_stream
    assert fq.illumina_record_bytes() == rb
    parity = {}

    def gen_illumina(first, count, seed, mate, perm):
        t = torch.empty(count * rb + 64, dtype=torch.uint8, device="cuda")
        piece = 8_192_000
        for s in range(0, count, piece):
            k = min(piece, count - s)
            fq.synth_illumina(t[s * rb:], first + s, k, seed=seed, mate=mate, perm_window=perm, stream=stream)
        t[count * rb:].zero_()
        return t

    # ---- inputs of this rank, resident in HBM
    lens = None
    if wl == "illumina_pe":
        first = rank * n
        bufs = [gen_illumina(first, n, 43, 1, 0), gen_illumina(first, n, 43, 2, 1024)]
        nb = n * rb
        total_bytes_rank, reads_rank = 2 * nb, 2 * n
        mode = fq.MODE_INDEX_PAIR
        name = f"illumina_pe_{n * world // 1_000_000}M_pairs_2x150"
        names = ("synthetic_1.fastq", "synthetic_2.fastq")
        want_clean = synth.expect_index(n * world, names[0], n2=n * world, name2=names[1])
    elif wl == "illumina_se":
        first = rank * n
        bufs = [gen_illumina(first, n, 42, 1, 0)]
        nb = n * rb
        total_bytes_rank, reads_rank = nb, n
        mode = fq.MODE_INDEX
        name = f"illumina_se_{n * world // 1_000_000}M_150bp_uniqueness_on"
        names = ("synthetic.fastq", None)
        want_clean = synth.expect_index(n * world, names[0])
    else:
        hdr = fq.lib().fqg_synth_long_header_bytes()
        nrec, lens, off = longread_layout(a.gb * 1e9, torch, hdr)
        nb = int(off[-1])
        t = torch.zeros(nb + 64, dtype=torch.uint8, device="cuda")
        fq.synth_longreads(t, off.cuda(), rank * nrec, nrec, seed=7, stream=stream)
        bufs = [t]
        n = nrec
        total_bytes_rank, reads_rank = nb, nrec
        mode = fq.MODE_SINGLE
        name = f"longread_skew_seed7_{nb * world / 1e9:.0f}GB_-r"
        names = ("synthetic.fastq", None)
        want_clean = None  # statistics checked against the lengths below
    torch.cuda.synchronize()
    config = {"workload": name, "mode": {fq.MODE_INDEX_PAIR: "fastq_info f1 f2 (index loop + mate loop)", fq.MODE_INDEX: "fastq_info f (index + validate)", fq.MODE_SINGLE: "fastq_info -r f"}[mode],
              "reads_per_gpu": reads_rank, "bytes_per_gpu": total_bytes_rank, "record_bytes": rb if wl != "longread" else None,
              "l2": f"inputs ({total_bytes_rank / 1e9:.1f} GB per GPU) far larger than L2; no flush between steps"}

    # ---- the job
    if world > 1:
        from fastq_utils_b200 import dist as fqdist
        runner = fqdist.ShardedFastqInfo(mode, local, n_hint=n)
        ctx = runner.ctx

        def run_job(ptrs, sizes):
            kw = {}
            if mode == fq.MODE_INDEX_PAIR:
                kw = {"ptr2": ptrs[1], "nbytes2": sizes[1], "name2": names[1]}
            return runner.run_device(ptrs[0], sizes[0], name=names[0], **kw)

        def step():
            res = run_job([b.data_ptr() for b in bufs], [nb] * len(bufs))
            assert res["event_key"] == KEY_NONE, res["event_key"]
            return res

        def transcript_of(res):
            return res.get("transcript")
    else:
        ctx = fq.FastqInfo(mode, device=local, index_capacity_hint=n if mode != fq.MODE_SINGLE else 0)

        def run_pieces(pieces):
            """pieces: [(file, ptr, nbytes, last)]"""
            ctx.reset()
            for f, p, k, last in pieces:
                ctx.feed_device(f, p, k, last=last)
            return ctx.finish()

        def step():
            rep = run_pieces([(f, b.data_ptr(), nb, True) for f, b in enumerate(bufs)])
            assert rep.error.code == 0, rep.error.code
            return rep

        def transcript_of(rep):
            return ctx.render(rep, names[0], names[1])

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize()

    # ---- parity, before the timed region: negative twins of the workload against the reference's text (by construction)
    if wl in ("illumina_pe", "illumina_se") and world == 1:
        j = n // 3 + 5  # the record that goes missing / is duplicated / spoilt
        p0 = bufs[0].data_ptr()
        if wl == "illumina_pe":
            p1 = bufs[1].data_ptr()
            s = next(s for s in range(j // 1024 * 1024, j // 1024 * 1024 + 1024) if synth.perm_source(s, 1024) == j)  # where the mate of record j sits
            # twin A: file 1 lacks record j -> its mate is an unpaired read, at its line of file 2
            rep = run_pieces([(0, p0, j * rb, False), (0, p0 + (j + 1) * rb, (n - j - 1) * rb, True), (1, p1, nb, True)])
            tail = (3, "", f"\nERROR: Error in file {names[1]}: line {4 * (s + 1)}: unpaired read - {synth.illumina_name(first + j)}\n")
            _same(transcript_of(rep), synth.expect_index(n - 1, names[0], n2=s, name2=names[1], tail=tail), "mate_removed_from_file1", parity)
            # twin B: file 2 lacks that mate -> one name of file 1 is left over
            rep = run_pieces([(0, p0, nb, True), (1, p1, s * rb, False), (1, p1 + (s + 1) * rb, (n - s - 1) * rb, True)])
            tail = (3, "\n", f"\nERROR: Error in file {names[0]}: found 1 unpaired reads\n")
            _same(transcript_of(rep), synth.expect_index(n, names[0], n2=n - 1, name2=names[1], tail=tail), "extra_name_in_file1", parity)
        # twin C: record 100 once more behind record j -> duplicated sequence at that line (line = 4 x records read so far)
        rep = run_pieces([(0, p0, (j + 1) * rb, False), (0, p0 + 100 * rb, rb, False), (0, p0 + (j + 1) * rb, (n - j - 1) * rb, True)] + ([(1, bufs[1].data_ptr(), nb, True)] if wl == "illumina_pe" else []))
        tail = (3, "", f"\nERROR: Error in file {names[0]}: line {4 * (j + 2)}: duplicated sequence {synth.illumina_name(first + 100)}\n")
        want = synth.expect_index(j + 1, names[0], tail=tail)
        want = (want[0], want[1], want[2].replace(f"Scanning complete.\n\nReads processed: {j + 1}\nMemory used in indexing: ~{(8 + (j + 1) * (synth.NAME_LEN + 41)) // (1024 * 1024)} MB\n", ""))
        _same(transcript_of(rep), want, "duplicate_name", parity)
    elif wl in ("illumina_pe", "illumina_se"):
        # N > 1: the twins on a small job of the same shape (1 M records per rank), through the same sharded path
        m = 1024 * 1024
        small = [gen_illumina(rank * m, m, 43, 1, 0)] + ([gen_illumina(rank * m, m, 43, 2, 1024)] if wl == "illumina_pe" else [])
        torch.cuda.synchronize()
        sizes = [m * rb] * len(small)
        res = run_job([b.data_ptr() for b in small], sizes)
        want = synth.expect_index(m * world, names[0], n2=m * world if wl == "illumina_pe" else None, name2=names[1])
        if rank == 0:
            _same(transcript_of(res), want, "small_clean", parity)
        j = m // 3 + 5
        if wl == "illumina_pe":
            s = next(s for s in range(j // 1024 * 1024, j // 1024 * 1024 + 1024) if synth.perm_source(s, 1024) == j)
            # rank 0's file 2 without the mate of ITS record j: one name left over
            cut = small[1].clone()
            if rank == 0:
                cut[s * rb:(m - 1) * rb] = small[1][(s + 1) * rb:m * rb].clone()
            torch.cuda.synchronize()
            res = run_job([small[0].data_ptr(), cut.data_ptr()], [m * rb, (m - 1) * rb if rank == 0 else m * rb])
            tail = (3, "\n", f"\nERROR: Error in file {names[0]}: found 1 unpaired reads\n")
            if rank == 0:
                _same(transcript_of(res), synth.expect_index(m * world, names[0], n2=m * world - 1, name2=names[1], tail=tail), "small_extra_name_in_file1", parity)
            # rank 0's file 1 without record j: its mate is an unpaired read at its line of file 2
            cut1 = small[0].clone()
            if rank == 0:
                cut1[j * rb:(m - 1) * rb] = small[0][(j + 1) * rb:m * rb].clone()
            torch.cuda.synchronize()
            res = run_job([cut1.data_ptr(), small[1].data_ptr()], [(m - 1) * rb if rank == 0 else m * rb, m * rb])
            tail = (3, "", f"\nERROR: Error in file {names[1]}: line {4 * (s + 1)}: unpaired read - {synth.illumina_name(j)}\n")
            if rank == 0:
                _same(transcript_of(res), synth.expect_index(m * world - 1, names[0], n2=s, name2=names[1], tail=tail), "small_mate_removed_from_file1", parity)
            del cut, cut1
        # the last rank's last record once more at its end: a duplicated name; and an invalid base on rank 0 that must win over it
        dup = torch.empty((m + 1) * rb + 64, dtype=torch.uint8, device="cuda")
        dup[:m * rb] = small[0][:m * rb]
        dup[m * rb:(m + 1) * rb] = small[0][(m - 1) * rb:m * rb]
        dup[(m + 1) * rb:].zero_()
        torch.cuda.synchronize()
        last = rank == world - 1
        res = run_job([dup.data_ptr() if last else small[0].data_ptr()] + [b.data_ptr() for b in small[1:]], [(m + 1) * rb if last else m * rb] + sizes[1:])
        tail = (3, "", f"\nERROR: Error in file {names[0]}: line {4 * (m * world + 1)}: duplicated sequence {synth.illumina_name(m * world - 1)}\n")
        want = synth.expect_index(m * world, names[0], tail=tail)
        want = (want[0], want[1], want[2].replace(f"Scanning complete.\n\nReads processed: {m * world}\nMemory used in indexing: ~{(8 + m * world * (synth.NAME_LEN + 41)) // (1024 * 1024)} MB\n", ""))
        if rank == 0:
            _same(transcript_of(res), want, "small_duplicate_name", parity)
        if rank == 0:
            small[0][j * rb + 60] = ord("*")
        torch.cuda.synchronize()
        res = run_job([dup.data_ptr() if last and world > 1 else small[0].data_ptr()] + [b.data_ptr() for b in small[1:]], [(m + 1) * rb if last and world > 1 else m * rb] + sizes[1:])
        tail = (3, "", f"\nERROR: Error in file {names[0]}: line {4 * (j + 1) + 1}: invalid character '*' (hex. code:'2a'), expected ACGTUacgtu0123nN.\n")
        want = synth.expect_index(j, names[0], tail=tail)
        want = (want[0], want[1], want[2].replace(f"Scanning complete.\n\nReads processed: {j}\nMemory used in indexing: ~{(8 + j * (synth.NAME_LEN + 41)) // (1024 * 1024)} MB\n", ""))
        if rank == 0:
            _same(transcript_of(res), want, "small_invalid_base_wins", parity)
        del small, dup
        torch.cuda.empty_cache()

    for _ in range(a.warmup):
        step()
    if world > 1:
        runner.phase_ms.clear()
        for k in runner.host_ms:
            runner.host_ms[k] = 0.0
    ctx.kernel_stats(reset=True)
    if world > 1 and runner.shard is not None:
        runner.shard.kernel_stats(reset=True)
    l0 = ctx.launch_count() + (runner.shard.launch_count() if world > 1 and runner.shard is not None else 0)
    # (one sampler for all GPUs of the job, on rank 0: every nvidia-smi call takes the driver's attention for a moment)
    sampler = ClockSampler(list(range(world)) if world > 1 else [local], period=0.05 if world == 1 else 0.25)
    if rank == 0:
        sampler.start()
    barrier()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev0.record()  # (torch's stream is idle here: the event marks the device's clock at the start of the timed region)
    t0 = time.perf_counter()
    dev_ms = 0.0
    for _ in range(a.steps):
        rep = step()
        dev_ms += ctx.device_ms()
    barrier()
    ev1.record()
    torch.cuda.synchronize()
    wall = time.perf_counter() - t0
    span_ms = ev0.elapsed_time(ev1)  # device clock over the whole timed region, every stream's work and every host gap included
    sampler.stop_flag = True
    if rank == 0:
        sampler.join(timeout=2)
    launches = ctx.launch_count() - l0
    ks = ctx.kernel_stats()
    paths = ctx.path_counts()
    if world > 1 and runner.shard is not None:  # the index shard lives in its own context
        launches += runner.shard.launch_count()
        sk = runner.shard.kernel_stats()
        for k in ("index", "mate"):
            ks[k] = sk[k]
    if world > 1:
        dev_ms = span_ms  # the sharded step runs on several streams of two contexts: the span between the two events is its device time
    # the step is host-driven (several synchronising read-backs); device-event time and wall time are both reported, the larger one counts
    per_step = max(dev_ms / 1e3, wall) / a.steps
    rank_ms = per_step * 1e3
    if world > 1:
        tt = torch.tensor([per_step], device="cuda", dtype=torch.float64)
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        per_step = float(tt.item())
        allms = [None] * world
        dist.all_gather_object(allms, round(rank_ms, 3))
    value = total_bytes_rank * world / per_step / 1e9

    # ---- parity of the timed job itself, at full size
    if rank == 0:
        tr = transcript_of(rep)
        if a.dump_outputs:
            dump_outputs(a.dump_outputs, rep if world == 1 else rep["report"], tr)
        if want_clean is not None:
            _same(tr, want_clean, "timed_job_transcript", parity)
        else:  # long reads: number of reads, length range and median from the generator's lengths; qualities 35..93 are `sanger`
            srt = torch.sort(lens).values
            med = int(srt[len(srt) // 2]) if world == 1 else None
            txt = tr[2]
            ok = tr[0] == 0 and f"Number of reads: {n * world}\n" in txt and "Quality encoding range: 35 93\nQuality encoding: sanger\n" in txt
            if world == 1:
                ok = ok and f"Read length: {int(lens.min())} {int(lens.max())} {med}\n" in txt
            parity["timed_job_statistics"] = "ok" if ok else {"got": [tr[0], txt[-300:]]}
    parity_ok = all(v == "ok" for v in parity.values())

    # ---- dominant kernel and its roofline
    peak, peak_kind = measured_peak()
    dom = max(["scan", "records", "tile", "lanes"], key=lambda k: ks[k]["ms"])
    kd = ks[dom]
    ach = kd["bytes"] / (kd["ms"] / 1e3) / 1e9 if kd["ms"] > 0 else 0.0
    # DRAM traffic of the dominant kernel per launch: the latest committed `ncu --set full` capture of the same kernel, scaled by launch size
    traffic, traffic_src = None, None
    try:
        import glob
        import re
        if dom == "lanes":
            f = sorted(glob.glob(os.path.join(ROOT, "profiles", "r*_lanes_*ncu_summary.txt")),
                       key=lambda x: (int(re.match(r"r(\d+)", os.path.basename(x)).group(1)), os.path.basename(x)))[-1]  # the latest round's
            txt = open(f, errors="ignore").read()
            rd = float(re.search(r"dram__bytes_read\.sum\s+([\d.]+)\s+Gbyte", txt).group(1))
            wr = re.search(r"dram__bytes_write\.sum\s+([\d.]+)\s+(M|G)byte", txt)
            wrg = float(wr.group(1)) / (1e3 if wr.group(2) == "M" else 1.0)
            per_byte = (rd + wrg) * 1e9 / 2.1181e9
            traffic, traffic_src = per_byte * (kd["bytes"] / max(1, kd["launches"])), os.path.basename(f)
    except Exception:
        traffic = None
    pv_ms = sum(ks[k]["ms"] for k in ("scan", "records", "tile", "lanes"))
    roof = {"bound": "hbm", "kernel": {"scan": "fq_scan_kernel", "records": "fq_records_kernel", "tile": "fq_tile_kernel", "lanes": "fq_lanes_kernel"}[dom], "achieved": ach, "peak": peak, "peak_kind": peak_kind,
            "unit": "GB/s", "frac": ach / peak, "traffic": traffic, "traffic_unit": f"bytes per launch (ncu dram__bytes_read+write of {traffic_src}, scaled by launch size)", "launches": kd["launches"], "avg_launch_ms": kd["ms"] / max(1, kd["launches"]),
            "algorithmic_bytes_per_launch": kd["bytes"] / max(1, kd["launches"]),
            "all_kernels_ms_per_step": {k: v["ms"] / a.steps for k, v in ks.items()},
            "parse_validate_GBps": total_bytes_rank * a.steps / (pv_ms / 1e3) / 1e9 if pv_ms > 0 else None,
            "index_Mops_per_s": ks["index"]["items"] / (ks["index"]["ms"] / 1e3) / 1e6 if ks["index"]["ms"] > 0 else None,
            "mate_Mops_per_s": ks["mate"]["items"] / (ks["mate"]["ms"] / 1e3) / 1e6 if ks["mate"]["ms"] > 0 else None}

    out = {"metric": "fastq_info_validated_GBps", "value": value, "unit": "GB/s", "n_gpus": world, "steps": a.steps, "warmup": a.warmup,
           "ms_per_step": per_step * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u8", "data": "synthetic",
           "config": config, "reads_per_s": reads_rank * world / per_step, "device_ms_per_step": dev_ms / a.steps, "wall_ms_per_step": wall / a.steps * 1e3,
           "gpu_launches": int(launches), "paths": paths, "parity": dict(parity, all_ok=parity_ok), "roofline": roof, "clocks": sampler.summary()}
    if world > 1:
        out["config"]["parallelism"] = f"byte-range shards x{world}, names routed by hash to the owner of their index shard ({runner.route_description()}), stats all-reduced"
        out["config"]["routing_rounds"] = runner.rounds_done
        out["rank_ms_per_step"] = allms
        out["host_phase_ms_per_step_rank0"] = {k: round(v / a.steps, 2) for k, v in runner.phase_ms.items()}  # wall time of the phases of ShardedFastqInfo.run_device
        out["host_round_ms_per_step_rank0"] = {k: round(v / a.steps, 2) for k, v in runner.host_ms.items()}  # ... inside the routing rounds: waiting for the barrier, queueing copies
        out["e2e"] = {"value": None, "unit": "GB/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0, "note": "measured at N=1 only"}

    if rank == 0 and world == 1:
        # ---------------- the dominant kernel without the index kernels beside it: the first file through the -r loop (no name index)
        try:
            solo = fq.FastqInfo(fq.MODE_SINGLE, device=local)
            for i in range(3):
                if i == 1:
                    solo.kernel_stats(reset=True)
                solo.reset()
                solo.feed_device(0, bufs[0].data_ptr(), nb, last=True)
                r1 = solo.finish()
                assert r1.error.code == 0
            ks1 = solo.kernel_stats()[dom]
            solo.close()
            if ks1["ms"] > 0:
                a1 = ks1["bytes"] / (ks1["ms"] / 1e3) / 1e9
                out["roofline"]["alone"] = {"achieved": a1, "frac": a1 / peak, "avg_launch_ms": ks1["ms"] / max(1, ks1["launches"]),
                                            "note": "same kernel, same bytes, -r loop: no index kernel running beside it"}
        except Exception as ex:
            out["roofline"]["alone"] = {"error": str(ex)[:200]}
        # ---------------- `also`: the other single-GPU configurations
        if not a.no_extras and wl == "illumina_pe":
            out["also"] = {}
            try:
                out["also"]["illumina_pe_streamed"] = streamed_pairs(fq, synth, torch, local, 8 * n, bufs)
            except Exception as ex:
                out["also"]["illumina_pe_streamed"] = {"error": str(ex)[:300]}
        # ---------------- e2e: the same job through fqg_feed from pinned host memory (H2D inside the timed region)
        if not a.no_e2e:
            try:
                e2e_bytes = sum([nb] * len(bufs))
                hosts = []
                for b in bufs:
                    h = torch.empty(nb, dtype=torch.uint8, pin_memory=True)
                    h.copy_(b[:nb])
                    hosts.append(h)
                torch.cuda.synchronize()
                # what the link itself delivers from the same pinned memory (PCIe roof of the end-to-end number)
                dst = bufs[0][:nb]
                torch.cuda.synchronize()
                tp = time.perf_counter()
                dst.copy_(hosts[0], non_blocking=True)
                torch.cuda.synchronize()
                pcie = nb / (time.perf_counter() - tp) / 1e9
                del bufs, dst
                torch.cuda.empty_cache()
                chunk = 1 << 30

                def e2e_step():
                    ctx.reset()
                    for f, h in enumerate(hosts):
                        for off in range(0, nb, chunk):
                            k = min(chunk, nb - off)
                            ctx.feed(f, (h.data_ptr() + off, k), last=(off + k == nb))
                    r = ctx.finish()
                    assert r.error.code == 0
                    return r
                e2e_step()
                torch.cuda.synchronize()
                t1 = time.perf_counter()
                reps = max(1, min(a.steps, 2))
                for _ in range(reps):
                    r = e2e_step()
                torch.cuda.synchronize()
                e2e_t = (time.perf_counter() - t1) / reps
                ms = ctx.memory_stats()
                out["e2e"] = {"value": e2e_bytes / e2e_t / 1e9, "unit": "GB/s", "h2d_bytes_per_step": e2e_bytes, "d2h_bytes_per_step": 4096,
                              "ms_per_step": e2e_t * 1e3, "reads_per_s": reads_rank / e2e_t, "pcie_h2d_GBps": pcie, "pcie_frac": e2e_bytes / e2e_t / 1e9 / pcie,
                              "device_chunk_bytes_held_at_end": ms["chunk_bytes_held"], "arena_bytes": ms["arena_bytes"],
                              "note": "fqg_feed from pinned host memory in 1 GiB pieces + fqg_finish report; validated chunks are released as the job goes (only the read names stay on the device); pcie_h2d_GBps = one cudaMemcpy of the same pinned buffer"}
            except Exception as ex:  # e.g. not enough pinned memory on this host
                out["e2e"] = {"value": None, "unit": "GB/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0, "error": str(ex)[:200]}
        # ---------------- CPU baseline: the unmodified reference binary on a bounded sample of the same workload
        try:
            if wl == "longread":
                nrec_s, lens_s, _ = longread_layout(0.5e9, torch, 82)
                files, head, ns = [longread_sample_bytes(nrec_s, lens_s)], ["-r"], nrec_s
            else:
                files, head, ns = host_sample(wl, a.cpu_sample_reads)
            dt, rc, kind = time_reference(files, head)
            sb = sum(len(f) for f in files)
            out["cpu_baseline"] = {"value": sb / dt / 1e9, "unit": "GB/s", "cores": 1, "kind": kind, "reads_per_s": ns * (2 if wl == "illumina_pe" else 1) / dt, "exit_status": rc,
                                   "sample": f"first {ns} {'pairs' if wl == 'illumina_pe' else 'records'} ({sb / 1e6:.0f} MB plain text) of the workload; reference is single-threaded; host nproc={os.cpu_count()}"}
        except Exception as ex:
            out["cpu_baseline"] = {"value": None, "error": str(ex)[:200]}
        # ---------------- the command line on gzip files, host inflate included (the CPU baseline's sample, gzipped)
        if not a.no_extras and wl in ("illumina_pe", "illumina_se") and out["cpu_baseline"].get("value"):
            try:
                from fastq_utils_b200 import synth as _synth
                k = ns * _synth.ILL_REC  # (the CPU baseline's sample)
                part = [f[:k] for f in files]
                g = time_gz_cli(part, head)
                pb = sum(len(f) for f in part)
                g.update({"plain_bytes": pb, "ours_GBps_inflated": pb / g["ours_wall_s"] / 1e9,
                          "note": "wall clock of the whole process on .gz operands: zlib inflate on the host (one thread, as in the reference), pinned pieces, H2D, kernels; "
                                  "ours includes CUDA start-up; GB/s counts inflated bytes"})
                if g.get("reference_wall_s"):
                    g["reference_GBps_inflated"] = pb / g["reference_wall_s"] / 1e9
                out.setdefault("also", {})["gz_cli"] = g
            except Exception as ex:
                out.setdefault("also", {})["gz_cli"] = {"error": str(ex)[:300]}
    if rank == 0:
        print(json.dumps(out))
    if world > 1:
        dist.destroy_process_group()
    if rank == 0 and not parity_ok:
        sys.exit(3)


def streamed_pairs(fq, synth, torch, device, npairs, resident):
    """BASELINE configs[3] on ONE GPU: 2 x npairs records (about 287 GB for 400 M pairs) do not fit the 180 GB of a B200, so the
    job is streamed: pieces are generated on the device into two alternating buffers and handed to fqg_feed_device, which keeps
    only the read names (the arena) and the index.  The timed region holds the generation of every piece; the generation alone is
    timed too.  The transcript must equal the reference's by construction; two negative twins follow."""
    import time
    rb = synth.ILL_REC
    st = torch.cuda.current_stream().cuda_stream
    piece = 4 * 1024 * 1024  # records per piece: 1.5 GB
    stage = [torch.empty(piece * rb + 64, dtype=torch.uint8, device="cuda") for _ in range(2)]
    for s in stage:
        s[piece * rb:].zero_()
    names = ("synthetic_1.fastq", "synthetic_2.fastq")
    h = fq.FastqInfo(fq.MODE_INDEX_PAIR, device=device, index_capacity_hint=npairs, flags=fq.FLAG_BORROW_FOR_CALL)

    def run(skip1=None, skip2=None, feed=True):
        """skip1 / skip2: slot of file 1 / file 2 that is left out"""
        if feed:
            h.reset()
        k = 0
        for f, mate, perm, skip in ((0, 1, 0, skip1), (1, 2, 1024, skip2)):
            for s0 in range(0, npairs, piece):
                cnt = min(piece, npairs - s0)
                buf = stage[k & 1]
                k += 1
                fq.synth_illumina(buf, s0, cnt, seed=43, mate=mate, perm_window=perm, stream=st)
                if not feed:
                    continue
                torch.cuda.current_stream().synchronize()
                last = s0 + cnt == npairs
                if skip is not None and s0 <= skip < s0 + cnt:
                    a_ = skip - s0
                    if a_:
                        h.feed_device(f, buf.data_ptr(), a_ * rb, last=False)
                    if cnt - a_ - 1 or last:
                        h.feed_device(f, buf.data_ptr() + (a_ + 1) * rb, (cnt - a_ - 1) * rb, last=last)
                else:
                    h.feed_device(f, buf.data_ptr(), cnt * rb, last=last)
        torch.cuda.synchronize()
        return h.finish() if feed else None

    res = {"pairs": npairs, "bytes": 2 * npairs * rb, "piece_bytes": piece * rb}
    run()  # warm-up (allocations, table)
    t0 = time.perf_counter()
    rep = run()
    dt = time.perf_counter() - t0
    tr = h.render(rep, names[0], names[1])
    ms = h.memory_stats()
    t0 = time.perf_counter()
    run(feed=False)
    gen = time.perf_counter() - t0
    par = {}
    _same(tr, synth.expect_index(npairs, names[0], n2=npairs, name2=names[1]), "transcript", par)
    j = npairs // 3 + 5
    s = next(s for s in range(j // 1024 * 1024, j // 1024 * 1024 + 1024) if synth.perm_source(s, 1024) == j)
    rep = run(skip1=j)
    tail = (3, "", f"\nERROR: Error in file {names[1]}: line {4 * (s + 1)}: unpaired read - {synth.illumina_name(j)}\n")
    _same(h.render(rep, names[0], names[1]), synth.expect_index(npairs - 1, names[0], n2=s, name2=names[1], tail=tail), "mate_removed_from_file1", par)
    rep = run(skip2=s)
    tail = (3, "\n", f"\nERROR: Error in file {names[0]}: found 1 unpaired reads\n")
    _same(h.render(rep, names[0], names[1]), synth.expect_index(npairs, names[0], n2=npairs - 1, name2=names[1], tail=tail), "extra_name_in_file1", par)
    h.close()
    res.update({"workload": f"illumina_pe_{npairs // 1_000_000}M_pairs_2x150_streamed_through_one_GPU", "ms": dt * 1e3, "GBps": 2 * npairs * rb / dt / 1e9, "reads_per_s": 2 * npairs / dt,
                "generation_only_ms": gen * 1e3, "GBps_net_of_generation": 2 * npairs * rb / max(dt - gen, 1e-9) / 1e9,
                "device_memory": ms, "parity": dict(par, all_ok=all(v == "ok" for v in par.values())),
                "note": "timed region = on-device generation of every 1.5 GB piece + fqg_feed_device + fqg_finish; chunks are released once validated"})
    return res


if __name__ == "__main__":
    main()
