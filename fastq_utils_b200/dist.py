"""Multi-GPU fastq_info: one process per GPU, torch.distributed (NCCL over NVLink on GPUs, gloo in the CPU tests) for
the plumbing, libfastq_gpu for every byte of work (SURVEY.md §8e, DESIGN.md §5).

Each rank holds a contiguous byte range of every input file.

  1. every rank counts the line feeds of its range (`fqg_prescan_device`); an all-gather of (line feeds, ends-with-LF,
     first line ends) fixes each range's line phase; the bytes before a range's first record start are sent to the
     previous rank, which appends them to its stream (the library's chunk-bridging joins them with its tail).  The rank
     that holds a file's first record sniffs the read-name format / colour space and everyone adopts it;
  2. validation runs locally with global record indices (`fqg_set_stream_start`);
  3. index modes: read names are routed by hash to their owner rank with two all-to-alls (24-byte tuples + name bytes);
     the owner inserts file 1's names into its shard of the index (`fqg_shard_insert`, duplicates) and lets file 2's
     names claim them (`fqg_shard_claim`, unpaired reads), always confirming equal hashes on the bytes;
  4. the earliest event (smallest key in the reference's sequential order) wins; statistics are reduced and the merged
     report is rendered with `fqg_render`, so the text and exit status equal the reference's.

Supported: MODE_SINGLE (-r), MODE_INDEX (default, one file), MODE_INDEX_PAIR (default, two files).  A clean early end of
file caused by a NUL-led header line (src/fastq.c:248) sends a one-file job to rank 0 as a whole (its engine knows the rule); with two
files it is refused on every rank (the single-GPU path handles it).
"""
import ctypes
import os
import pickle
import time

import torch
import torch.distributed as dist

from . import api

KEY_NONE = (1 << 64) - 1
FLAG_AREA = 4 << 20     # head of every rank's arena: the flag words its sources write behind their regions (8 bytes per file, round and source)
FLAG_ROUNDS = 2048      # rounds per file the flag area has words for
R_STOP, R_NAME = 0, 3
E_DUP, E_UNPAIRED, E_LEFTOVER = 13, 14, 15
MAX_READ_LENGTH = 2_500_000


class ShardedFastqInfo:
    def __init__(self, mode, device=0, n_hint=0, tensor_device=None):
        if mode not in (api.MODE_SINGLE, api.MODE_INDEX, api.MODE_INDEX_PAIR, api.MODE_INTERLEAVED, api.MODE_SORTED_PAIR):
            raise NotImplementedError("sharded runs support the five fastq_info modes")
        # MODE_INTERLEAVED is sharded like a one-file job, with the ranges cut at PAIR boundaries (eight lines instead of four: the exact
        # path only — the lines of a range do not say whether its first record is a first or a second mate).  MODE_SORTED_PAIR is NOT
        # sharded: file 2 would have to be cut by record index, not by byte offset (SURVEY.md §8e), which byte ranges do not give.  The
        # ranks' ranges are gathered on rank 0, whose engine runs the loop (at most 64 GiB in all); every rank gets the result.
        self.gathered = mode == api.MODE_SORTED_PAIR
        self.lines_per_step = 8 if mode == api.MODE_INTERLEAVED else 4  # a range starts where a loop iteration starts
        self.mode = mode
        self.rank = dist.get_rank() if dist.is_initialized() else 0
        self.world = dist.get_world_size() if dist.is_initialized() else 1
        self.tdev = tensor_device if tensor_device is not None else torch.device("cuda", device)
        indexed = mode in (api.MODE_INDEX, api.MODE_INDEX_PAIR)
        self.ctx = api.FastqInfo(mode, device=device, flags=api.FLAG_EXTERNAL_INDEX if indexed else 0)
        self.shard = api.FastqInfo(api.MODE_INDEX, device=device, index_capacity_hint=n_hint) if indexed else None
        self._keep = []
        # small host objects travel over a gloo group of their own: no device round trip, and no NCCL kernel that would have to
        # find room on SMs filled by a running clean-data pass (the per-round size exchange of the pipelined routing)
        self._cpu_group = None
        if self.world > 1 and dist.get_backend() != "gloo":
            import datetime
            self._cpu_group = dist.new_group(backend="gloo", timeout=datetime.timedelta(seconds=int(os.environ.get("FQG_GLOO_TIMEOUT_S", "120"))))  # a rank that died must not hang the others for half an hour
        # routing rounds over peer memory (CUDA IPC) instead of all-to-all exchanges: the default on GPUs.  Test hooks: FQG_P2P=0 runs
        # the exchanges (the fallback when a peer cannot be mapped) on GPUs; FQG_P2P=1 runs peer memory on CPU tensors (the gloo tests:
        # the stand-in device maps shared memory between the ranks)
        self.p2p = os.environ.get("FQG_P2P", "1" if self.tdev.type == "cuda" else "0") not in ("", "0")
        self._nccl_gather = self.world > 1 and self.tdev.type == "cuda" and dist.get_backend() == "nccl"
        self._gbuf = None
        # One copy stream per peer for the regions of a round.  Measured on 8 B200s: 43.3 ms per job with one stream — seven copies
        # of 60 MB one after the other take longer than the pass they should hide behind — 38.8 ms with seven; with four ranks no
        # difference (34.2 / 34.5 ms).
        self._copy_lanes = min(7, self.world - 1)
        self._arena, self._peer, self._arena_failed, self._p2p_ok, self._stage, self._zero = None, None, False, False, None, None
        self.rounds_done = 0  # routing rounds of the last run (tests, bench)
        self._plan, self._job, self._flagvals = None, 0, None
        self.gathered_jobs = 0  # feeds that sent every range to rank 0 (tiny inputs, a NUL-led header line, the sorted-pair mode)
        self.exact_reruns = 0  # jobs the speculative / pipelined path handed to the exact path (tests)
        self.host_ms = {"pack": 0.0}  # host time inside the peer-memory rounds, accumulated
        self.phase_ms = {}  # host wall time of the phases of run_device, accumulated over jobs (bench.py reports them)

    def route_description(self):
        """how the names of the last job reached their owners (bench.py's config line)"""
        if self.shard is None:
            return "no name index in this mode"
        if self.rounds_done and self._p2p_ok and self._plan and self._plan[0]["mode"] == "pass":
            return "written by the clean-data pass into per-owner regions, moved chunk by chunk into the owners' peer memory over NVLink (CUDA IPC) by the copy engines"
        if self.rounds_done and self._p2p_ok:
            return "chunk by chunk into the owners' peer memory over NVLink (CUDA IPC), beside the next chunk's pass"
        if self.rounds_done:
            return "chunk by chunk with all-to-all exchanges"
        return "one all-to-all over NCCL after the pass"

    # ------------------------------------------------------------------ helpers
    def _mine(self, rep, local_key, dup, unp, claimed, pair, with_hist=False):
        """this rank's part of the merged report"""
        f0, f1 = rep.file[0], rep.file[1]
        mine = {"key": local_key, "dup": dup, "unp": unp, "claimed": claimed,
                "err": bytes(ctypes.string_at(ctypes.addressof(rep.error), ctypes.sizeof(api.Error))) if local_key != KEY_NONE else None,
                "nrec": (int(f0.n_records), int(f1.n_records)), "num_rds": int(f0.num_rds), "min_rl": int(f0.min_rl), "max_rl": int(f0.max_rl),
                "rl1": (int(f1.min_rl), int(f1.max_rl)), "min_q": int(f0.min_qual), "max_q": int(f0.max_qual), "names": int(rep.n_index_entries),
                "mem": int(rep.index_mem) - 8, "sniff": ((int(f0.sniff_format), int(f0.color_space)), (int(f1.sniff_format), int(f1.color_space)))}
        if with_hist:
            mine["hist"] = _local_hist(self.ctx, f0, f1)
        return mine

    def _gather(self, obj):
        """Small host objects, one per rank, to every rank.  On GPUs: pickled into a fixed 16 KiB slot and gathered by one NCCL
        all-gather (the device is idle at the two places a job gathers — before its first pass and after its last owner kernel; a
        gloo gather of Python objects costs 0.7 ms with four ranks and 1 ms with eight, this 0.15 ms).  An object that does not
        fit says so in its slot and every rank repeats the gather over gloo."""
        if self.world == 1:
            return [obj]
        if self._nccl_gather:
            blob = pickle.dumps(obj, protocol=pickle.HIGHEST_PROTOCOL)
            n = len(blob) if len(blob) <= GATHER_SLOT - 8 else GATHER_SLOT  # (GATHER_SLOT: does not fit)
            if self._gbuf is None:
                self._gbuf = (torch.zeros(GATHER_SLOT, dtype=torch.uint8).pin_memory(), torch.zeros(GATHER_SLOT, dtype=torch.uint8, device=self.tdev),
                              torch.zeros(GATHER_SLOT * self.world, dtype=torch.uint8, device=self.tdev), torch.zeros(GATHER_SLOT * self.world, dtype=torch.uint8).pin_memory())
            mine_h, mine_d, all_d, all_h = self._gbuf
            mine_h[:8] = torch.frombuffer(bytearray(int(n).to_bytes(8, "little")), dtype=torch.uint8)
            if n < GATHER_SLOT:
                mine_h[8:8 + n] = torch.frombuffer(bytearray(blob), dtype=torch.uint8)
            mine_d.copy_(mine_h, non_blocking=True)
            dist.all_gather_into_tensor(all_d, mine_d)
            all_h.copy_(all_d, non_blocking=True)
            torch.cuda.current_stream().synchronize()
            raw = all_h.numpy()
            sizes = [int.from_bytes(raw[k * GATHER_SLOT:k * GATHER_SLOT + 8].tobytes(), "little") for k in range(self.world)]
            if all(x < GATHER_SLOT for x in sizes):
                return [pickle.loads(raw[k * GATHER_SLOT + 8:k * GATHER_SLOT + 8 + sizes[k]].tobytes()) for k in range(self.world)]
        out = [None] * self.world
        dist.all_gather_object(out, obj, group=self._cpu_group)
        return out

    def _sync(self):
        if self.tdev.type == "cuda":
            torch.cuda.synchronize()

    def _a2a(self, send, in_splits, out_splits):
        recv = torch.empty(sum(out_splits) + 64, dtype=torch.uint8, device=self.tdev)
        if self.world == 1:
            recv[:sum(out_splits)] = send[:sum(in_splits)]
        else:
            dist.all_to_all_single(recv[:sum(out_splits)], send[:sum(in_splits)], output_split_sizes=out_splits, input_split_sizes=in_splits)
        return recv

    def _feed_file(self, f, ptr, nbytes, gather0=False):
        """Steps 1-2 for one file: line phase, head exchange, sniff, feed.  Returns (records expected on this rank or None
        when the file was gathered on rank 0, records of the file over all ranks)."""
        W, r, ctx = self.world, self.rank, self.ctx
        last_rank = r == W - 1
        M = self.lines_per_step
        if nbytes > 0:
            nlines, ends_lf, first = ctx.prescan_device(f, ptr, nbytes, at_eof=last_rank)
            if M > 4:
                first = self._first_line_ends(ptr, nbytes, M)
        else:
            nlines, ends_lf, first = 0, True, [KEY_NONE] * M
        virt = 1 if (last_rank and nbytes > 0 and not ends_lf) else 0
        lfs = nlines - virt
        info = self._gather((lfs, ends_lf, first, nbytes, virt))
        G = [0] * (W + 1)
        for i in range(W):
            G[i + 1] = G[i] + info[i][0]
        skip, firstrec, cut = [0] * W, [0] * W, [0] * W
        degenerate = False
        for i in range(W):
            prev_lf = True if i == 0 else info[i - 1][1]
            skip[i] = 0 if (i == 0 or (prev_lf and G[i] % M == 0)) else ((M - G[i] % M) % M or M)
            if i > 0 and (info[i][0] < skip[i] or info[i][3] == 0):
                degenerate = True  # a range without a record start of its own (tiny inputs)
                break
            firstrec[i] = (G[i] + skip[i]) // 4
            cut[i] = info[i][2][skip[i] - 1] if skip[i] > 0 else 0
        total_lines = G[W] + info[W - 1][4]
        total_records = total_lines // 4
        if degenerate or info[0][3] == 0 or gather0:
            self.gathered_jobs += 1  # (tests: which jobs were NOT sharded)
            if sum(info[i][3] for i in range(W)) > (64 << 30):  # (every rank sees the same sizes: the refusal is collective)
                raise NotImplementedError("a sharded run that must be redone on one GPU, with more than 64 GiB of input")
            # tiny input: everything goes to rank 0, the other ranks hold an empty stream (the collectives below still run)
            sizes = [info[i][3] for i in range(W)]
            if r == 0:
                whole = torch.zeros(sum(sizes) + 64, dtype=torch.uint8, device=self.tdev)
                if sizes[0]:
                    whole[:sizes[0]] = _as_tensor(ptr, sizes[0], self.tdev)
                off = sizes[0]
                for s in range(1, W):
                    if sizes[s]:
                        dist.recv(whole[off:off + sizes[s]], s)
                    off += sizes[s]
                self._keep.append(whole)
                ctx.set_stream_start(f, 0, 0)
                if off:
                    ctx.feed_device(f, whole.data_ptr(), off, last=True)
                else:
                    ctx.feed(f, b"", last=True)
            else:
                if nbytes:
                    dist.send(_as_tensor(ptr, nbytes, self.tdev), 0)
                ctx.set_stream_start(f, 0, 0 if (self.gathered or M > 4) else total_records)  # (gathered / interleaved: this rank's empty report is not used)
                ctx.feed(f, b"", last=True)
            return None, total_records
        # the read-name format and colour space come from the file's first record, which rank 0 holds
        sn = ctx.sniff_device(f, ptr, nbytes, 0) if r == 0 else None
        sn = self._gather(sn)[0]
        if sn[0] >= 0:
            ctx.set_sniff(f, sn[0], sn[1])
        ctx.set_stream_start(f, skip[r], firstrec[r])
        self._feed_range(f, ptr, nbytes, cut)
        expected = (lfs + virt - skip[r] + (skip[r + 1] if r < W - 1 else 0)) // 4
        return expected, total_records

    def _head_line_ends(self, ptr, nbytes, k, enough=None, limit=None):
        """Ends (offsets behind the line feed) of the first k lines of this rank's range, fewer where the window has fewer, and the
        window's bytes.  The window starts at 16 KiB and grows sixteenfold until `enough(head, ends)` holds (by default: k ends were
        found), it holds the whole range, or it has reached `limit` bytes."""
        want = 1 << 14
        while True:
            n = min(nbytes, want)
            head = bytes(_as_tensor(ptr, n, self.tdev).cpu().numpy())
            ends, pos = [], -1
            while len(ends) < k:
                pos = head.find(b"\n", pos + 1)
                if pos < 0:
                    break
                ends.append(pos + 1)
            if (enough(head, ends) if enough else len(ends) == k) or n == nbytes or (limit and want >= limit):
                return head, ends
            want *= 16

    def _first_line_ends(self, ptr, nbytes, k):
        """ends of the first k lines of this rank's range, KEY_NONE where the range has fewer"""
        ends = self._head_line_ends(ptr, nbytes, k)[1]
        return ends + [KEY_NONE] * (k - len(ends))

    def _guess_phase(self, ptr, nbytes):
        """Line class (0 header, 1 sequence, 2 plus, 3 quality) of the line this range starts in, from the range's own first lines:
        a complete line that is exactly "+" is a plus line.  Returns (ok, class, ends of the first four lines, ends with LF, bytes
        per record over the first complete records, raw length of the first complete sequence line)."""
        if nbytes < 4096:
            return (False, 0, [KEY_NONE] * 4, True, 0.0, 0, b"")
        # long lines: the window grows to 256 KiB (short reads are answered by the first 16 KiB)
        head, ends = self._head_line_ends(ptr, nbytes, 64, enough=lambda h, e: len(e) >= 5 and _plus_line_class(h, e) is not None, limit=1 << 18)
        last = bytes(_as_tensor(ptr + nbytes - 1, 1, self.tdev).cpu().numpy())
        cls = _plus_line_class(head, ends)
        if cls is None or len(ends) < 5:
            return (False, 0, [KEY_NONE] * 4, last == b"\n", 0.0, 0, b"")
        k = (len(ends) - 1) // 4
        seq = next(ends[i] - ends[i - 1] for i in range(1, 5) if (cls + i) % 4 == 1)
        return (True, cls, ends[:4], last == b"\n", (ends[4 * k] - ends[0]) / k, seq, head[:min(ends[0], 1024)])

    def _plan_routes(self, infos, pair):
        """The routing rounds of a job, from the ranks' guesses about their ranges (infos[f][rank]): per file the number of rounds
        (as many as the longest range has chunks, so that no round carries more than one chunk; ranks with fewer chunks add empty
        rounds: the rounds are collective), the shape of a region, and where the file's regions start in every rank's arena.
        Three ways for the names of a chunk to reach their owners (`mode`):
          pass  the clean-data pass writes them into per-owner regions while it validates (GPU, peer memory); the copy engines move
                the regions; what the per-record kernels validated (the seams of the byte ranges) follows in one packed round
          pack  a pack kernel fills dense regions beside the next pass, the copy engines move them (peer memory)
          a2a   the same pack kernel, regions exchanged with all-to-all (no peer memory; the gloo tests)"""
        W = self.world
        chunk = api.feed_chunk_bytes()
        # (a chunk restarts at the record the chunk before it cut, so a range may take one chunk more than its bytes suggest:
        # count with slightly shorter chunks; a round too many is an empty round, a round too few would overflow the last one)
        step = chunk - min(chunk // 4, 8 << 20)
        # name bytes travel with the tuples when the mate loop has to compare them: 16-byte units for the length of the first
        # record's name and a few bytes more (a longer name later in the file overflows its slot: the exact path takes over)
        units = 0
        if pair:
            first = infos[0][0][6]
            line = first[1:first.index(b"\n")] if b"\n" in first else first[1:]
            name = line.split(b" ")[0] if self._sniff[0][0] == 1 else line
            units = max(1, -(-(len(name) + 3) // 16))
        # (test hook: FQG_ROUTE_IN_PASS=0 takes mode `pack` on GPUs, the mode of the stand-in device, whose pass routes nothing)
        nb = self.ctx.route_blocks() if (self.p2p and os.environ.get("FQG_ROUTE_IN_PASS", "1") not in ("", "0")) else 0
        tiny = os.environ.get("FQG_TEST_SLOT_CAP")  # test hook: regions far too small, so that the overflow path is taken
        plan, base = [], FLAG_AREA
        self._job += 1
        for info in infos:
            rounds = min(FLAG_ROUNDS - 2, max(1, max(-(-x[7] // step) for x in info)))
            names_chunk = min(chunk, max(x[7] for x in info)) / max(min(x[4] for x in info), 16.0)  # (the estimate comes from the first records of every range)
            pl = {"rounds": rounds, "units": units, "round": 0, "fires": 0, "base": base}
            if nb:  # one stretch per CTA of the pass and owner, with room to spare
                # (the CTAs claim tiles as they go: a CTA may get a few tiles more than its share)
                per_tile = 31744.0 / max(min(x[4] for x in info), 16.0)
                stride = int(tiny) if tiny else int(names_chunk / nb / W * 1.2 + 4 * (per_tile / W + 16)) + 32
                left = int(tiny) if tiny else 16384
                pl.update(mode="pass", nblocks=nb, stride=stride, region=api.route_region_bytes(nb, stride, units),
                          left_stride=left, left_region=api.route_region_bytes(1, left, units))
                base += rounds * W * pl["region"]
                pl["left_base"] = base
                base += W * pl["left_region"]
            else:  # names of one chunk for one owner, with room to spare
                cap = int(tiny) if tiny else int(names_chunk / W * 1.25) + 4096
                pl.update(mode="pack", nblocks=1, stride=cap, region=api.route_region_bytes(1, cap, units))
                base += rounds * W * pl["region"]
            plan.append(pl)
        est = sum(x[7] / max(x[4], 16.0) for x in infos[0]) / W
        self.shard.shard_reserve(int(est * 1.05) + 4096)
        self._plan, self._inflight, self._hook_exc = plan, [], None
        self._p2p_ok = self.p2p and self._ensure_arena(base)
        if not self._p2p_ok:
            for pl in plan:
                pl["mode"] = "a2a"
        need = max([2 * W * pl["region"] for pl in plan if pl["mode"] == "pass"] + [W * pl["region"] for pl in plan if pl["mode"] == "pack"] + [0])
        if need and (self._stage is None or self._stage.numel() < need + 64):
            self._stage = torch.zeros(need + 64, dtype=torch.uint8, device=self.tdev)
        if self._zero is None:
            self._zero = torch.zeros(64, dtype=torch.uint8, device=self.tdev)
        # the flag words this rank will write behind its regions: job and round, never the same value twice
        self._flagvals = torch.arange(1, FLAG_ROUNDS + 1, dtype=torch.int64, device=self.tdev) + (self._job << 20)
        self._sync()

    def _feed_file_speculative(self, f, ptr, nbytes, info, routed=False):
        """Steps 1-2 without counting the line feeds of the range first: every rank takes the line phase of its range from its own
        first plus line (`info`: the ranks' guesses, gathered).  A wrong guess cannot go unnoticed on a valid file (a sequence line
        lands where a header or a plus line is expected), so any error afterwards simply sends the whole job through the exact path."""
        W, r, ctx = self.world, self.rank, self.ctx
        skip, cut = [0] * W, [0] * W
        for i in range(1, W):
            cls0, prev_lf = info[i][1], info[i - 1][3]
            skip[i] = 0 if (prev_lf and cls0 == 0) else ((4 - cls0) % 4 or 4)
            cut[i] = info[i][2][skip[i] - 1] if skip[i] > 0 else 0
        sn = self._sniff[f]
        if sn[0] >= 0:
            ctx.set_sniff(f, sn[0], sn[1])
        ctx.set_stream_start(f, skip[r], 0)  # record numbers inside the range: they only matter when something is wrong
        ctx.set_line_hint(f, info[r][5])  # a range that starts inside the file never sees the first record's sequence line
        if routed:
            self._cur = f
            pl = self._plan[f]
            if pl["mode"] == "pass":  # the clean-data pass of every chunk writes into two alternating sets of W regions
                st = self._stage.data_ptr()
                ctx.set_route(f, [st + o * 2 * pl["region"] for o in range(W)], pl["region"], 2, pl["stride"], pl["units"])
            ctx.set_chunk_hook(self._on_chunk)
        t0 = time.perf_counter()
        try:
            self._feed_range(f, ptr, nbytes, cut)
        finally:
            self.host_ms["feed"] = self.host_ms.get("feed", 0.0) + (time.perf_counter() - t0) * 1e3
            if routed:
                ctx.set_chunk_hook(None)
        if routed:
            pl = self._plan[f]
            if pl["mode"] == "pass":
                while pl["round"] < pl["rounds"]:
                    self._pass_round(beside=False)  # (no pass is running any more: the owner's kernel may take the whole GPU)
                self._left_round()
            else:
                while pl["round"] < pl["rounds"] - 1:
                    self._route_round(False)
                self._route_round(True)
            self.rounds_done += pl["round"]

    def _feed_range(self, f, ptr, nbytes, cut):
        """The seam between two byte ranges, then the feed.  cut[i]: bytes of range i in front of its first record start (the rest
        of the record the end of range i-1 cut).  This rank sends its own to rank r-1, receives those of range r+1 and feeds its
        range followed by them."""
        W, r, ctx = self.world, self.rank, self.ctx
        head, reqs = None, []
        if r > 0 and cut[r] > 0:
            view = _as_tensor(ptr, cut[r], self.tdev)
            reqs.append(dist.isend(view, r - 1))
            self._keep.append(view)
        if r < W - 1 and cut[r + 1] > 0:
            head = torch.zeros(cut[r + 1] + 64, dtype=torch.uint8, device=self.tdev)
            reqs.append(dist.irecv(head[:cut[r + 1]], r + 1))
            self._keep.append(head)
        _dbg(f"rank {r} file {f} seam exchange, {len(reqs)} requests")
        for q in reqs:
            q.wait()
        if reqs:
            self._sync()  # the library reads the head on its own stream
        _dbg(f"rank {r} file {f} seam exchange done")
        if r == W - 1:
            ctx.feed_device(f, ptr, nbytes, last=True)
        else:
            ctx.feed_device(f, ptr, nbytes, last=False)
            if head is not None:
                ctx.feed_device(f, head.data_ptr(), cut[r + 1], last=True)
            else:
                ctx.feed(f, b"", last=True)

    # ------------------------------------------------------------------ pipelined routing (one file, tuples only)
    def _on_chunk(self, file):
        """Chunk hook of the feeding context (fqg_set_chunk_hook): called once per chunk, for a chunk of the clean-data pass while
        that pass runs on the GPU.  Every rank performs exactly the planned number of rounds per file (they are collective); the
        first call of a file has nothing to route yet."""
        pl = self._plan[self._cur]
        pl["fires"] += 1
        t0 = time.perf_counter()
        if self._hook_exc is None:
            try:
                if pl["mode"] == "pass":
                    done = self.ctx.route_chunks(self._cur)[0]  # chunks whose regions the pass has completed
                    while pl["round"] < min(done, pl["rounds"]):
                        self._pass_round()
                elif pl["fires"] >= 2 and pl["round"] < pl["rounds"] - 1:
                    self._route_round(False)
            except BaseException as ex:  # an exception cannot cross the C frames above us
                self._hook_exc = ex
        self.host_ms["hook"] = self.host_ms.get("hook", 0.0) + (time.perf_counter() - t0) * 1e3

    def _pass_round(self, beside=True):
        """Round j of the current file, mode `pass`: the regions the clean-data pass of this rank's chunk j filled (none: an empty
        header) go to their owners' arenas through the copy engines; the pass that will reuse the regions waits for the copies."""
        W, r, f, ctx = self.world, self.rank, self._cur, self.ctx
        pl = self._plan[f]
        j, region = pl["round"], pl["region"]
        have = j < self.ctx.route_chunks(f)[0]
        if os.environ.get("FQG_DEBUG_ROUTE"):
            _dbg(f"rank {r} file {f} pass round {j} of {pl['rounds']} have={have} chunks={self.ctx.route_chunks(f)}")
        off = pl["base"] + (j * W + r) * region
        st = self._stage.data_ptr()
        t1 = time.perf_counter()
        for d in range(W):
            o = (r + d) % W
            src, n = (st + (o * 2 + j % 2) * region, region) if have else (self._zero.data_ptr(), 16)
            self._send_region(o, off, src, n, f, j, lane=0 if d == 0 else 1 + (d - 1) % self._copy_lanes)  # (the peers' regions on copy streams side by side)
        self.ctx.side_mark()
        self.host_ms["pack"] += (time.perf_counter() - t1) * 1e3
        # The owner's kernel waits for its sources on the device (their flag words).  It takes the whole device between two passes:
        # behind the pass that is running now (launched ahead), in front of the next one.  Squeezed in beside a pass (one block
        # per SM) it was measured at a quarter of its speed, and the pass lost a third of its own.
        if beside:
            self.shard.order_after(True, ctx, False)
        self._owner_round(self._arena[0] + pl["base"] + j * W * region, region, pl["nblocks"], pl["stride"], pl["units"], f, False, flag_round=j)
        if beside and j + 2 < pl["rounds"]:  # (the last rounds have no pass behind them that would have to wait: the next file starts at once)
            ctx.order_after(False, self.shard, True)
        pl["round"] += 1

    def _left_round(self):
        """After the last chunk of a file, mode `pass`: what the per-record kernels validated (the seams between byte ranges, a short
        last chunk) has name descriptors; one packed round takes them to their owners.  Then every round of the file lands."""
        f = self._cur
        pl = self._plan[f]
        if os.environ.get("FQG_DEBUG_ROUTE"):
            _dbg(f"rank {self.rank} file {f} left round, names left {self.ctx.names_new(f)}")
        # (the pack kernel runs on the side stream, behind the copies out of the staging regions it overwrites: fqg_side_mark of the
        # last round joined the copy lanes into that stream)
        self._packed_round(f, pl["left_base"], pl["left_region"], pl["left_stride"], pl["units"], pl["rounds"], False)
        self.ctx.side_mark()  # the next file's first pass writes into the staging regions: behind these copies

    def _packed_round(self, f, base, region, cap, units, flag_round, beside):
        """One round of names packed by the pack kernel (mode `pack`, and the left round of mode `pass`), over peer memory: the
        region of every owner is `region` bytes at base + (source rank) * region in the owner's arena.  The pack kernel writes this
        rank's own region straight into its arena and the others into staging, the copy engines move those to their owners with a
        flag word behind each, and this rank's index shard takes the round (beside the running pass if `beside`).  The pack kernel
        runs on the side stream, behind the copies of the round before out of the staging regions it overwrites.  (Stores from the
        pack kernel straight into the peers' arenas were as fast with two ranks but slowed every pass threefold at eight: 5.9 M
        remote stores per round and rank.)"""
        W, r = self.world, self.rank
        off = base + r * region
        st = self._stage.data_ptr()
        t0 = time.perf_counter()
        self.ctx.names_pack_slots(f, [self._arena[0] + off if o == r else st + o * region for o in range(W)], cap, units)
        for d in range(W):
            o = (r + d) % W
            self._send_region(o, off, None if o == r else st + o * region, region, f, flag_round)
        self.host_ms["pack"] += (time.perf_counter() - t0) * 1e3
        self._owner_round(self._arena[0] + base, region, 1, cap, units, f, beside, flag_round=flag_round)

    def _flag_off(self, f, j):
        return 8 * ((f * FLAG_ROUNDS + j) * self.world)

    def _send_region(self, o, off, src, n, f, j, lane=0):
        """n bytes from src to `off` in owner o's arena (src None: nothing to copy), then, behind them on the same copy stream, the flag
        word of round j that tells o's kernel they are there"""
        arena = self._arena[0] if o == self.rank else self._peer[o]
        if src is not None:
            self.ctx.side_copy_lane(lane, arena + off, src, n)
        self.ctx.side_copy_lane(lane, arena + self._flag_off(f, j) + 8 * self.rank, self._flagvals.data_ptr() + 8 * j, 8)

    def _ensure_arena(self, need):
        """Peer-writable receive memory (CUDA IPC over NVLink): `need` bytes on every rank, mapped by every other rank.  Collective;
        False when some rank cannot map a peer (the rounds then use all-to-all exchanges)."""
        W, r = self.world, self.rank
        if self._arena is not None and self._arena[1] >= need:
            return True
        if self._arena_failed:
            return False
        self._sync()
        ok = True
        try:
            if self._arena is not None:
                for s, pp in enumerate(self._peer):
                    if s != r:
                        self.ctx.ipc_close(pp)
                self._gather(0)  # nobody maps the old arena any more
                self.shard.ipc_free(self._arena[0])
                self._arena = None
            size = int(need * 1.1) + (1 << 20)
            ptr, handle = self.shard.ipc_alloc(size)
            _as_tensor(ptr, FLAG_AREA, self.tdev).zero_()  # no flag word has been written yet (the gathers below: before anybody writes one)
            self._sync()
        except RuntimeError:
            ok, ptr, handle, size = False, 0, b"", 0
        handles = self._gather(handle if ok else None)
        peers = [ptr] * W
        if all(h is not None for h in handles):
            for s in range(W):
                if s != r:
                    try:
                        peers[s] = self.ctx.ipc_open(handles[s])
                    except RuntimeError:
                        ok = False
        else:
            ok = False
        if not all(self._gather(ok)):
            # some rank could not allocate or map: nobody keeps half an arena (the rounds use all-to-all exchanges from now on)
            for sidx in range(W):
                if sidx != r and peers[sidx] != ptr:
                    try:
                        self.ctx.ipc_close(peers[sidx])
                    except RuntimeError:
                        pass
            self._gather(0)  # nobody maps this rank's memory any more
            if ptr:
                self.shard.ipc_free(ptr)
            self._arena_failed = True
            return False
        self._arena, self._peer = (ptr, size), peers
        return True

    def _owner_round(self, regions_ptr, region_bytes, nblocks, stride, units, f, beside, flag_round=None):
        """this rank's index shard takes a round: file 1's names are inserted, file 2's claim them"""
        kw = {}
        if flag_round is not None:
            kw = {"flags_ptr": self._arena[0] + self._flag_off(f, flag_round), "expect": (self._job << 20) + flag_round + 1}
        if f == 0:
            self.shard.shard_insert_slots(regions_ptr, self.world, region_bytes, nblocks, stride, beside=beside, units=units, **kw)
        else:
            self.shard.shard_claim_slots(regions_ptr, self.world, region_bytes, nblocks, stride, beside=beside, units=units, **kw)

    def _route_round(self, final):
        """Modes `pack` and `a2a`: pack the names that were not routed yet into one fixed-capacity region per owner.  Over peer memory
        the round is one packed round; otherwise start their exchange and hand the rounds whose exchange has finished to this rank's
        index shard.  Either way the shard takes them beside the running pass unless this is the last round."""
        W, f = self.world, self._cur
        pl = self._plan[f]
        if self._p2p_ok:
            self._packed_round(f, pl["base"] + pl["round"] * W * pl["region"], pl["region"], pl["stride"], pl["units"], pl["round"], not final)
            pl["round"] += 1
            return
        units = pl["units"]
        mx = max(self._gather(self.ctx.names_new(f)))
        per = -(-mx // W)
        cap = max(1, mx) if mx <= 8192 else int(per * 1.03) + 6 * int(per ** 0.5) + 1024
        if os.environ.get("FQG_TEST_SLOT_CAP"):  # test hook: regions far too small, so that the overflow path is taken
            cap = int(os.environ["FQG_TEST_SLOT_CAP"])
        stride = api.route_region_bytes(1, cap, units)
        send = torch.empty(W * stride, dtype=torch.uint8, device=self.tdev)
        recv = torch.empty(W * stride, dtype=torch.uint8, device=self.tdev)
        self.ctx.names_pack_slots(f, [send.data_ptr() + o * stride for o in range(W)], cap, units)
        if W > 1:
            work = dist.all_to_all_single(recv, send, async_op=True)
        else:
            recv, work = send, None
        self._inflight.append((recv, send, cap, work, f))
        pl["round"] += 1
        while len(self._inflight) > (0 if final else 1):
            recv, send, cap, work, ff = self._inflight.pop(0)
            if work is not None:
                work.wait()
            if self.tdev.type == "cuda":
                torch.cuda.current_stream().synchronize()  # not the device: the pass on the library's stream keeps running
            self._owner_round(recv.data_ptr(), api.route_region_bytes(1, cap, self._plan[ff]["units"]), 1, cap, self._plan[ff]["units"], ff, not final)
            self._keep += [recv, send]

    def _route_names(self, f, with_bytes=True):
        """Step 3, sender side: pack the names of file f by owner and exchange them.  Returns what the owner needs.
        with_bytes=False sends the 24-byte tuples only (a quarter of the volume, no byte gathering)."""
        W, r = self.world, self.rank
        counts, nb = self.ctx.names_count(f, W)
        if not with_bytes:
            nb = [0] * W
        theirs = self._gather((counts, nb))
        in_meta, in_blob = [c * 24 for c in counts], list(nb)
        out_cnt = [theirs[s][0][r] for s in range(W)]
        out_meta, out_blob = [c * 24 for c in out_cnt], [theirs[s][1][r] for s in range(W)]
        meta_base, blob_base = [0] * W, [0] * W
        for o in range(1, W):
            meta_base[o] = meta_base[o - 1] + counts[o - 1]
            blob_base[o] = blob_base[o - 1] + nb[o - 1]
        send_meta = torch.empty(sum(in_meta) + 64, dtype=torch.uint8, device=self.tdev)
        send_blob = torch.empty(sum(in_blob) + 64, dtype=torch.uint8, device=self.tdev)
        self.ctx.names_pack(f, W, send_meta.data_ptr(), send_blob.data_ptr() if with_bytes else 0, meta_base, blob_base)
        self._sync()
        recv_meta = self._a2a(send_meta, in_meta, out_meta)
        recv_blob = self._a2a(send_blob, in_blob, out_blob)
        self._sync()
        ms, bs, acc = [0], [], 0
        for s in range(W):
            ms.append(ms[-1] + out_cnt[s])
            bs.append(acc)
            acc += out_blob[s]
        self._keep += [recv_meta, recv_blob]
        return recv_meta, recv_blob, ms, bs

    # ------------------------------------------------------------------ one job
    def _run_gathered(self, ptr, nbytes, name, ptr2, nbytes2, name2, empty_ok, no_enc_ok):
        """MODE_INTERLEAVED / MODE_SORTED_PAIR: the ranges travel to rank 0 (the path a tiny input takes in the other modes), whose
        engine sees the whole stream; the other ranks feed nothing."""
        ctx, r = self.ctx, self.rank
        ctx.reset()
        self._keep = []
        two = self.mode == api.MODE_SORTED_PAIR
        self._feed_file(0, ptr, nbytes, gather0=True)
        if two:
            self._feed_file(1, ptr2, nbytes2, gather0=True)
        rep = ctx.finish()
        tr = ctx.render(rep, name, name2 if two else None, empty_ok=empty_ok, no_enc_ok=no_enc_ok) if r == 0 else None
        mine = (int(rep.error.event_key) if rep.error.code != 0 else KEY_NONE, int(rep.file[0].n_records), int(rep.file[1].n_records), tr)
        got = self._gather(mine)[0]
        out = {"report": rep if r == 0 else None, "event_key": got[0], "n_records": got[1], "n_records2": got[2], "n_index_entries": 0, "n_index_left": 0}
        if r == 0:
            out["transcript"] = tr
        return out

    def run_device(self, ptr, nbytes, name="-", ptr2=None, nbytes2=0, name2=None, empty_ok=False, no_enc_ok=False, _exact=False, _gather0=False):
        """ptr/nbytes (and ptr2/nbytes2 for MODE_INDEX_PAIR): this rank's byte range of each file in device memory (16-byte
        aligned, 64 readable bytes after it).  Returns the merged report and, on rank 0, the rendered (rc, stdout, stderr)."""
        W, r, ctx = self.world, self.rank, self.ctx
        if self.gathered:
            return self._run_gathered(ptr, nbytes, name, ptr2, nbytes2, name2, empty_ok, no_enc_ok)
        tm = {"t": time.perf_counter()}

        def lap(name):
            now = time.perf_counter()
            self.phase_ms[name] = self.phase_ms.get(name, 0.0) + (now - tm["t"]) * 1e3
            tm["t"] = now
        ctx.reset()
        if self.shard:
            self.shard.reset()
        self._keep = []
        lap("reset")
        pair = self.mode == api.MODE_INDEX_PAIR
        allr = None  # every rank's report, once gathered
        again = dict(name=name, ptr2=ptr2, nbytes2=nbytes2, name2=name2, empty_ok=empty_ok, no_enc_ok=no_enc_ok, _exact=True)
        routed = self.shard is not None
        self.rounds_done = 0
        # (a world of one takes the same path when it has an index shard: the single-GPU tests of the pipelined routing)
        speculative = (not _exact) and (W > 1 or routed) and self.mode != api.MODE_INTERLEAVED
        files = [(0, ptr, nbytes)] + ([(1, ptr2, nbytes2)] if pair else [])
        if speculative:
            # every rank guesses the line phase of its ranges from their own first lines; rank 0, which holds the first record of each
            # file, sniffs the read-name format and colour space (src/fastq.c:459-485); all of it travels in one gather
            mine = [self._guess_phase(p, n) + (n,) for _, p, n in files]
            sn = [ctx.sniff_device(f, p, n, 0) if (r == 0 and n >= 4096) else None for f, p, n in files]
            got = self._gather((mine, sn))
            infos = [[g[0][k] for g in got] for k in range(len(files))]
            self._sniff = got[0][1]
            speculative = all(all(x[0] for x in info) and info[0][1] == 0 for info in infos) and all(x is not None for x in self._sniff)
        if speculative:
            lap("guess")
            if routed:
                self._plan_routes(infos, pair)
            lap("plan")
            if pair:
                ctx.set_file_total(0, 1 << 40)  # (the mate loop's event keys continue after file 1's: only their order matters here)
            for (f, p, n), info in zip(files, infos):
                self._feed_file_speculative(f, p, n, info, routed=routed)
                lap(f"file{f}")
            rep = ctx.finish()
            lap("finish")
            # a NUL-led header line ended this rank's range early and quietly (src/fastq.c:248): not an error here, but the ranges
            # behind it do not exist for the reference — the exact path sorts that out
            cut_short = any(int(rep.file[f].n_records) < ctx.records_fed(f) for f, _, _ in files)
            claimed = 0
            if routed:
                # The names went to their owners while the ranges were validated.  One file: tuples only — an equal hash decides
                # nothing.  Two files: with their bytes — the owner knows a duplicate, an unpaired mate or a name left over when it
                # sees one, but the reference's message (which record, which line) is the exact path's business.  So is a region,
                # slot or table that overflowed, a chunk redone by the two-pass kernels after its names had left, and any error.
                _dbg(f"rank {r} waits for its owner kernels")
                inserted, equal, overflow, claimed, unpaired = self.shard.shard_slots_result()
                broken = any(ctx.route_chunks(f)[1] for f, _, _ in files)  # a chunk whose names the pass should have routed went to the per-record kernels
                mine_bad = rep.error.code != 0 or cut_short or equal > 0 or unpaired > 0 or overflow or broken or ctx.path_counts()["two_pass_fallbacks"] > 0 or self._hook_exc is not None
                # (the merge below needs every rank's report: it travels in the same gather)
                sums = self._gather((bool(mine_bad), inserted, claimed, int(rep.n_index_entries), int(rep.file[1].n_records),
                                     None if mine_bad else self._mine(rep, KEY_NONE, (KEY_NONE, 0, b""), (KEY_NONE, 0, b""), claimed, pair, with_hist=True),
                                     self._hook_exc is not None))
                bad = any(x[0] for x in sums)
                tot_ins, tot_cl, tot_names, tot_mates = (sum(x[k] for x in sums) for k in (1, 2, 3, 4))
                _dbg(f"rank {r} verdict: error {rep.error.code} cut_short {cut_short} inserted {inserted} equal {equal} overflow {overflow} claimed {claimed} unpaired {unpaired} broken {broken} "
                     f"two_pass {ctx.path_counts()['two_pass_fallbacks']} | totals inserted {tot_ins} names {tot_names} claimed {tot_cl} mates {tot_mates}")
                if tot_ins != tot_names or (pair and (tot_cl != tot_names or tot_cl != tot_mates)):
                    bad = True  # a name was dropped on its way, a mate found nothing to claim, or names of file 1 are left over
                if self._hook_exc is not None:
                    raise self._hook_exc
                if any(x[6] for x in sums):  # every rank leaves together: nobody waits in a collective for the rank that failed
                    raise RuntimeError("the chunk hook of another rank failed (its exception is raised there)")
            else:
                bad = any(self._gather(rep.error.code != 0 or cut_short))  # every rank takes the same turn: the steps below are collective
            if bad:
                self.exact_reruns += 1
                return self.run_device(ptr, nbytes, **again)  # an error, a duplicate name or a wrong guess: the exact path decides
            if routed:
                allr = [x[5] for x in sums]
            local_key, T0, T1 = KEY_NONE, 0, 0
            dup, unp = (KEY_NONE, 0, b""), (KEY_NONE, 0, b"")
            lap("verdict")
        if not speculative:
            exp0, T0 = self._feed_file(0, ptr, nbytes, gather0=_gather0)
            exp1, T1 = None, 0
            if pair:
                ctx.set_file_total(0, T0)
                if T0 > 0:
                    exp1, T1 = self._feed_file(1, ptr2, nbytes2)
            rep = ctx.finish()
            local_key = rep.error.event_key if rep.error.code != 0 else KEY_NONE
            stopped = (exp0 is not None and rep.file[0].n_records < exp0) or (exp1 is not None and rep.file[1].n_records < exp1)
            # A NUL-led header line ends a file quietly (src/fastq.c:248): nothing behind it exists for the reference, on this rank
            # (the engine restricts itself) or on the ranks behind it.  Rare enough for the simplest cure: the ranges are gathered on
            # rank 0, whose engine knows the rule; the other ranks keep their part in the collectives with empty streams.
            if any(self._gather(bool(rep.error.code == 0 and stopped))):
                if pair or _gather0:
                    raise NotImplementedError("NUL-led header line (early clean EOF) in a sharded run of two files")
                self.exact_reruns += 1
                return self.run_device(ptr, nbytes, **dict(again, _gather0=True))
            # -- 3. names to their owners
            dup, unp, claimed = (KEY_NONE, 0, b""), (KEY_NONE, 0, b""), 0
            if self.shard is not None:
                # one file: the tuples travel alone first; only if some owner met an equal hash (a duplicate name or a 64-bit collision) is
                # the exchange repeated with the name bytes, which the owner then compares.  The mate loop needs the bytes anyway.
                coll = 1
                if not pair:
                    meta, blob, ms, bs = self._route_names(0, with_bytes=False)
                    self.shard.shard_insert(meta.data_ptr(), ms[-1], 0, ms, bs)
                    dkey, drec, dname, coll = self.shard.shard_result()
                    coll = sum(self._gather(coll))
                    if coll:
                        self.shard.reset()
                if coll:
                    meta, blob, ms, bs = self._route_names(0)
                    self.shard.shard_insert(meta.data_ptr(), ms[-1], blob.data_ptr(), ms, bs)
                    dkey, drec, dname, coll = self.shard.shard_result()
                dup = (dkey, drec, dname)
                if pair and T0 > 0:
                    meta2, blob2, ms2, bs2 = self._route_names(1)
                    self.shard.shard_claim(meta2.data_ptr(), ms2[-1], blob2.data_ptr(), ms2, bs2, T0 + 1)
                    ukey, urec, uname, claimed, coll2 = self.shard.shard_claim_result()
                    unp = (ukey, urec, uname)
                    coll += coll2
                # (two different names with one 64-bit hash are no event any more: the owners compare the bytes behind every equal
                # hash and walk on to the next slot, like the reference walks its chain, src/hash.c:38-45)
                if sum(self._gather(coll)):
                    raise RuntimeError("internal: an owner could not judge an equal hash although the name bytes travelled")
        # -- 4. merge
        if allr is None:
            allr = self._gather(self._mine(rep, local_key, dup, unp, claimed, pair))
        N0, N1 = sum(a["nrec"][0] for a in allr), sum(a["nrec"][1] for a in allr)
        names_total = sum(a["names"] for a in allr)
        left = names_total - sum(a["claimed"] for a in allr)
        cands = [(a["key"], "local", a) for a in allr] + [(a["dup"][0], "dup", a) for a in allr] + [(a["unp"][0], "unp", a) for a in allr]
        if pair and T0 > 0 and left > 0:
            cands.append((((T0 + 1 + N1 + 1) << 6), "left", None))
        best, kind, holder = min(cands, key=lambda c: c[0])
        merged = api.Report()
        merged.mode = self.mode
        m0 = merged.file[0]
        m0.n_records, merged.file[1].n_records = N0, N1
        m0.num_rds = sum(a["num_rds"] for a in allr)
        m0.min_rl = min(a["min_rl"] for a in allr)
        m0.max_rl = max(a["max_rl"] for a in allr)
        m0.min_qual = min(a["min_q"] for a in allr)
        m0.max_qual = max(a["max_q"] for a in allr)
        for f in (0, 1):  # sniff lines: decided by the rank that holds the file's first record
            fmt, col = next((a["sniff"][f] for a in allr if a["nrec"][f] > 0), allr[0]["sniff"][f])
            merged.file[f].sniff_format, merged.file[f].color_space = fmt, col
        merged.n_index_entries = names_total
        merged.n_index_left = left
        merged.index_mem = 8 + sum(a["mem"] for a in allr)
        merged.reads_before_error[0], merged.reads_before_error[1] = (N0 // 2 if self.mode == api.MODE_INTERLEAVED else N0), N1  # (loop iterations: pairs)
        if best != KEY_NONE:
            step = best >> 6
            e = merged.error
            if kind == "local":
                ctypes.memmove(ctypes.addressof(e), holder["err"], ctypes.sizeof(api.Error))
            elif kind == "dup":
                e.code, e.file, e.msg_file, e.record = E_DUP, 0, 0, holder["dup"][1]
                e.line = 4 * (holder["dup"][1] + 1)
                e.name = holder["dup"][2][:1023]
                e.name_len = len(holder["dup"][2][:1023])
            elif kind == "unp":
                e.code, e.file, e.msg_file, e.record = E_UNPAIRED, 1, 1, holder["unp"][1]
                e.line = 4 * (holder["unp"][1] + 1)
                e.name = holder["unp"][2][:1023]
                e.name_len = len(holder["unp"][2][:1023])
            else:
                e.code, e.file, e.msg_file, e.a = E_LEFTOVER, 0, 0, left
            e.event_key = best
            if pair and step >= T0 + 1:
                merged.reads_before_error[0], merged.reads_before_error[1] = T0, min(step - (T0 + 1), N1)
            else:
                merged.reads_before_error[0], merged.reads_before_error[1] = step, 0
        # median over the merged histogram (src/fastq_info.c:39-55); the mate loop counts into file 1's histogram too
        lo, hi = int(m0.min_rl), int(m0.max_rl)
        for a in allr:
            if a["rl1"][1] > 0:
                lo, hi = min(lo, a["rl1"][0]), max(hi, a["rl1"][1])
        med = MAX_READ_LENGTH
        if m0.num_rds == 1 and not (pair and T0 > 0):
            med = int(m0.min_rl)
        elif m0.num_rds > 1 and lo <= hi < MAX_READ_LENGTH and all("hist" in a for a in allr):
            # every rank's histogram came with its report: summed here
            total, acc, med = [0] * (hi - lo + 1), 0, MAX_READ_LENGTH
            for a in allr:
                if a["hist"] is not None:
                    for i, c in enumerate(a["hist"][1]):
                        total[a["hist"][0] - lo + i] += c
            for i, c in enumerate(total):
                acc += c
                if acc > m0.num_rds // 2:
                    med = lo + i
                    break
        elif m0.num_rds > 1 and lo <= hi < MAX_READ_LENGTH:
            h = torch.from_numpy(self.ctx.hist_range(0, lo, hi).astype("int64")).to(self.tdev)
            if W > 1:
                dist.all_reduce(h)
            c = torch.cumsum(h, 0)
            over = c > m0.num_rds // 2
            med = lo + int(torch.nonzero(over)[0]) if bool(over.any()) else MAX_READ_LENGTH
        merged.median_rl = med
        lap("merge")
        out = {"report": merged, "event_key": best, "n_records": N0, "n_records2": N1, "n_index_entries": names_total, "n_index_left": left}
        if r == 0:
            out["transcript"] = self.ctx.render(merged, name, name2 if pair else None, empty_ok=empty_ok, no_enc_ok=no_enc_ok)
        return out


GATHER_SLOT = 16384  # bytes per rank in the NCCL gather of small host objects


def _local_hist(ctx, f0, f1):
    """this rank's read lengths (src/fastq_info.c:39-55 counts the mates into the same histogram): (lowest length, counts)"""
    lo, hi = int(f0.min_rl), int(f0.max_rl)
    if int(f1.max_rl) > 0:
        lo, hi = min(lo, int(f1.min_rl)), max(hi, int(f1.max_rl))
    if not (lo <= hi < MAX_READ_LENGTH):
        return None
    return (lo, ctx.hist_range(0, lo, hi).tolist())


def _plus_line_class(head, ends):
    """line class of the range's first line, from the first complete line (line i = head[ends[i-1]:ends[i]-1]) that is exactly "+";
    None without one"""
    for i in range(1, len(ends)):
        if ends[i] - ends[i - 1] == 2 and head[ends[i - 1]] == 0x2B:
            return (2 - i) % 4
    return None


def _dbg(msg):
    if os.environ.get("FQG_DEBUG_ROUTE"):
        import sys
        print(f"[route] {time.perf_counter() % 1000:9.4f} " + msg, file=sys.stderr, flush=True)


def _as_tensor(ptr, n, device):
    """uint8 tensor view of raw device (or, in the CPU tests, host) memory."""
    if device.type == "cuda":
        class _Holder:
            pass
        h = _Holder()
        h.__cuda_array_interface__ = {"shape": (n,), "typestr": "|u1", "data": (ptr, False), "version": 2}
        return torch.as_tensor(h, device=device)
    buf = (ctypes.c_uint8 * n).from_address(ptr)
    return torch.frombuffer(buf, dtype=torch.uint8)
