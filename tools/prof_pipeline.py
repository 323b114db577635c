"""World-1 run of the pipelined sharded orchestration on synthetic reads: step time and kernel times per class.
    python tools/prof_pipeline.py [records]"""
import os, sys, time
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
import fastq_utils_b200 as fq
from fastq_utils_b200 import dist as fqdist

import torch.distributed as dist
if int(os.environ.get("WORLD_SIZE", "1")) > 1:  # experiment: NCCL initialised (two ranks, one all-reduce), every rank then works alone
    torch.cuda.set_device(int(os.environ["LOCAL_RANK"]))
    dist.init_process_group("nccl", device_id=torch.device("cuda", int(os.environ["LOCAL_RANK"])))
    x = torch.ones(1 << 20, device="cuda"); dist.all_reduce(x); torch.cuda.synchronize()
n = int(sys.argv[1]) if len(sys.argv) > 1 else 40_000_000
rb = fq.illumina_record_bytes()
t = torch.zeros(n * rb + 64, dtype=torch.uint8, device="cuda")
st = torch.cuda.current_stream().cuda_stream
for s in range(0, n, 8_000_000):
    k = min(8_000_000, n - s)
    fq.synth_illumina(t[s * rb:], s, k, seed=42, mate=1, perm_window=0, stream=st)
torch.cuda.synchronize()
if os.environ.get("PEER") and torch.cuda.device_count() > 1:  # does an enabled peer mapping change the index kernels?
    a = torch.zeros(1 << 20, device="cuda:1"); b = a.to("cuda:0"); torch.cuda.synchronize(); print("peer access enabled", torch.cuda.can_device_access_peer(0, 1))
dev = torch.cuda.current_device()
run = fqdist.ShardedFastqInfo(fq.MODE_INDEX, device=dev, n_hint=n)
run.world, run.rank = 1, 0
ts = []
for i in range(5):
    if i == 2:
        run.ctx.kernel_stats(reset=True); run.shard.kernel_stats(reset=True)
    torch.cuda.synchronize(); t0 = time.perf_counter()
    res = run.run_device(t.data_ptr(), n * rb, name="a.fq")
    torch.cuda.synchronize(); ts.append((time.perf_counter() - t0) * 1e3)
if dist.is_initialized() and dist.get_rank() != 0:
    sys.exit(0)
print("rounds", run.rounds_done, "step ms", [round(x, 2) for x in ts], "GB/s", round(n * rb / min(ts[2:]) / 1e6, 1), "rc", res["transcript"][0], res["n_index_entries"])
for nm, c in (("ctx", run.ctx), ("shard", run.shard)):
    ks = c.kernel_stats()
    print(nm, {k: (round(v["ms"] / 3, 3), v["launches"] // 3) for k, v in ks.items() if v["launches"]})
print("paths", run.ctx.path_counts())
