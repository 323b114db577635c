"""Run by tests/test_dist_gloo.py::test_world_of_one: fastq_utils_b200.dist without a process group (a world of one) on the
stand-in device — every routing variant and fallback of the orchestration, checked against the CPU oracle."""
import ctypes
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

import torch  # noqa: E402

import fastq_utils_b200 as fq  # noqa: E402
from sim_lib import use_sim_library  # noqa: E402
from fastq_utils_b200 import dist as fqdist  # noqa: E402
from _util import oracle_run  # noqa: E402

use_sim_library()

big = [f"@M0:1:FC:1:11:{i}:{i * 7} 1:N:0:AC\n{'ACGTN' * (3 + i % 5)}\n+\n{'F' * (5 * (3 + i % 5))}\n" for i in range(4000)]
dup = list(big); dup[3900] = dup[17]
nul = list(big); nul[1500] = "\x00" + nul[1500]
bad = list(big); bad[3000] = bad[3000].replace("ACGTN", "ACXTN", 1)
HOOKS = ("FQG_MAX_CHUNK_BYTES", "FQG_P2P", "FQG_TEST_WEAK_HASH", "FQG_TEST_SLOT_CAP")
n = 0
for nm, rr in (("clean", big), ("dup", dup), ("nul", nul), ("bad", bad)):
    for mode, argv in ((fq.MODE_INDEX, ["a.fq"]), (fq.MODE_SINGLE, ["-r", "a.fq"])):
        for env in ({}, {"FQG_MAX_CHUNK_BYTES": "8192"}, {"FQG_P2P": "1", "FQG_MAX_CHUNK_BYTES": "8192"}, {"FQG_TEST_WEAK_HASH": "1"},
                    {"FQG_P2P": "1", "FQG_TEST_SLOT_CAP": "5", "FQG_MAX_CHUNK_BYTES": "16384"}):
            for k in HOOKS:
                os.environ.pop(k, None)
            os.environ.update(env)
            data = "".join(rr).encode("latin-1")
            mine = bytearray(data) + bytearray(64)
            buf = (ctypes.c_uint8 * len(mine)).from_buffer(mine)
            run = fqdist.ShardedFastqInfo(mode, device=0, tensor_device=torch.device("cpu"))
            res = run.run_device(ctypes.addressof(buf), len(data), name="a.fq")
            want = oracle_run(argv, data, None)
            assert tuple(res["transcript"]) == want, (nm, mode, env, res["transcript"], want)
            n += 1
print("ok", n)
