"""bench.py's command line: the reference arm runs without a GPU (and without loading libfastq_gpu.so) and its JSON line carries the
keys a reader of the result needs; --steps and --dump-outputs of our arm."""
import json
import os
import subprocess
import sys

import pytest

from _util import ROOT


@pytest.mark.parametrize("workload", ["illumina_pe", "illumina_se"])
def test_reference_arm_line(workload):
    # without the reference binary (oracle/_ref, built only where the reference's sources are) the arm times the oracle's restatement
    kind = "reference" if os.path.exists(os.path.join(ROOT, "oracle", "_ref", "fastq_info")) else "port"
    env = dict(os.environ, CUDA_VISIBLE_DEVICES="")
    p = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "0", "--cpu-sample-reads", "20480",
                        "--workload", workload], capture_output=True, text=True, env=env, timeout=300)
    assert p.returncode == 0, p.stderr[-2000:]
    line = [l for l in p.stdout.splitlines() if l.startswith("{")][-1]
    d = json.loads(line)
    assert d["impl"] == "reference" and d["metric"] == "fastq_info_validated_GBps" and d["unit"] == "GB/s" and d["higher_is_better"] is True
    assert d["value"] > 0 and d["steps"] == 1 and d["n_gpus"] == 1 and d["scaling"] == "weak" and d["dtype"] == "u8" and d["data"] == "synthetic"
    assert d["cpu_baseline"]["kind"] == kind and d["cpu_baseline"]["cores"] == 1 and d["cpu_baseline"]["value"] == d["value"]
    assert d["e2e"] == {"value": d["value"], "unit": "GB/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert "workload" in d["config"]


@pytest.mark.gpu
def test_steps_and_dump_outputs(tmp_path):
    """--steps sets how many jobs run in the timed region (its launch count scales with it); --dump-outputs writes the last step's
    report and transcript, which do not depend on the run or on the number of steps."""
    import numpy as np
    from fastq_utils_b200 import synth
    n = 4096
    lines, dumps = [], []
    for steps in (1, 3):
        d = tmp_path / f"steps{steps}"
        p = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", str(steps), "--warmup", "1", "--reads", str(n), "--no-extras", "--no-e2e",
                            "--cpu-sample-reads", "1024", "--dump-outputs", str(d)], capture_output=True, text=True, timeout=600)
        assert p.returncode == 0, p.stderr[-2000:]
        line = json.loads([l for l in p.stdout.splitlines() if l.startswith("{")][-1])
        assert line["steps"] == steps and line["parity"]["all_ok"], line["parity"]
        lines.append(line)
        dumps.append({f: np.load(d / f) for f in sorted(os.listdir(d))})
    assert lines[0]["gpu_launches"] > 0 and lines[1]["gpu_launches"] == 3 * lines[0]["gpu_launches"], [l["gpu_launches"] for l in lines]
    assert lines[1]["roofline"]["launches"] == 3 * lines[0]["roofline"]["launches"]
    got = dumps[0]
    assert sorted(got) == ["exit_status.npy", "report_error.npy", "report_files.npy", "report_index.npy", "stderr.npy", "stdout.npy"]
    assert all(v.dtype in (np.float32, np.float64) for v in got.values()) and sum(v.nbytes for v in got.values()) <= 64 << 20
    text = lambda k: bytes(got[k].astype(np.uint8)).decode("latin-1")  # noqa: E731
    assert (int(got["exit_status.npy"][0]), text("stdout.npy"), text("stderr.npy")) == synth.expect_index(n, "synthetic_1.fastq", n2=n, name2="synthetic_2.fastq")
    files = got["report_files.npy"]  # (file, field, (high 32 bits, low 32 bits))
    assert files.shape == (2, 8, 2) and files[:, 0].tolist() == [[0, n], [0, n]]
    assert got["report_error.npy"][0].tolist() == [0, 0] and got["report_error.npy"][8].tolist() == [2**32 - 1, 2**32 - 1]  # no error: event_key ~0
    assert dumps[0].keys() == dumps[1].keys() and all(np.array_equal(dumps[0][k], dumps[1][k]) for k in got)


def test_reference_arm_does_not_load_the_product_library():
    src = open(os.path.join(ROOT, "bench.py")).read()
    arm = src[src.index('if a.impl == "reference":'):src.index("# ------------------------------------------------------------------ our arm")]
    assert "fastq_utils_b200 as fq" not in arm and ".lib()" not in arm and "import torch" in arm  # (torch only for the long-read layout)
