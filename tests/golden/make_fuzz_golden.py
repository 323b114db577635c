"""What the UNMODIFIED reference binaries return on the seeded fuzz inputs of the tests → tests/golden/fuzz/<name>.json.

The fuzz tests compare with the live binaries when oracle/_ref is built (`make -C oracle ref ref-tools` with the reference's sources)
and with these files otherwise.  Each test module's `reference_result` runs the binary; this script only calls it for every seed
the tests use.  Run it where oracle/_ref is built:

    python tests/golden/make_fuzz_golden.py
"""
import json
import os
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))

import test_filterpair  # noqa: E402
import test_oracle_fuzz  # noqa: E402
import test_reader_tools  # noqa: E402
import test_stream_entry  # noqa: E402
import test_trim_poly_at  # noqa: E402
import test_writer_tools  # noqa: E402
from _util import have_ref  # noqa: E402

SETS = {
    "oracle_fuzz": ("fastq_info", test_oracle_fuzz.reference_result, [str(s) for s in test_oracle_fuzz.SEEDS]),
    "stream_operands": ("fastq_info", lambda k: test_stream_entry.reference_result(k.split(" ")), [" ".join(a) for a in test_stream_entry.OPERAND_ARGVS]),
    "reader_fuzz": ("fastq_num_reads", test_reader_tools.reference_result, [str(s) for s in test_reader_tools.SEEDS]),
    "writer_fuzz": ("fastq_truncate", test_writer_tools.reference_result, [str(s) for s in test_writer_tools.SEEDS]),
    "trim_fuzz": ("fastq_trim_poly_at", test_trim_poly_at.reference_result, [str(s) for s in (*test_trim_poly_at.SEEDS_SIM, *test_trim_poly_at.SEEDS_GPU)]),
    "filterpair_fuzz": ("fastq_filterpair", test_filterpair.reference_result, [str(s) for s in (*test_filterpair.SEEDS_SIM, *test_filterpair.SEEDS_GPU)]),
}


def main():
    out_dir = os.path.join(HERE, "fuzz")
    os.makedirs(out_dir, exist_ok=True)
    for name, (tool, run, keys) in SETS.items():
        if not have_ref(tool):
            sys.exit(f"oracle/_ref/{tool} missing: build it with `make -C oracle ref ref-tools REF=<reference checkout>` first")
        res = {k: run(int(k) if k.lstrip("-").isdigit() else k) for k in keys}
        with open(os.path.join(out_dir, name + ".json"), "w") as fh:
            json.dump(res, fh, indent=0, sort_keys=True)
        print(name, len(res), "cases")


if __name__ == "__main__":
    main()
