"""Records the outputs of the compiled reference that the suite replays (tests/golden/reference_replay/<module>.npz, see
ReferenceReplay in tests/helpers.py): every test that takes the `reference` fixture runs once against the reference's own
code, compiled from a checkout of the original LEANN into oracle/_ref/, and its calls are stored.
    make -C oracle ref REF=<checkout of the original LEANN>
    python tests/golden/make_reference_replay.py
"""
import os
import subprocess
import sys
from pathlib import Path

ROOT = Path(__file__).resolve().parents[2]
MODULES = ["tests/test_oracle_golden.py", "tests/test_oracle_pq_pruning.py", "tests/test_vamana_oracle.py"]


def main():
    os.environ["LEANN_RECORD_REFERENCE"] = "1"
    subprocess.run([sys.executable, "-m", "pytest", "-q", "-p", "no:cacheprovider", *MODULES], cwd=ROOT, check=True)
    # the GPU test's reference leg runs on the CPU: record it directly, with the sizes the test uses
    sys.path[:0] = [str(ROOT), str(ROOT / "tests")]
    import test_gpu_graph_build as t
    from helpers import ReferenceReplay

    rr = ReferenceReplay("test_gpu_graph_build", "test_incremental_builder_against_the_reference_builder")
    print("reference builder: recall@10 %.3f, %.1f links/node" % rr.proxy(t.reference_builder_recall, 100_000, 64, 16, 100))
    rr.finish()


if __name__ == "__main__":
    main()
