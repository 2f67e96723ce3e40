"""The conv epilogue has one reduction: the 31-shuffle transpose-reduce of epilogue.cuh (DESIGN §3.1).  The shared-memory
transpose it replaced is gone, and so is the build switch that selected it."""
import os
import re

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CSRC = os.path.join(ROOT, "unet.cu_b200", "csrc")


def test_no_transpose_reduce_switch():
    found = []
    for f in sorted(os.listdir(CSRC)):
        with open(os.path.join(CSRC, f), encoding="utf-8") as fh:
            if re.search(r"\bUB_EPI_SHUFFLE_REDUCE\b", fh.read()):
                found.append(f)
    assert not found, f"UB_EPI_SHUFFLE_REDUCE is still defined or tested in {found}"
