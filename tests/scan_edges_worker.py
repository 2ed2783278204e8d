"""Worker of tests/test_gpu_scan_edges.py::test_fallback_kernels.  The scan's A/B switches (R2D2_SCAN_L2XCHG=0: the
H = 512 forward on the 16/32-row tcgen05 kernels and the BPTT without the L2 exchange; R2D2_SCAN_PINGPONG=0: the
plain 32-row forward kernel for H <= 256) are read once per process, so the caller starts this script with the switch
in its environment.  It runs the tiling-sweep rows those kernels take on the tcgen05 implementation and prints one
JSON line: the tiling and error records of every case and the scan status flag."""
import json
import os
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
for p in (HERE, ROOT, os.path.join(ROOT, "pytorch-r2d2-dpg_b200")):
    if p not in sys.path:
        sys.path.insert(0, p)

import torch  # noqa: E402

import test_gpu_scan_edges as edges  # noqa: E402
from r2d2_b200 import native  # noqa: E402


def main():
    native.lib()
    cases = []
    for H, label in edges.fallback_cases():
        B = edges.resolve(label, edges.fits(native, H))
        descs, recs = edges.run_scan_case(native, H, B, 1, seed=H * 7919 + B)
        cases.append({"H": H, "B": B, "label": label, "tiling": descs, "records": recs})
    torch.cuda.synchronize()
    print(json.dumps({"cases": cases, "status": edges.scan_status(native)}))


if __name__ == "__main__":
    main()
