#!/usr/bin/env python
"""Generate tests/golden/ref_kernels.json: the outputs of the reference's own CUDA kernels (oracle/_ref/libsp1ref.so, built by
`make -C oracle ref` from the reference sources) on the seeded inputs of tests/test_gpu_ref_kernels.py.  Needs that library and a GPU.
Every output is stored as its shape and the SHA-256 of its little-endian words; outputs of at most 64 words also word for word.

  python tools/gen_ref_kernels_golden.py [OUT]      # default OUT: tests/golden/ref_kernels.json
"""
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from tests import ref_lib as R  # noqa: E402
from tests import test_gpu_ref_kernels as T  # noqa: E402


def main():
    path = sys.argv[1] if len(sys.argv) > 1 else T.GOLDEN
    outs = T.reference_outputs(R)
    doc = {"source": "oracle/_ref/libsp1ref.so (the reference's CUDA kernels, sp1 v6.4.0) via tests/ref_lib.py; tools/gen_ref_kernels_golden.py",
           "outputs": {k: T.golden_entry(v) for k, v in outs.items()}}
    with open(path, "w") as f:
        json.dump(doc, f, indent=0, sort_keys=True)
    print(f"{len(outs)} reference outputs -> {path}")


if __name__ == "__main__":
    main()
