"""Records the lines of the CUDA toolkit's CUPTI sample cuda_memory_trace/memory_trace.cu that
oracle/vadd_oracle.c cites (an NVIDIA derivative of the vectorAdd sample with float operands):
the VectorAdd kernel, the rand() fill loop and the block size, plus whether the file calls
srand() anywhere.  Written to tests/golden/cupti_memory_trace_recipe.json, which
tests/test_oracle.py checks the oracle's recipe against.

    python tests/golden/make_cupti_recipe.py [CUDA toolkit root, default $CUDA_HOME or /usr/local/cuda]
"""
import hashlib
import json
import os
import sys

REL = "extras/CUPTI/samples/cuda_memory_trace/memory_trace.cu"
OUT = os.path.join(os.path.dirname(os.path.abspath(__file__)), "cupti_memory_trace_recipe.json")


def _block(lines: list[str], first: int) -> list[int]:
    """Line indices from `first` through the brace that closes the block opened after it."""
    depth, i = 0, first
    while True:
        depth += lines[i].count("{") - lines[i].count("}")
        if "}" in lines[i] and depth == 0:
            return list(range(first, i + 1))
        i += 1


def extract(cuda_home: str) -> dict:
    raw = open(os.path.join(cuda_home, REL), "rb").read()
    lines = raw.decode().splitlines()
    kernel = next(i for i, l in enumerate(lines) if l.startswith("VectorAdd(")) - 1          # the __global__ line
    first_rand = next(i for i, l in enumerate(lines) if "rand()" in l)
    fill = max(i for i in range(first_rand) if lines[i].strip().startswith("for "))            # the loop around it
    block = next(i for i, l in enumerate(lines) if "dim3 block(" in l)
    keep = _block(lines, kernel) + _block(lines, fill) + [block]
    return {"source": REL, "sha256": hashlib.sha256(raw).hexdigest(),
            "lines": {str(i + 1): lines[i] for i in keep}, "calls_srand": "srand" in raw.decode()}


if __name__ == "__main__":
    home = sys.argv[1] if len(sys.argv) > 1 else os.environ.get("CUDA_HOME", "/usr/local/cuda")
    json.dump(extract(home), open(OUT, "w"), indent=1)
    print(open(OUT).read())
