"""Extract the golden vectors the reference's own tests hold for the dense-LA path into reference_golden.json.

Given a checkout of tracel-ai/cubecl at 4057f39e (the tests only read the JSON this writes):
    python tests/golden/make_golden.py <path to the cubecl checkout>
The reference cannot be executed here (Rust, no toolchain), so the goldens are the LITERAL expected arrays and input
generators written in its test sources; this script parses them so nothing is transcribed by hand.
"""
from __future__ import annotations

import json
import re
import sys
from pathlib import Path

OUT = Path(__file__).resolve().parent / "reference_golden.json"
NUM = r"-?\d+(?:\.\d*)?"


def literal_after(text: str, anchor: str, opener: str) -> tuple[list[float], int]:
    """Numbers of the first `opener ... ]` literal after `anchor`; also the 1-based line of the literal."""
    a = text.index(anchor)
    s = text.index(opener, a) + len(opener)
    e = text.index("]", s)
    nums = [float(x) for x in re.findall(NUM, text[s:e])]
    return nums, text.count("\n", 0, s) + 1


def main(ref: Path) -> None:
    cmma = (ref / "crates/cubecl-core/src/runtime_tests/cmma.rs").read_text()
    sums = (ref / "examples/sum_things/src/lib.rs").read_text()
    gold = {"_generated_by": "tests/golden/make_golden.py", "_reference": "tracel-ai/cubecl @ 4057f39e"}

    v, line = literal_after(cmma, "pub fn test_simple_1_expected", "vec![")
    assert len(v) == 256
    gold["cmma_simple_1"] = {
        "source": f"crates/cubecl-core/src/runtime_tests/cmma.rs:{line}",
        "desc": "f16 16x16x16, lhs[i]=i row-major, rhs[i]=i%8 col-major (stored [N,K]), f32 acc, Out = Lhs @ Rhs.T",
        "m": 16, "n": 16, "k": 16, "expected": v,
    }
    v, line = literal_after(cmma, "pub fn test_simple_tf32", "let expected = [")
    assert len(v) == 256
    gold["cmma_tf32"] = {
        "source": f"crates/cubecl-core/src/runtime_tests/cmma.rs:{line}",
        "desc": "tf32 16x16x8, lhs[i]=i row-major [16,8], rhs[i]=i%8 ROW-major [8,16] (stride 16), f32 acc",
        "m": 16, "n": 16, "k": 8, "expected": v,
    }
    v, line = literal_after(cmma, "pub fn test_cmma_strided", "let expected = [")
    assert len(v) == 256
    gold["cmma_strided"] = {
        "source": f"crates/cubecl-core/src/runtime_tests/cmma.rs:{line}",
        "desc": "m16 n16 k32 buffers, only the left 16x16 k-tile is multiplied: lhs row stride 32 (left tile = i, right 0), "
                "rhs[i]=i%8 col-major with stride 16",
        "m": 16, "n": 16, "k": 16, "lhs_row_stride": 32, "expected": v,
    }
    v, line = literal_after(sums, "pub fn launch", "&[")
    gold["sum_things"] = {
        "source": f"examples/sum_things/src/lib.rs:{line}",
        "desc": "input of the sum_things demo; every unit's sum is 15, series (SumThenMul) = sum * input[unit]",
        "input": v, "expected_sum": 15.0, "expected_series": [-15.0, 150.0, 15.0, 75.0],
    }
    # generator-defined goldens (the reference computes the expectation in the test): recorded as formulas
    gold["cmma_manual"] = {
        "source": "crates/cubecl-core/src/runtime_tests/cmma.rs:1099-1196",
        "desc": "lhs[i,j]=2i+j [m,k] row-major, rhs[i,j]=3i+j [k,n] row-major, expected integer dot products, 3% rel tol",
        "shapes": [[16, 8, 16], [16, 8, 8]],
    }
    gold["simple_cube"] = {
        "source": "crates/cubecl-core/src/runtime_tests/cmma.rs:695-721",
        "desc": "lhs[i]=i [m,k] row-major f16, rhs[i]=i%8 stored [n,k], f32 sum += l*r ascending k",
    }
    gold["plane_sum"] = {
        "source": "crates/cubecl-core/src/runtime_tests/plane.rs:154-189",
        "desc": "32 lanes x vec, value = flat index; expected[v] = sum_k input[v + k*vec] (vec1: 496)",
        "vec_sizes": [1, 2, 4],
    }
    gold["all_reduce"] = {
        "source": "crates/cubecl-core/src/runtime_tests/all_reduce.rs:5-62",
        "desc": "8 handles x 100 f32 per device, value = dev + j; expected sum(dev ids) + j * ndev on every device, exact",
        "size": 100, "num_handles": 8,
    }
    OUT.write_text(json.dumps(gold, indent=1) + "\n")
    print("wrote", OUT, {k: len(v.get("expected", [])) for k, v in gold.items() if isinstance(v, dict)})


if __name__ == "__main__":
    if len(sys.argv) != 2:
        raise SystemExit("usage: python tests/golden/make_golden.py <path to the cubecl checkout>")
    main(Path(sys.argv[1]))
