"""Every bf16 stack case of tests/test_gpu_attention_relevance.py on the GPU: the worst-row and median-row ratio of the kernel's gradient-map
error to the bf16 emulation's, written as JSON together with the card's name, power limit and max SM clock read in the same run.  K_GMAP
in that test is 1.5 x the largest worst-row ratio this reports, rounded up to two decimals.

    python tools/gradmap_budget_ratios.py --out profiles/r13_gradmap_budget_ratios.json"""
import argparse
import json
import math
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

import test_gpu_attention_relevance as T  # noqa: E402
from head_budget_ratios import card  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    args = ap.parse_args()
    rows = []
    for name in T.GEOMS:
        for masked in (False, True):
            gm, g64, emu, _ = T.stack_case(name, masked, "bf16")
            worst, median = T.gmap_ratios(gm, g64, emu)
            rows.append({"case": name, "masked": masked, "worst_row_ratio": round(worst, 4), "median_row_ratio": round(median, 4)})
            print(rows[-1], flush=True)
    top = max(r["worst_row_ratio"] for r in rows)
    res = {**card(), "cases": rows, "max_worst_row_ratio": top, "k_gmap": math.ceil(1.5 * top * 100) / 100}
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps({k: v for k, v in res.items() if k != "cases"}))


if __name__ == "__main__":
    main()
