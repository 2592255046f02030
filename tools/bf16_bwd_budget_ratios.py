"""Every case of tests/test_gpu_bf16_bwd_budget.py on the GPU: the worst-unit and median-unit ratio of the kernel's error to the bf16
emulation's, per tensor, written as JSON together with the card's name, power limit and max SM clock read in the same run.  K_BWD in
tests/bf16_bwd_oracle.py is 1.5 x the largest worst-unit ratio this reports.

    python tools/bf16_bwd_budget_ratios.py --out profiles/r08_bf16_bwd_budget_ratios.json"""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

import bf16_bwd_oracle as BB  # noqa: E402
import test_gpu_bf16_bwd_budget as T  # noqa: E402


def card():
    q = subprocess.run(["nvidia-smi", "--id=0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader,nounits"],
                       capture_output=True, text=True, check=True).stdout.strip().split(", ")
    return {"gpu": q[0], "power_limit_w": float(q[1]), "max_sm_clock_mhz": int(q[2])}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    args = ap.parse_args()
    results = []
    for case in BB.ATT_CASES + BB.STACK_CASES:
        try:
            r = T.run_att_case(case) if case["kind"] == "att" else T.run_stack_case(case)
        except AssertionError as e:          # a structural check of the case failed: recorded, the budgets of the others still count
            results.append({"case": case["name"], "error": str(e)})
            print(f"{case['name']}: {e}", flush=True)
            continue
        for k, (worst, median) in r.items():
            results.append({"case": case["name"], "tensor": k, "worst": round(worst, 4), "median": None if median is None else round(median, 4)})
        top = max(r.items(), key=lambda kv: kv[1][0])
        print(f"{case['name']}: worst {top[1][0]:.3f} ({top[0]})", flush=True)
    ok = [e for e in results if "error" not in e]
    worst = max(ok, key=lambda e: e["worst"])
    meds = [e["median"] for e in ok if e["median"] is not None]
    out = dict(card(), what="per case and tensor of tests/test_gpu_bf16_bwd_budget.py: worst-unit and median-unit ratio of the kernel's "
                            "per-unit RMS error (against fp64) to the bf16 emulation's (median: rows and slices only)",
               largest_worst=worst, median_range=[min(meds), max(meds)], K_BWD=round(1.5 * worst["worst"], 2), results=results)
    with open(args.out, "w") as f:
        json.dump(out, f, indent=0)
    print(f"largest worst-unit ratio {worst['worst']} ({worst['case']} {worst['tensor']}), medians {min(meds)}-{max(meds)}, "
          f"K_BWD = 1.5 x = {1.5 * worst['worst']:.3f}; {out['gpu']} at {out['power_limit_w']} W, {out['max_sm_clock_mhz']} MHz")


if __name__ == "__main__":
    main()
