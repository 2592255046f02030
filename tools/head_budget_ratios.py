"""Every bf16 case of tests/test_gpu_head_train.py on the GPU: the worst-unit and median-unit ratio of the kernel's error to the bf16
emulation's, per tensor, written as JSON together with the card's name, power limit and max SM clock read in the same run.  K_HEAD in
tests/head_oracle.py is 1.5 x the largest worst-unit ratio this reports, rounded up to two decimals.

    python tools/head_budget_ratios.py --out profiles/r12_head_budget_ratios.json"""
import argparse
import json
import math
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

import head_oracle as H  # noqa: E402
import test_gpu_head_train as T  # noqa: E402


def card():
    q = subprocess.run(["nvidia-smi", "--id=0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader,nounits"],
                       capture_output=True, text=True, check=True).stdout.strip().split(", ")
    return {"gpu": q[0], "power_limit_w": float(q[1]), "max_sm_clock_mhz": int(q[2])}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    args = ap.parse_args()
    cases = [(f"front-train-{'batch' if bs else 'running'}-n{n}", lambda n=n, bs=bs: T.run_front_case(n, "bf16", bs))
             for bs in (True, False) for n in H.CLIPS]
    cases += [(f"front-eval-ntok{nt}-n{n}", lambda n=n, nt=nt: T.run_eval_front_case(n, "bf16", nt)) for nt in (12, 2) for n in H.CLIPS]
    results = []
    for name, run in cases:
        try:
            r = run()
        except AssertionError as e:          # a bound or sentinel check of the case failed: recorded, the ratios of the others still count
            results.append({"case": name, "error": str(e)})
            print(f"{name}: {e}", flush=True)
            continue
        for k, (worst, median) in r.items():
            results.append({"case": name, "tensor": k, "worst": round(worst, 4), "median": None if median is None else round(median, 4)})
        top = max(r.items(), key=lambda kv: kv[1][0])
        print(f"{name}: worst {top[1][0]:.3f} ({top[0]})", flush=True)
    ok = [e for e in results if "error" not in e]
    worst = max(ok, key=lambda e: e["worst"])
    meds = [e["median"] for e in ok if e["median"] is not None]
    out = dict(card(), sm_count=T.sms(), what="per bf16 case and tensor of tests/test_gpu_head_train.py: worst-unit and median-unit ratio of "
                                              "the kernel's per-unit RMS error (against fp64) to the bf16 emulation's (median: row units only)",
               largest_worst=worst, median_range=[min(meds), max(meds)], K_HEAD=math.ceil(150 * worst["worst"]) / 100, results=results)
    with open(args.out, "w") as f:
        json.dump(out, f, indent=0)
    print(f"largest worst-unit ratio {worst['worst']} ({worst['case']} {worst['tensor']}), medians {min(meds)}-{max(meds)}, "
          f"K_HEAD = 1.5 x = {1.5 * worst['worst']:.3f}; {out['gpu']} at {out['power_limit_w']} W, {out['max_sm_clock_mhz']} MHz")


if __name__ == "__main__":
    main()
