"""GPU time of the TFormer with and without an attention mask at bench.py's batch (512 clips x T=16 frames, one GPU), from CUDA events:

  unmasked               TFormer.cls_features(x): the library's inference TFormer, one call
  masked_all_kept        cls_features(x, mask) with every frame kept (the masked kernels, same result bits)
  masked_random_lengths  cls_features(x, mask) with clip lengths drawn uniformly from 1..16

The three cases run alternately, ROUNDS times ITERS calls each, so that clock and neighbour drift hit them alike; each figure is the
median over the rounds of (event time / ITERS).  The mask pad (a torch op) is part of the masked calls.
Usage: python tools/mask_probe.py [out.json] [precision]"""
import json
import os
import statistics
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch

import avformer_b200 as A

B, T, DIM, ITERS, ROUNDS, SEED = 512, 16, 512, 100, 15, 2024


def gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True,
                             text=True, timeout=30).stdout.strip().splitlines()
        return out[0] if out else "unknown"
    except (OSError, subprocess.SubprocessError):
        return "unknown"


def main():
    out_path = sys.argv[1] if len(sys.argv) > 1 else ""
    precision = sys.argv[2] if len(sys.argv) > 2 else "bf16"
    torch.manual_seed(SEED)
    tf = A.TFormer(num_patches=T, dim=DIM).cuda().eval()
    tf.spatial_transformer.precision = precision
    x = torch.randn(B * T, DIM, device="cuda")
    lengths = torch.randint(1, T + 1, (B,), device="cuda")
    cases = {"unmasked": None,
             "masked_all_kept": torch.ones(B, T, dtype=torch.bool, device="cuda"),
             "masked_random_lengths": torch.arange(T, device="cuda")[None, :] < lengths[:, None]}
    L = A._lib.lib()
    launches = {}
    with torch.no_grad():
        for name, m in cases.items():
            for _ in range(10):
                tf.cls_features(x, m)
            n0 = L.avf_launch_count()
            tf.cls_features(x, m)
            launches[name] = L.avf_launch_count() - n0
        torch.cuda.synchronize()
        times = {name: [] for name in cases}
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        for _ in range(ROUNDS):
            for name, m in cases.items():
                ev0.record()
                for _ in range(ITERS):
                    tf.cls_features(x, m)
                ev1.record()
                ev1.synchronize()
                times[name].append(ev0.elapsed_time(ev1) / ITERS)
    med = {name: statistics.median(v) for name, v in times.items()}
    res = {"probe": "mask_probe", "gpu": gpu_info(), "precision": precision, "clips": B, "frames": T,
           "ms_per_call_median": {k: round(v, 5) for k, v in med.items()},
           "ms_per_call_min_max": {k: [round(min(v), 5), round(max(v), 5)] for k, v in times.items()},
           "ratio_to_unmasked": {k: round(v / med["unmasked"], 4) for k, v in med.items()},
           "library_launches_per_call": launches, "mean_clip_length": float(lengths.float().mean())}
    line = json.dumps(res)
    print(line)
    if out_path:
        with open(out_path, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
