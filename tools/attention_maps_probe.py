"""Cost of the attention maps at sizes a user runs, with CUDA events, on one GPU.

Full model (bf16 stacks, fp32 conv trunks), 64 clips x 16 frames: model(x) with the fused kernel on, model(x) with it off, and
attention_maps for all stacks and for stacks=["tformer"]; the TFormer alone at T = 128 over 64 clips: cls_features against
attention_maps.  The four (resp. two) calls alternate inside each round; the medians over rounds are reported, with the map bytes
written and the write rate they imply against the 7.7 TB/s of HBM3e: bytes over the whole map call (a lower bound on the kernels'
rate), and bytes over the extra time against the fused-off forward.  The card's name, power limit and max SM clock are read in the
same run.

    python tools/attention_maps_probe.py --out profiles/r11_attention_maps_probe.json
"""
import argparse
import json
import os
import statistics
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import avformer_b200 as A  # noqa: E402
from oracle import avformer_oracle as O  # noqa: E402

AF = A.functional
HBM_TBPS = 7.7


def _card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True)
    name, power, clock = (s.strip() for s in q.stdout.strip().split("\n")[0].split(","))
    return {"name": name, "power_limit": power, "max_sm_clock": clock}


def _time(fn, reps):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(reps):
        fn()
    b.record()
    b.synchronize()
    return a.elapsed_time(b) / reps


def _rounds(calls, rounds, reps):
    for f in calls.values():                                   # warm-up of every shape the timed window uses
        f()
    torch.cuda.synchronize()
    times = {k: [] for k in calls}
    for _ in range(rounds):
        for k, f in calls.items():
            times[k].append(_time(f, reps))
    return {k: statistics.median(v) for k, v in times.items()}


def _fused(flag, fn):
    def run():
        prev = AF.set_fused_enabled(flag)
        try:
            return fn()
        finally:
            AF.set_fused_enabled(prev)
    return run


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--rounds", type=int, default=7)
    ap.add_argument("--reps", type=int, default=5)
    args = ap.parse_args()
    torch.backends.cudnn.benchmark = False
    res = {"card": _card(), "rounds": args.rounds, "reps_per_round": args.reps}

    T, n_clips = 16, 64
    m = A.TwoStreamAuralVisualFormer(video_pretrained=False, audio_pretrained=False, task="AU")
    m.load_state_dict(O.make_state_dict(1, T), strict=True)
    m = m.cuda().eval().set_precision("bf16")
    clip, audio, _ = O.synth_inputs(1, n_clips, T)
    x = {"clip": clip.cuda(), "audio_features": audio.cuda()}
    with torch.no_grad():
        _, maps_all = m.attention_maps(x)
        _, maps_tf = m.attention_maps(x, ["tformer"])
        bytes_all = sum(v.numel() * 4 for v in maps_all.values())
        bytes_tf = sum(v.numel() * 4 for v in maps_tf.values())
        t = _rounds({"model_fused_on": _fused(True, lambda: m(x)), "model_fused_off": _fused(False, lambda: m(x)),
                     "maps_all": lambda: m.attention_maps(x), "maps_tformer": lambda: m.attention_maps(x, ["tformer"])}, args.rounds, args.reps)
    model = {"clips": n_clips, "T": T, "ms": t, "map_bytes": {"all": bytes_all, "tformer": bytes_tf},
             "map_bytes_by_stack": {k: v.numel() * 4 for k, v in maps_all.items()}}
    for key, nbytes in (("all", bytes_all), ("tformer", bytes_tf)):
        tm, extra = t["maps_" + key], t["maps_" + key] - t["model_fused_off"]
        model[f"write_TBps_{key}_over_call"] = nbytes / tm / 1e9
        model[f"write_TBps_{key}_over_extra"] = nbytes / extra / 1e9 if extra > 0 else None
    res["model_64x16"] = model

    T = 128
    tf = A.TFormer(num_patches=T).cuda().eval()
    spec = [("cls_token", (1, 1, 512), "normal"), ("pos_embedding", (1, T + 1, 512), "normal")] + list(
        O._encoder_spec("spatial_transformer.", 512, 3, 512, 1024))
    tf.load_state_dict(O.params_from_spec(spec, 2), strict=True)
    tf.spatial_transformer.precision = "bf16"
    frames = torch.randn(n_clips * T, 512, device="cuda")
    with torch.no_grad():
        nbytes = tf.attention_maps(frames)[1].numel() * 4
        t = _rounds({"cls_features": lambda: tf.cls_features(frames), "attention_maps": lambda: tf.attention_maps(frames)}, args.rounds,
                    args.reps * 4)
    extra = t["attention_maps"] - t["cls_features"]
    res["tformer_64x128"] = {"clips": n_clips, "T": T, "ms": t, "map_bytes": nbytes, "write_TBps_over_call": nbytes / t["attention_maps"] / 1e9,
                             "write_TBps_over_extra": nbytes / extra / 1e9 if extra > 0 else None}
    res["hbm_TBps_datasheet"] = HBM_TBPS
    line = json.dumps(res)
    print(line)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        f.write(line + "\n")


if __name__ == "__main__":
    main()
