"""Per-stage GPU time of the chain behind the TFormer at bench.py's batch (512 clips x 16 frames, one GPU), from CUDA events:

  video_au_former   AU_former.tokens_into on the TFormer's cls rows (BN, front GEMM, positional add, 2 encoder layers)
  audio_au_former   the same for the audio features
  fusion_head       former_AU_head.logits21_ (positional add, 3 encoder layers, AU logits and decisions)
  graphed_step      GraphedHotPath.replay(), the step bench.py times

Each stage is captured REPS times into its own CUDA graph and replayed, so the numbers are device time with the launch gaps of a
graph, not Python launch overhead (fusion_head includes a 6 MB device copy that restores its input, which the kernel-per-operation
path updates in place).  Each stage is timed ROUNDS times.
Usage: python tools/chain_breakdown.py [out.json] [rounds]"""
import json
import os
import statistics
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch

import avformer_b200 as A

B, T, SEED, REPS, REPLAYS = 512, 16, 2024, 20, 10
L = A._lib.lib()


def graph_of(fn):
    for _ in range(2):
        fn()
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        for _ in range(REPS):
            fn()
    return g


def time_graph(g, per_replay):
    g.replay()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(REPLAYS):
        g.replay()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / (REPLAYS * per_replay)


def launches(fn):
    n0 = L.avf_launch_count()
    fn()
    torch.cuda.synchronize()
    return int(L.avf_launch_count() - n0)


def main():
    out_path = sys.argv[1] if len(sys.argv) > 1 else "chain_breakdown.json"
    rounds = int(sys.argv[2]) if len(sys.argv) > 2 else 3
    dev = torch.device("cuda")
    torch.manual_seed(SEED)
    model = A.TwoStreamAuralVisualFormer(video_pretrained=False, audio_pretrained=False, task="AU").to(dev).eval().set_precision("bf16")
    g = torch.Generator().manual_seed(SEED)
    stage3 = torch.clamp(torch.randn(B * T, 256, 7, 7, generator=g) * 1.7 + 0.6, min=0).bfloat16().to(dev)
    frame = (torch.randn(B * T, 512, generator=g).abs() * 1.2).bfloat16().to(dev)
    audio = torch.randn(B, 512, generator=g).abs().to(dev)
    vm = model.video_model.video_model
    with torch.no_grad():
        cls = vm.t_former.cls_features(frame)
        tokens = torch.empty((B * 12, 256), dtype=torch.float32, device=dev)
        model.audio_model.au_head.tokens_into(audio, audio.shape[1], B, out=tokens, ld_out=256)
        model.video_model.au_head.tokens_into(cls, cls.shape[1], B, out=tokens[:, 128:], ld_out=256)
    scratch = tokens.clone()

    stages = {
        "video_au_former": lambda: model.video_model.au_head.tokens_into(cls, cls.shape[1], B, out=tokens[:, 128:], ld_out=256),
        "audio_au_former": lambda: model.audio_model.au_head.tokens_into(audio, audio.shape[1], B, out=tokens, ld_out=256),
        "fusion_head": lambda: (scratch.copy_(tokens), model.au_head.logits21_(scratch, B, True)),
    }
    with torch.no_grad():
        graphs = {name: graph_of(fn) for name, fn in stages.items()}
        graphs["graphed_step"] = A.GraphedHotPath(model, stage3, frame, audio)
        counts = {name: launches(fn) for name, fn in stages.items()}
        counts["graphed_step"] = launches(lambda: model.hot_path(stage3, frame, audio, want_decisions=True))     # eager, same kernels
    samples = {name: [] for name in graphs}
    for _ in range(rounds):
        for name, gr in graphs.items():
            if name == "graphed_step":
                samples[name].append(time_graph_replay(gr))
            else:
                samples[name].append(time_graph(gr, REPS))
    gpu = torch.cuda.get_device_name(0)
    try:
        smi = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.sm,clocks.max.sm,clocks_throttle_reasons.active", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=20).stdout.strip()
    except Exception as ex:      # the numbers stand without it; say why it is missing
        smi = f"nvidia-smi unavailable: {ex}"
    res = {"gpu": gpu, "nvidia_smi_after": smi, "clips": B, "frames": T, "rounds": rounds, "graph_reps_per_stage": REPS,
           "ms": {n: {"median": statistics.median(v), "min": min(v), "max": max(v), "samples": v} for n, v in samples.items()},
           "launches": counts}
    with open(out_path, "w") as f:
        json.dump(res, f, indent=1)
    print({n: round(v["median"], 4) for n, v in res["ms"].items()}, counts)


def time_graph_replay(graphed):
    graphed.replay()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    n = 50
    e0.record()
    for _ in range(n):
        graphed.replay()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / n


if __name__ == "__main__":
    main()
