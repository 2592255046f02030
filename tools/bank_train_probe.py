"""Training over a frame bank: a full-model training step clip by clip against TwoStreamAuralVisualFormer.forward_indexed, and the
scatter-add backward alone, on one GPU, from CUDA events.

A step is forward, AU loss, backward and FusedAdam.step on the whole model in train() (BatchNorm on batch statistics), bf16 transformer
precision, fp32 conv trunks.  It covers a window of W consecutive processed frames of a longer video, with T = 16 and the README's
offsets 3 * (arange(16) - 15), clamped (one clip per processed frame):

  (a) clips      model({"clip": frames[idx] as [W, 3, 16, 112, 112], ...}): 16 W frames through the video trunk
  (b) indexed    model.forward_indexed(frames, idx, audio): the W + 45 frames the window's clips touch, each through the trunk once

(a) and (b) run alternately, ROUNDS times each after WARMUP runs of each; figures are medians.  Reports ms per step and per processed
frame, trunk frames, library launches per step (eager), and the loss of each path on the first step from the same weights.

The scatter alone: avf_tformer_embed_indexed_bwd at 256 clips x 16 slots from a 300-frame bank against torch's backward of bank[idx]
(torch.autograd.grad of the gathered rows), S_ITERS calls per round, S_ROUNDS rounds.

The card's name, power limit and max SM clock are read in the same process.
Usage: python tools/bank_train_probe.py [out.json]"""
import json
import os
import statistics
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch

import avformer_b200 as A

T, WINDOWS, WARMUP, ROUNDS = 16, (64, 256), 2, 5
S_CLIPS, S_BANK, S_ITERS, S_ROUNDS = 256, 300, 100, 11
SEED = 2026
EDGE = 3 * (T - 1)                                               # frames before a clip's processed frame: 45


def gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True,
                             text=True, timeout=30).stdout.strip().splitlines()
        return out[0] if out else "unknown"
    except (OSError, subprocess.SubprocessError):
        return "unknown"


def elapsed_ms(fn):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    a.record()
    res = fn()
    b.record()
    b.synchronize()
    return a.elapsed_time(b), res


def main():
    out_path = sys.argv[1] if len(sys.argv) > 1 else ""
    torch.manual_seed(SEED)
    torch.backends.cudnn.benchmark = True
    dev = torch.device("cuda")
    L = A._lib.lib()
    model = A.TwoStreamAuralVisualFormer(video_pretrained=False, audio_pretrained=False, task="AU").set_clip_length(T)
    model = model.to(dev).train().set_precision("bf16")
    opt = A.FusedAdam(model.parameters(), lr=1e-5, weight_decay=5e-5)
    offsets = 3 * (torch.arange(T) - (T - 1))
    windows = {}
    for W in WINDOWS:
        n_frames = W + EDGE
        frames = torch.randn(n_frames, 3, 112, 112, device=dev)
        idx = (EDGE + torch.arange(W))[:, None] + offsets        # the window's clips, inside the window's frames
        idx = idx.clamp(0, n_frames - 1)
        audio = torch.randn(W, 1, 64, 1001, device=dev)
        labels = (torch.rand(W, 12, device=dev) > 0.7).float()
        clips = frames[idx.to(dev)].permute(0, 2, 1, 3, 4).contiguous()          # built outside the timed window
        windows[W] = (frames, idx, audio, labels, clips)

    def step(W, path):
        frames, idx, audio, labels, clips = windows[W]
        opt.zero_grad()
        out = model({"clip": clips, "audio_features": audio}) if path == "a_clips" else model.forward_indexed(frames, idx, audio)
        loss = model.get_au_loss(out, labels)
        loss.backward()
        opt.step()
        return loss

    res_w = {}
    for W in WINDOWS:
        state = {k: v.clone() for k, v in model.state_dict().items()}
        first = {}
        for path in ("a_clips", "b_indexed"):                  # the first step of each path from the same weights and statistics
            model.load_state_dict(state)
            first[path] = float(step(W, path))
        launches = {}
        for path in ("a_clips", "b_indexed"):
            n0 = L.avf_launch_count()
            step(W, path)
            torch.cuda.synchronize()
            launches[path] = L.avf_launch_count() - n0
        for _ in range(WARMUP):
            step(W, "a_clips"), step(W, "b_indexed")
        times = {"a_clips": [], "b_indexed": []}
        for _ in range(ROUNDS):
            for path in times:
                ms, _ = elapsed_ms(lambda: step(W, path))
                times[path].append(ms)
        model.load_state_dict(state)
        med = {k: statistics.median(v) for k, v in times.items()}
        res_w[f"W{W}"] = {"clips": W, "trunk_frames": {"a_clips": T * W, "b_indexed": W + EDGE},
                          "ms_per_step_median": {k: round(v, 3) for k, v in med.items()},
                          "ms_per_step_min_max": {k: [round(min(v), 3), round(max(v), 3)] for k, v in times.items()},
                          "ms_per_processed_frame": {k: round(v / W, 4) for k, v in med.items()},
                          "speedup_b_over_a": round(med["a_clips"] / med["b_indexed"], 3),
                          "library_launches_per_step": launches, "first_step_loss": first}
        del windows[W]
        torch.cuda.empty_cache()

    # the scatter alone
    g = torch.Generator(device=dev).manual_seed(SEED)
    bank = torch.randn(S_BANK, 512, device=dev, requires_grad=True)
    centre = torch.arange(S_CLIPS) * (S_BANK - 1) // (S_CLIPS - 1)
    sidx = (centre[:, None] + offsets).clamp(0, S_BANK - 1).to(dev)
    sidx32 = sidx.to(torch.int32)
    dtok = torch.randn(S_CLIPS * (T + 1), 512, device=dev, generator=g)
    dslots = dtok.view(S_CLIPS, T + 1, 512)[:, 1:].reshape(-1, 512).contiguous()
    gathered = bank[sidx.reshape(-1)]
    cases = {"avf_tformer_embed_indexed_bwd": lambda: A.functional.tformer_embed_indexed_bwd(dtok, sidx32, S_BANK, T),
             "torch_index_backward": lambda: torch.autograd.grad(gathered, bank, dslots, retain_graph=True)[0]}
    s_out, s_launch = {}, {}
    for name, fn in cases.items():
        for _ in range(5):
            fn()
        n0 = L.avf_launch_count()
        s_out[name] = fn()
        s_launch[name] = L.avf_launch_count() - n0
    s_times = {name: [] for name in cases}
    for _ in range(S_ROUNDS):
        for name, fn in cases.items():
            ms, _ = elapsed_ms(lambda: [fn() for _ in range(S_ITERS)])
            s_times[name].append(ms / S_ITERS)
    s_med = {k: statistics.median(v) for k, v in s_times.items()}
    diff = (s_out["avf_tformer_embed_indexed_bwd"] - s_out["torch_index_backward"]).abs().max().item()

    res = {"probe": "bank_train_probe", "gpu": gpu_info(), "clip_frames": T, "offsets": "3 * (arange(16) - 15), clamped",
           "precision": "bf16 transformers, fp32 conv trunks", "mode": "train() (BatchNorm batch statistics), FusedAdam", "warmup": WARMUP,
           "rounds": ROUNDS, "training_step": res_w,
           "scatter_256x16_from_300": {"ms_per_call_median": {k: round(v, 5) for k, v in s_med.items()},
                                       "ms_per_call_min_max": {k: [round(min(v), 5), round(max(v), 5)] for k, v in s_times.items()},
                                       "library_launches_per_call": s_launch, "max_abs_diff_to_torch": diff,
                                       "max_abs_result": s_out["torch_index_backward"].abs().max().item()}}
    line = json.dumps(res)
    print(line)
    if out_path:
        with open(out_path, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
