"""Long clips on one GPU: the attention kernels alone at 64..256 tokens, the TFormer at T = 16..255, and a full-model bank training
step at T = 64 and 128.  Times are medians of CUDA-event rounds after warm-up of every shape.

  attention   bf16, 8 heads x 64, n_tok in {64 (the <= 64-token kernel), 65, 129, 256}, 8192 // n_tok sequences per call (about 8192
              token rows).  Achieved TFLOP/s from the shape: 4 N^2 inner per sequence forward, 10 N^2 inner backward (five contractions;
              the kernels' recomputation is not counted).  torch.nn.functional.scaled_dot_product_attention on the same unmasked bf16
              q / k / v ([n_seq, 8, N, 64]) is the yardstick, its backward timed alone through torch.autograd.grad.  The qkv working set
              (25 MB) fits the 126 MB L2: repeated calls read it from there.
  tformer     TFormer(num_patches=T) in bf16 on FRAME_ROWS frame rows (FRAME_ROWS // T clips): cls_features unmasked and with a
              random frames-kept mask (the library call), and a training step (forward + backward through autograd, dropout 0).  The
              attention kernels' share is their summed device time over all kernels' device time, from torch.profiler in a separate
              pass after the timings.
  model       TwoStreamAuralVisualFormer.forward_indexed training step (train(), FusedAdam, bf16 transformers, fp32 conv trunks) on a
              window of W clips with consecutive frames (offsets arange(T) - (T - 1), clamped), as tools/bank_train_probe.py does at
              T = 16.

The card's name, power limit and max SM clock are read in the same process.
Usage: python tools/long_clip_probe.py [out.json]"""
import json
import os
import statistics
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
import torch.nn.functional as F

import avformer_b200 as A

AF = A.functional
HEADS, DH = 8, 64
ATT_NTOK, ATT_ROWS, ATT_ITERS = (64, 65, 129, 256), 8192, 50
TF_T, FRAME_ROWS, TF_ITERS = (16, 63, 64, 128, 255), 16384, 10
MODEL_T, MODEL_W = (64, 128), 64
WARMUP, ROUNDS = 3, 7
SEED = 2026


def gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True,
                             text=True, timeout=30).stdout.strip().splitlines()
        return out[0] if out else "unknown"
    except (OSError, subprocess.SubprocessError):
        return "unknown"


def elapsed_ms(fn, iters):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    a.record()
    for _ in range(iters):
        fn()
    b.record()
    b.synchronize()
    return a.elapsed_time(b) / iters


def timed(cases, iters):
    """{name: fn} -> {name: (median ms, min ms, max ms)}, the cases alternating round by round."""
    for fn in cases.values():
        for _ in range(WARMUP):
            fn()
    times = {k: [] for k in cases}
    for _ in range(ROUNDS):
        for k, fn in cases.items():
            times[k].append(elapsed_ms(fn, iters))
    return {k: (statistics.median(v), min(v), max(v)) for k, v in times.items()}


def attention_share(fn, iters=3):
    """Summed device time of the attention kernels over that of every kernel while fn runs (torch.profiler)."""
    from torch.profiler import ProfilerActivity, profile
    fn()
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(iters):
            fn()
        torch.cuda.synchronize()
    tot = att = 0.0
    for e in prof.key_averages():
        t = getattr(e, "device_time_total", None)
        if t is None:
            t = e.cuda_time_total
        if t <= 0 or e.key.startswith(("cudaLaunch", "cudaMemcpy", "Memcpy", "Memset", "cudaStream", "cudaDevice", "cudaEvent")):
            continue
        tot += t
        if "attention" in e.key:
            att += t
    return round(att / tot, 4) if tot > 0 else None


def probe_attention():
    dev = torch.device("cuda")
    g = torch.Generator(device=dev).manual_seed(SEED)
    res = {}
    for n in ATT_NTOK:
        n_seq = ATT_ROWS // n
        inner = HEADS * DH
        qkv = torch.randn(n_seq * n, 3 * inner, device=dev, generator=g).bfloat16()
        dout = torch.randn(n_seq * n, inner, device=dev, generator=g).bfloat16()
        q, k, v = (t.reshape(n_seq, n, HEADS, DH).transpose(1, 2).contiguous().requires_grad_(True) for t in qkv.split(inner, dim=1))
        do4 = dout.reshape(n_seq, n, HEADS, DH).transpose(1, 2).contiguous()
        o4 = F.scaled_dot_product_attention(q, k, v)
        cases = {"avf_fwd": lambda: AF.attention_fwd(qkv, n_seq, n, HEADS, DH),
                 "avf_bwd": lambda: AF.attention_bwd(qkv, dout, n_seq, n, HEADS, DH),
                 "sdpa_fwd": lambda: F.scaled_dot_product_attention(q, k, v),
                 "sdpa_bwd": lambda: torch.autograd.grad(o4, (q, k, v), do4, retain_graph=True)}
        t = timed(cases, ATT_ITERS)
        flops = {"fwd": 4.0 * n * n * inner * n_seq, "bwd": 10.0 * n * n * inner * n_seq}
        ref = F.scaled_dot_product_attention(q, k, v).transpose(1, 2).reshape(n_seq * n, inner).float()
        res[f"t{n}"] = {"n_tok": n, "n_seq": n_seq, "token_rows": n_seq * n,
                        "kernel": "attention_mma_kernel / attention_bwd_mma_kernel" if n <= 64 else
                                  "attention_long_mma_kernel / attention_bwd_long_mma_kernel",
                        "ms_median": {k: round(v[0], 5) for k, v in t.items()},
                        "ms_min_max": {k: [round(v[1], 5), round(v[2], 5)] for k, v in t.items()},
                        "tflops": {k: round(flops[k.split("_")[1]] / (v[0] * 1e-3) / 1e12, 2) for k, v in t.items()},
                        "max_abs_diff_fwd_to_sdpa": (AF.attention_fwd(qkv, n_seq, n, HEADS, DH).float() - ref).abs().max().item()}
    return res


def probe_tformer():
    dev = torch.device("cuda")
    res = {}
    for T in TF_T:
        torch.manual_seed(SEED + T)
        n_clips = FRAME_ROWS // T
        tf = A.TFormer(num_patches=T).to(dev)
        tf.spatial_transformer.precision = "bf16"
        frames = torch.randn(n_clips * T, 512, device=dev)
        mask = torch.rand(n_clips, T, device=dev) < 0.8
        dcls = torch.randn(n_clips, 512, device=dev)
        fr = frames.clone().requires_grad_(True)

        def train_step():
            tf.zero_grad(set_to_none=True)
            fr.grad = None
            tf(fr).backward(dcls)

        def infer(m=None):
            with torch.no_grad():
                return tf.cls_features(frames, m)

        tf.eval()
        t_inf = timed({"cls_features": lambda: infer(), "cls_features_masked": lambda: infer(mask)}, TF_ITERS)
        share = {"cls_features": attention_share(lambda: infer()), "cls_features_masked": attention_share(lambda: infer(mask))}
        tf.train()
        t_tr = timed({"train_step": train_step}, TF_ITERS)
        share["train_step"] = attention_share(train_step)
        t = {**t_inf, **t_tr}
        res[f"T{T}"] = {"T": T, "n_tok": T + 1, "clips": n_clips, "frame_rows": n_clips * T,
                        "ms_median": {k: round(v[0], 4) for k, v in t.items()},
                        "ms_min_max": {k: [round(v[1], 4), round(v[2], 4)] for k, v in t.items()},
                        "attention_share_of_kernel_time": share}
        del tf
        torch.cuda.empty_cache()
    return res


def probe_model():
    dev = torch.device("cuda")
    res = {}
    for T in MODEL_T:
        torch.manual_seed(SEED + T)
        model = A.TwoStreamAuralVisualFormer(video_pretrained=False, audio_pretrained=False, task="AU").set_clip_length(T)
        model = model.to(dev).train().set_precision("bf16")
        opt = A.FusedAdam(model.parameters(), lr=1e-5, weight_decay=5e-5)
        n_frames = MODEL_W + T - 1
        frames = torch.randn(n_frames, 3, 112, 112, device=dev)
        idx = ((T - 1 + torch.arange(MODEL_W))[:, None] + torch.arange(T) - (T - 1)).clamp(0, n_frames - 1)
        audio = torch.randn(MODEL_W, 1, 64, 1001, device=dev)
        labels = (torch.rand(MODEL_W, 12, device=dev) > 0.7).float()

        def step():
            opt.zero_grad()
            loss = model.get_au_loss(model.forward_indexed(frames, idx, audio), labels)
            loss.backward()
            opt.step()

        t = timed({"forward_indexed_train_step": step}, 1)["forward_indexed_train_step"]
        res[f"T{T}"] = {"T": T, "clips": MODEL_W, "trunk_frames": n_frames, "ms_per_step_median": round(t[0], 3),
                        "ms_per_step_min_max": [round(t[1], 3), round(t[2], 3)], "ms_per_clip": round(t[0] / MODEL_W, 4)}
        del model, opt
        torch.cuda.empty_cache()
    return res


def main():
    out_path = sys.argv[1] if len(sys.argv) > 1 else ""
    torch.backends.cudnn.benchmark = True
    torch.backends.cuda.matmul.allow_tf32 = False
    res = {"probe": "long_clip_probe", "gpu": gpu_info(), "warmup": WARMUP, "rounds": ROUNDS,
           "attention_bf16_8x64": probe_attention(), "tformer_bf16": probe_tformer(), "model_forward_indexed_train_step": probe_model()}
    line = json.dumps(res)
    print(line)
    if out_path:
        with open(out_path, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
