"""Whole-video inference: today's clip-by-clip engine against the per-video frame bank, on one GPU, from CUDA events.

A synthetic video of F = 2048 processed frames, T = 16, the README's example offsets 3 * (arange(16) - 15) with clamped edges (one
clip per processed frame, so each frame lies in up to 16 clips), bf16 backbones and bf16 transformer precision:

  (a) clips      eng({"clip": gathered clips, "audio_features": ...}) in batches of 64 clips (one CUDA graph per batch shape); the
                 clips are gathered before the timed window, so (a) is not charged for building them
  (b) bank       eng.frame_features over 256-frame chunks, torch.cat, then eng.clips over 256-clip chunks (eager; the index table
                 is built on the host and copied per chunk)
  (c) tformer    TFormer.cls_features_indexed against bank[idx] + cls_features(mask=idx >= 0), 512 clips x 16 from a 600-frame bank
                 with -1 edges (the TFormer alone), and the library call behind cls_features_indexed without its Python-side range
                 check (which reads a device index on the host: one stream synchronisation per call)

(a) and (b) run alternately, ROUNDS times each after one warm-up run of each; (c) alternates its three calls C_ITERS times per round.
Figures are medians over the rounds.  Reports ms per processed frame, the speed-up, library launches per chunk, the max |logit
difference| between (a) and (b) and their decision agreement where |logit (a)| > 0.25, with the card's name, power limit and max SM
clock read in the same process.
Usage: python tools/video_probe.py [out.json]"""
import json
import os
import statistics
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch

import avformer_b200 as A

F, T, BATCH_A, CHUNK, ROUNDS = 2048, 16, 64, 256, 5
C_CLIPS, C_BANK, C_ITERS, C_ROUNDS = 512, 600, 50, 11
SEED = 2026


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
    model = A.TwoStreamAuralVisualFormer(video_pretrained=False, audio_pretrained=False, task="AU").set_clip_length(T)
    model = model.to(dev).eval().set_precision("bf16")
    eng = A.InferenceEngine(model, backbone_dtype=torch.bfloat16)
    L = A._lib.lib()

    frames = torch.randn(F, 3, 112, 112, device=dev)
    audio = torch.randn(F, 1, 64, 1001, device=dev)                # one mel window per processed frame
    idx_host = (torch.arange(F)[:, None] + 3 * (torch.arange(T) - (T - 1))).clamp(0, F - 1)     # built on the host, as a caller would
    idx = idx_host.to(dev)
    batches = [{"clip": frames[idx[i: i + BATCH_A]].permute(0, 2, 1, 3, 4).contiguous(), "audio_features": audio[i: i + BATCH_A]}
               for i in range(0, F, BATCH_A)]

    def run_a():
        return torch.cat([eng(x).clone() for x in batches])

    def run_b():
        bank = torch.cat([eng.frame_features(frames[i: i + CHUNK]) for i in range(0, F, CHUNK)])
        res = [eng.clips(bank, idx_host[i: i + CHUNK], audio[i: i + CHUNK]) for i in range(0, F, CHUNK)]
        return torch.cat([r[0] for r in res]), torch.cat([r[1] for r in res])

    with torch.no_grad():
        # library launches: (a) per 64-clip batch as captured in its graph (an eager run of the same forward), (b) per chunk
        n0 = L.avf_launch_count()
        eng._forward(batches[0]["clip"], batches[0]["audio_features"])
        n1 = L.avf_launch_count()
        bank0 = eng.frame_features(frames[:CHUNK])
        n2 = L.avf_launch_count()
        eng.clips(torch.cat([bank0] * (F // CHUNK)), idx_host[:CHUNK], audio[:CHUNK])
        n3 = L.avf_launch_count()
        launches = {"a_per_64_clip_batch": n1 - n0, "b_frame_features_per_256_frames": n2 - n1, "b_clips_per_256_clips": n3 - n2}
        del bank0

        run_a(), run_b()                                              # warm-up: graphs captured, cuDNN algorithms picked
        t_a, t_b = [], []
        for _ in range(ROUNDS):
            ms, out_a = elapsed_ms(run_a)
            t_a.append(ms)
            ms, (out_b, dec_b) = elapsed_ms(run_b)
            t_b.append(ms)
        la, lb = out_a[:, :12], out_b[:, :12]
        sure = la.abs() > 0.25
        agree = ((la > 0) == (lb > 0)) | ~sure

        # (c) the TFormer alone: indexed call against explicit gather + mask
        tf = model.video_model.video_model.t_former
        cbank = torch.randn(C_BANK, 512, device=dev)
        centre = torch.arange(C_CLIPS) * C_BANK // C_CLIPS
        raw = centre[:, None] + 3 * (torch.arange(T) - T // 2)
        cidx = torch.where((raw >= 0) & (raw < C_BANK), raw, torch.full_like(raw, -1)).to(dev)
        cidx32 = cidx.to(torch.int32)
        st = tf.spatial_transformer
        cases = {"indexed": lambda: tf.cls_features_indexed(cbank, cidx32),
                 "indexed_library_call": lambda: A.functional.tformer_fwd_indexed(cbank, cidx32, tf.cls_token.view(-1), tf.pos_embedding[0],
                                                                                  st.packed(), st.shape(C_CLIPS, T + 1)),
                 "gather_plus_mask": lambda: tf.cls_features(cbank[cidx.clamp(min=0)].reshape(-1, 512), mask=cidx >= 0)}
        c_launch, c_out = {}, {}
        for name, fn in cases.items():
            for _ in range(5):
                fn()
            m0 = L.avf_launch_count()
            c_out[name] = fn()
            c_launch[name] = L.avf_launch_count() - m0
        c_times = {name: [] for name in cases}
        for _ in range(C_ROUNDS):
            for name, fn in cases.items():
                ms, _ = elapsed_ms(lambda: [fn() for _ in range(C_ITERS)])
                c_times[name].append(ms / C_ITERS)

    med_a, med_b = statistics.median(t_a), statistics.median(t_b)
    c_med = {k: statistics.median(v) for k, v in c_times.items()}
    res = {"probe": "video_probe", "gpu": gpu_info(), "processed_frames": F, "clip_frames": T, "offsets": "3 * (arange(16) - 15), clamped",
           "backbone_dtype": "bf16", "precision": "bf16", "batch_a_clips": BATCH_A, "chunk_b": CHUNK, "rounds": ROUNDS,
           "ms_per_processed_frame": {"a_clips": round(med_a / F, 5), "b_frame_bank": round(med_b / F, 5)},
           "ms_per_video_min_max": {"a_clips": [round(min(t_a), 3), round(max(t_a), 3)], "b_frame_bank": [round(min(t_b), 3), round(max(t_b), 3)]},
           "speedup_b_over_a": round(med_a / med_b, 3),
           "library_launches": launches,
           "max_abs_logit_diff_a_vs_b": float((la - lb).abs().max()),
           "decisions_compared_where_abs_logit_a_gt_0.25": int(sure.sum()), "decisions_disagreeing": int((~agree).sum()),
           "decisions_b_equal_own_logits": bool(torch.equal(dec_b, (lb > 0).to(torch.int32))),
           "logit_std_over_clips_a": float(la.std(dim=0).mean()), "logit_range_a": [float(la.min()), float(la.max())],
           "tformer_512x16_from_600": {"ms_per_call_median": {k: round(v, 5) for k, v in c_med.items()},
                                       "ms_per_call_min_max": {k: [round(min(v), 5), round(max(v), 5)] for k, v in c_times.items()},
                                       "ratio_to_gather_plus_mask": {k: round(v / c_med["gather_plus_mask"], 4) for k, v in c_med.items()},
                                       "library_launches_per_call": c_launch,
                                       "bit_identical": all(torch.equal(v, c_out["gather_plus_mask"]) for v in c_out.values())}}
    line = json.dumps(res)
    print(line)
    if out_path:
        with open(out_path, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
