"""Cost of the attention relevance at sizes a user runs, with CUDA events, on one GPU.

Full model (bf16 stacks, fp32 conv trunks), 64 clips x 16 frames, in eval(): model(x), attention_maps(x), and attention_relevance(x, au)
for all stacks and for stacks=["tformer"], alternating inside each round; the gradient-map bytes written.  Then the encoder-stack
backward (activations only, no weight gradients) with and without the gradient maps at the SFormer's shape (64 x 16 frames of 49
tokens, dim 256, depth 1) and the TFormer's (64 clips of 17 tokens, dim 512, depth 3), alternating; each call starts from a fresh copy
of the same incoming gradient, in both variants.  Medians over rounds.  The card's name, power limit and max SM clock are read in the
same run.

    python tools/attention_relevance_probe.py --out profiles/r13_attention_relevance_probe.json
"""
import argparse
import json
import os
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))
import avformer_b200 as A  # noqa: E402
from attention_maps_probe import HBM_TBPS, _card, _rounds  # noqa: E402
from oracle import avformer_oracle as O  # noqa: E402

AF = A.functional


def _stack_bwd(name, dim, depth, heads, dh, mlp, n_seq, n_tok, rounds, reps):
    m = A.Transformer(dim, depth, heads, dh, mlp)
    m.load_state_dict(O.params_from_spec(list(O._encoder_spec("", dim, depth, heads * dh, mlp)), 3), strict=True)
    m = m.cuda().eval()
    m.precision = "bf16"
    x = torch.randn(n_seq * n_tok, dim, device="cuda")
    dy = torch.randn(n_seq * n_tok, dim, device="cuda")
    d = torch.empty_like(dy)
    with torch.no_grad():
        _, tape = m.relevance_fwd_(x, n_seq, n_tok)

        def plain():
            d.copy_(dy)
            m.relevance_bwd_(d, tape, n_seq, n_tok, maps=False)

        def gmaps():
            d.copy_(dy)
            m.relevance_bwd_(d, tape, n_seq, n_tok)
        t = _rounds({"bwd": plain, "bwd_gradmaps": gmaps}, rounds, reps)
    nbytes = depth * n_seq * heads * n_tok * n_tok * 4
    extra = t["bwd_gradmaps"] - t["bwd"]
    return {"stack": name, "n_seq": n_seq, "n_tok": n_tok, "dim": dim, "depth": depth, "ms": t, "gmap_bytes": nbytes,
            "extra_ms": extra, "write_TBps_over_extra": nbytes / extra / 1e9 if extra > 0 else None}


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
    _, rel_all = m.attention_relevance(x, 0)
    _, rel_tf = m.attention_relevance(x, 0, ["tformer"])
    with torch.no_grad():
        t = _rounds({"model": lambda: m(x), "maps_all": lambda: m.attention_maps(x), "relevance_all": lambda: m.attention_relevance(x, 0),
                     "relevance_tformer": lambda: m.attention_relevance(x, 0, ["tformer"])}, args.rounds, args.reps)
    res["model_64x16"] = {"clips": n_clips, "T": T, "ms": t,
                          "gmap_bytes": {"all": sum(g.numel() * 4 for g, _ in rel_all.values()), "tformer": sum(g.numel() * 4 for g, _ in rel_tf.values())},
                          "gmap_bytes_by_stack": {k: g.numel() * 4 for k, (g, _) in rel_all.items()}}
    res["stack_bwd"] = [_stack_bwd("sformer", 256, 1, 8, 32, 512, n_clips * T, 49, args.rounds, args.reps * 4),
                        _stack_bwd("tformer", 512, 3, 8, 64, 1024, n_clips, T + 1, args.rounds, args.reps * 4)]
    res["hbm_TBps_datasheet"] = HBM_TBPS
    line = json.dumps(res)
    print(line)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        f.write(line + "\n")


if __name__ == "__main__":
    main()
