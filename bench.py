#!/usr/bin/env python
"""bench.py — AVFormer hot-path throughput on B200 (clips/s), with roofline and CPU baseline.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--mode fwd|train] [--check] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

`--dump-outputs DIR` writes what the last timed step computed on rank 0 as DIR/<name>.npy (fp32; sample indices in fp64), so
that two builds can be compared output for output: the inputs and weights are seeded, identical from run to run.

`--mode train` makes the hot-path TRAINING step (BASELINE config 4 restricted to the transformer stack: forward with tape,
AULoss, backward, gradient all-reduce overlapped with the backward at N > 1, fused Adam) the measured thing, with the same JSON
schema, its own end-to-end number and its own CPU reference arm (`--impl reference --mode train`).  `--check` (any N, meant
for N > 1 under torchrun) runs the data-parallel parity checks instead of timing: the gathered logits of N ranks against the
one-GPU result on the concatenated batch, and the all-reduced gradient bucket against the one-GPU large-batch gradient.

A *step* is one pass of the transformer hot path (SURVEY.md §8: SFormer -> TFormer -> AU_former x2 ->
fusion head -> logits/decisions) over one synthetic batch of 512 clips x 16 frames PER GPU (weak scaling;
BASELINE.json config 3's clip count with config 2's per-frame SFormer in front of it):
    stage-3 maps   [8192, 256, 7, 7] bf16   (205 MB: larger than the 126 MB L2, so no flush is needed)
    frame features [8192, 512]       bf16   (stand-in for conv stage 4, which is outside the hot path)
    audio features [512, 512]        fp32
`value` times it with the inputs resident in HBM; `e2e` times the same call from pinned HOST buffers,
H2D copies and the D2H read of logits+decisions included.  At N > 1 every rank processes its own 512 clips and
the step ends with the evaluation-time logit all-gather over NCCL.

`--impl reference` times the CPU arm: the oracle port of the reference's PyTorch path (fp32, all host threads) on
a bounded sample of the same workload.  The reference itself is Python source that cannot travel to the GPU box.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True           # a benchmark run leaves the tree as it found it (no __pycache__ of the modules it imports)

CLIPS_PER_GPU = 512
N_FRAMES = 16
SEED = 2024

# algorithmic FLOPs, SURVEY.md §8(a)/(d)  (F(N,D,I,M) = 2ND3I + 4N^2 I + 2NID + 4NDM)
FLOP_SFORMER_PER_FRAME = 53_838_848
FLOP_TFORMER_PER_CLIP = {8: 113_743_872, 16: 215_685_120, 32: 421_926_912}
FLOP_AU_FORMER_PER_CLIP = 11_308_032
FLOP_FUSION_PER_CLIP = 28_760_064


def hot_path_flops_per_clip(T):
    return T * FLOP_SFORMER_PER_FRAME + FLOP_TFORMER_PER_CLIP[T] + 2 * FLOP_AU_FORMER_PER_CLIP + FLOP_FUSION_PER_CLIP


# --dump-outputs: the full SFormer output (8192 maps, 411 MB in fp32) and the flat parameter / gradient buckets of the training step
# (41.7 MB each) are larger than the dump may be, so a fixed, seeded sample of them is written
DUMP_MAX_BYTES = 64 << 20
DUMP_SFORMER_FRAMES = 512                # 25.7 MB in fp32
DUMP_BUCKET_ELEMENTS = 1 << 20           # 4 MB per bucket in fp32


def dump_sample(n, k):
    """k indices of range(n), sorted, the same in every run."""
    import torch
    return torch.randperm(n, generator=torch.Generator().manual_seed(SEED))[:k].sort().values


def dump_outputs(out_dir, arrays):
    """Write each tensor as out_dir/<name>.npy: fp64 stays fp64, everything else becomes fp32."""
    import numpy as np
    import torch
    host = {k: v.detach().cpu() for k, v in arrays.items()}
    host = {k: (v.double() if v.dtype == torch.float64 else v.float()).numpy() for k, v in host.items()}
    total = sum(a.nbytes for a in host.values())
    if total > DUMP_MAX_BYTES:
        raise RuntimeError(f"--dump-outputs: {total} bytes exceed the {DUMP_MAX_BYTES} byte budget")
    os.makedirs(out_dir, exist_ok=True)
    for name, a in host.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


def measured_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        p = json.load(open(path))
        return {"bf16_tflops": p["bf16_tflops"], "bf16_tflops_sustained": p.get("bf16_tflops_sustained", p["bf16_tflops"]),
                "hbm_gbs": p["hbm_gbs"], "source": "measured"}
    return {"bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0, "hbm_gbs": 6650.0, "source": "fallback"}


# --------------------------------------------------------------------------------------------
# clocks (sampled DURING the timed region)
# --------------------------------------------------------------------------------------------
class ClockSampler:
    REASONS = {0x8: "hw_slowdown", 0x40: "hw_thermal_slowdown", 0x20: "sw_thermal_slowdown", 0x4: "sw_power_cap",
               0x80: "hw_power_brake", 0x2: "applications_clocks", 0x100: "display_clocks", 0x10: "sync_boost"}

    def __init__(self, index):
        self.index, self.samples, self.reasons, self.max_mhz = index, [], set(), None
        self._stop = threading.Event()
        self._thread = None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception:
            self.nv = None

    def _run(self):
        while not self._stop.is_set():
            try:
                self.samples.append(self.nv.nvmlDeviceGetClockInfo(self.h, self.nv.NVML_CLOCK_SM))
                mask = self.nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for bit, name in self.REASONS.items():
                    if mask & bit:
                        self.reasons.add(name)
            except Exception:
                pass
            self._stop.wait(0.02)

    def __enter__(self):
        if self.nv is not None:
            self._thread = threading.Thread(target=self._run, daemon=True)
            self._thread.start()
        return self

    def __exit__(self, *a):
        self._stop.set()
        if self._thread is not None:
            self._thread.join()

    def summary(self):
        if not self.samples:
            try:
                out = subprocess.run(["nvidia-smi", "-i", str(self.index), "--query-gpu=clocks.sm,clocks.max.sm", "--format=csv,noheader,nounits"],
                                     capture_output=True, text=True, timeout=10).stdout.strip().split(",")
                return {"sm_mhz": float(out[0]), "sm_max_mhz": float(out[1]), "reasons": [], "samples": 0, "note": "sampled after the region"}
            except Exception:
                return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        return {"sm_mhz": float(statistics.median(self.samples)), "sm_max_mhz": float(self.max_mhz), "reasons": sorted(self.reasons),
                "samples": len(self.samples)}


# --------------------------------------------------------------------------------------------
# CPU arm (oracle port of the reference)
# --------------------------------------------------------------------------------------------
def cpu_hot_path_clips_per_s(sample_clips, repeats, T=N_FRAMES):
    import torch
    from oracle import avformer_oracle as O
    torch.set_num_threads(os.cpu_count())
    p = O.make_state_dict(SEED, T, hot_path_only=True)
    stage3, frame, audio = O.synth_hot_path_inputs(SEED, sample_clips, T)
    best = float("inf")
    with torch.no_grad():
        O.hot_path_forward(stage3[: T * 2], frame[: T * 2], audio[:2], p, T)          # warm-up
        for _ in range(repeats):
            t0 = time.perf_counter()
            O.hot_path_forward(stage3, frame, audio, p, T)
            best = min(best, time.perf_counter() - t0)
    return sample_clips / best, best, torch.get_num_threads()


def cpu_train_step_clips_per_s(sample_clips, repeats, T=N_FRAMES):
    """Oracle port of one training step of the hot path on the host CPU: forward, AULoss, autograd backward, Adam on every
    hot-path parameter (train.py:206-236)."""
    import torch
    from oracle import avformer_oracle as O
    torch.set_num_threads(os.cpu_count())
    p = O.make_state_dict(SEED, T, hot_path_only=True)
    stage3, frame, audio = O.synth_hot_path_inputs(SEED, sample_clips, T)
    labels = (torch.rand(sample_clips, 12, generator=torch.Generator().manual_seed(SEED)) < 0.3).float()
    state = {}

    def one_step(step):
        loss, grads, _, _ = O.hot_path_grads(stage3, frame, audio, labels, p, T, batch_stats=True, sformer_loss_weight=1.0)
        for k, g in grads.items():
            m, v = state.get(k, (torch.zeros_like(g), torch.zeros_like(g)))
            p[k], m, v = O.adam_update(p[k], g, m, v, step, lr=5e-4, weight_decay=5e-5)
            state[k] = (m, v)
        return loss

    one_step(1)                                                                        # warm-up
    best = float("inf")
    for r in range(repeats):
        t0 = time.perf_counter()
        one_step(2 + r)
        best = min(best, time.perf_counter() - t0)
    return sample_clips / best, best, torch.get_num_threads()


def run_reference_arm(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    if args.mode == "train":
        return run_reference_arm_train(args)
    import torch
    from oracle import avformer_oracle as O
    torch.set_num_threads(os.cpu_count())
    T = N_FRAMES
    p = O.make_state_dict(SEED, T, hot_path_only=True)
    # size the per-step sample so that the whole run stays within ~2 minutes
    probe = 8
    s3, fr, au = O.synth_hot_path_inputs(SEED, probe, T)
    with torch.no_grad():
        O.hot_path_forward(s3, fr, au, p, T)
        t0 = time.perf_counter()
        O.hot_path_forward(s3, fr, au, p, T)
        per_clip = (time.perf_counter() - t0) / probe
    budget = 100.0 / max(1, args.steps + args.warmup)
    sample = int(max(4, min(CLIPS_PER_GPU, budget / per_clip)))
    s3, fr, au = O.synth_hot_path_inputs(SEED, sample, T)
    with torch.no_grad():
        for _ in range(args.warmup):
            O.hot_path_forward(s3, fr, au, p, T)
        t0 = time.perf_counter()
        for _ in range(args.steps):
            O.hot_path_forward(s3, fr, au, p, T)
        dt = time.perf_counter() - t0
    value = sample * args.steps / dt
    cores = torch.get_num_threads()
    line = {
        "impl": "reference", "metric": "AVFormer hot-path clips/sec (forward)", "value": value, "unit": "clips/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": dt / args.steps * 1e3,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": workload_config(sample_note=f"each step = {sample} clips of the workload on the host CPU"),
        "cpu_baseline": {"value": value, "unit": "clips/s", "cores": cores, "kind": "port",
                         "sample": f"{sample} clips x {T} frames per step, {args.steps} steps, torch {torch.__version__} fp32, {cores} threads"},
        "e2e": {"value": value, "unit": "clips/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line))


def run_reference_arm_train(args):
    import torch
    T = N_FRAMES
    v1, t1, cores = cpu_train_step_clips_per_s(4, 1)                                    # size the per-step sample: ~100 s for the whole run
    per_clip = t1 / 4
    budget = 100.0 / max(1, args.steps + args.warmup)
    sample = int(max(2, min(TRAIN_CLIPS_PER_GPU, budget / per_clip)))
    from oracle import avformer_oracle as O
    torch.set_num_threads(os.cpu_count())
    p = O.make_state_dict(SEED, T, hot_path_only=True)
    stage3, frame, audio = O.synth_hot_path_inputs(SEED, sample, T)
    labels = (torch.rand(sample, 12, generator=torch.Generator().manual_seed(SEED)) < 0.3).float()
    state = {}

    def one_step(step):
        _, grads, _, _ = O.hot_path_grads(stage3, frame, audio, labels, p, T, batch_stats=True, sformer_loss_weight=1.0)
        for k, g in grads.items():
            m, v = state.get(k, (torch.zeros_like(g), torch.zeros_like(g)))
            p[k], m, v = O.adam_update(p[k], g, m, v, step, lr=5e-4, weight_decay=5e-5)
            state[k] = (m, v)

    for i in range(args.warmup):
        one_step(1 + i)
    t0 = time.perf_counter()
    for i in range(args.steps):
        one_step(1 + args.warmup + i)
    dt = time.perf_counter() - t0
    value = sample * args.steps / dt
    line = {
        "impl": "reference", "metric": TRAIN_METRIC, "value": value, "unit": "clips/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": dt / args.steps * 1e3,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": train_config(sample_note=f"each step = {sample} clips of the workload on the host CPU"),
        "cpu_baseline": {"value": value, "unit": "clips/s", "cores": cores, "kind": "port",
                         "sample": f"{sample} clips x {T} frames per step, {args.steps} steps: oracle forward + autograd backward + Adam, torch {torch.__version__} fp32, {cores} threads"},
        "e2e": {"value": value, "unit": "clips/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line))


TRAIN_METRIC = "AVFormer hot-path training step clips/sec (fwd + bwd + fused Adam, gradient all-reduce at N>1)"


def train_config(sample_note=None):
    cfg = {"workload": f"avformer_hot_path_train: {TRAIN_CLIPS_PER_GPU} clips/GPU x {N_FRAMES} frames (BASELINE config 4 restricted to the transformer "
                       f"stack: SFormer + TFormer + AU_former x2 + fusion head, all their parameters trainable, BatchNorm1d batch statistics, AULoss, "
                       f"Adam(lr 5e-4, wd 5e-5) as train.py:334; the conv backbones are outside the hot path)",
           "clips_per_gpu": TRAIN_CLIPS_PER_GPU, "n_frames": N_FRAMES,
           "parallelism": "clip-sharded data parallel; one NCCL sum-all-reduce of the flat fp32 gradient bucket behind the backward pass, 1/N folded into "
                          "the fused Adam kernel (AVF_OVERLAP_REDUCE=1: per-stack segments reduced from the backward bridges instead, measured slower)",
           "l2": "per-step working set (activations tape ~0.4 GB) is larger than the 126 MB L2; no explicit flush",
           "flop_per_clip": 3 * hot_path_flops_per_clip(N_FRAMES)}
    if sample_note:
        cfg["sample"] = sample_note
    return cfg


def workload_config(sample_note=None):
    cfg = {"workload": f"avformer_hot_path_eval: {CLIPS_PER_GPU} clips/GPU x {N_FRAMES} frames "
                       f"(SFormer on {CLIPS_PER_GPU * N_FRAMES} stage-3 maps [256,7,7] + TFormer + AU_former x2 + fusion head -> 12-AU logits)",
           "clips_per_gpu": CLIPS_PER_GPU, "n_frames": N_FRAMES, "parallelism": "clip-sharded data parallel; at N>1 every step contains the gather of the [512, 21] logits of all ranks, inside the timed region (pushed over NVLink peer memory from inside the captured graph right behind the fusion head; the step's graph ends with the wait for all N blocks)",
           "l2": "inputs (205 MB of stage-3 maps per step) are larger than the 126 MB L2; no explicit flush",
           "flop_per_clip": hot_path_flops_per_clip(N_FRAMES)}
    if sample_note:
        cfg["sample"] = sample_note
    return cfg


# --------------------------------------------------------------------------------------------
# GPU arm
# --------------------------------------------------------------------------------------------
def run_ours(args):
    import torch
    import torch.distributed as dist
    import avformer_b200 as A

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    T, B = N_FRAMES, CLIPS_PER_GPU

    torch.manual_seed(SEED)                      # random-init weights of the reference architecture (no checkpoints offline)
    model = A.TwoStreamAuralVisualFormer(video_pretrained=False, audio_pretrained=False, task="AU")
    model = model.to(dev).eval().set_precision("bf16")
    if args.check:
        ok = run_dp_check(model, A, dev, rank, world)
        if world > 1:
            dist.destroy_process_group()
        sys.exit(0 if ok else 1)
    if args.mode == "train":
        run_train(model, A, dev, rank, world, args)
        if world > 1:
            dist.destroy_process_group()
        return

    g = torch.Generator(device="cpu").manual_seed(SEED + rank)
    host = {
        "stage3": torch.clamp(torch.randn(B * T, 256, 7, 7, generator=g) * 1.7 + 0.6, min=0).bfloat16().pin_memory(),
        "frame": (torch.randn(B * T, 512, generator=g).abs() * 1.2).bfloat16().pin_memory(),
        "audio": torch.randn(B, 512, generator=g).abs().pin_memory(),
    }
    devin = {k: v.to(dev) for k, v in host.items()}
    gathered = torch.empty((world * B, 21), dtype=torch.float32, device=dev) if world > 1 else None

    def step(inp):
        s_out, out21, dec = model.hot_path(inp["stage3"], inp["frame"], inp["audio"], want_decisions=True)
        if world > 1:
            dist.all_gather_into_tensor(gathered, out21)
        return s_out, out21, dec

    L = A._lib.lib()
    with torch.no_grad():
        for _ in range(max(args.warmup, 3)):
            step(devin)
        torch.cuda.synchronize()
        n0 = L.avf_launch_count()
        step(devin)
        launches_per_step = L.avf_launch_count() - n0

        # ---- device-resident timing --------------------------------------------------------
        def barrier():
            if world > 1:
                dist.barrier()
            torch.cuda.synchronize()

        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        barrier()
        e0.record()
        for _ in range(args.steps):
            step(devin)
        e1.record()
        barrier()
        ms_eager = e0.elapsed_time(e1) / args.steps

        # the same step captured once as a CUDA graph (no launch gaps, audio branch on a parallel graph branch): the headline
        # (AVF_SM_SPLIT="116,32" runs the persistent SFormer kernel on 116 SMs NEXT TO the TFormer / head chain on the other 32 —
        #  measured on B200: 1.458 ms against 1.450 ms one after the other, so it is off by default)
        sm_split = None
        if os.environ.get("AVF_SM_SPLIT", "") not in ("", "0", "off"):
            sm_split = tuple(int(v) for v in os.environ["AVF_SM_SPLIT"].split(","))
        # AVF_SM_RESERVE=k (developer A/B, goes with AVF_GATHER=pipelined): leave k SMs out of the persistent grids for the NCCL CTAs of
        # an asynchronous gather — measured slower on 2 and 8 GPUs than the plain in-stream gather on all SMs, so 0 by default.
        n_sm = torch.cuda.get_device_properties(dev).multi_processor_count
        sm_reserve = int(os.environ.get("AVF_SM_RESERVE", "0"))
        if sm_reserve > 0:
            L.avf_set_sm_cap(n_sm - sm_reserve)
        # the logit gather of N > 1.  peer (default): pushes over NVLink peer memory inside the captured graph (csrc/avf_peer.cu: push behind
        # the fusion head, bounded wait at the end of the step); instream: an NCCL all-gather behind every replay (1.183 ms per step on 8 B200s
        # against 1.107 ms on one); ingraph: the NCCL all-gather as a graph branch under the SFormer kernel (1.303 ms: slower, the two grids
        # race for SMs); pipelined: NCCL, asynchronous, one batch late
        gather_mode = os.environ.get("AVF_GATHER", "peer") if world > 1 else "none"      # developer A/B: peer | ingraph | instream | pipelined | none
        peer, gather_note = None, None
        if gather_mode == "peer":
            try:
                peer = A.dp.PeerLogitGather(B, 21, timeout_s=30.0)
            except Exception as ex:                 # no peer mapping on this box (symmetric memory unavailable): NCCL in the stream instead, and say so
                gather_note = f"peer-memory gather unavailable ({type(ex).__name__}: {str(ex)[:160]}); NCCL all-gather in the stream instead"
            agree = torch.tensor([1 if peer is not None else 0], device=dev)
            dist.all_reduce(agree, op=dist.ReduceOp.MIN)
            if int(agree.item()) == 0:
                peer, gather_mode = None, "instream"
        graphed = A.GraphedHotPath(model, devin["stage3"], devin["frame"], devin["audio"], sm_split=sm_split,
                                   gather_into=peer if peer is not None else (gathered if gather_mode == "ingraph" else None))
        L.avf_set_sm_cap(0)

        pipe = A.dp.PipelinedLogitGather()       # N > 1: the gather of batch i runs under the kernels of batch i+1

        def gstep():
            _, out21, _ = graphed.replay()
            if gather_mode == "pipelined":
                pipe.submit(out21)
            elif gather_mode == "instream" and world > 1:
                dist.all_gather_into_tensor(gathered, out21)

        for _ in range(3):
            gstep()
        barrier()
        with ClockSampler(local) as clocks:
            e0.record()
            for _ in range(args.steps):
                gstep()
            pipe.wait()                          # every gather is complete inside the timed region
            e1.record()
            barrier()
        ms_total = e0.elapsed_time(e1)
        gather_ok = None
        if world > 1 and gather_mode in ("peer", "ingraph", "instream"):
            # what the timed step gathered: my own shard sits at my rank's offset, and every rank holds the same [N * 512, 21] table
            if peer is not None:
                peer.check()                     # no wait timed out, device and host step counts agree
            tbl = peer.table() if peer is not None else gathered
            mine_ok = torch.equal(tbl[rank * B:(rank + 1) * B], graphed.out[1])
            chk = torch.stack([tbl.double().sum(), -tbl.double().sum(), torch.tensor(0.0 if mine_ok else 1.0, dtype=torch.float64, device=dev)])
            dist.all_reduce(chk, op=dist.ReduceOp.MAX)
            gather_ok = bool(chk[0].item() == -chk[1].item() and chk[2].item() == 0.0)
        if args.dump_outputs and rank == 0:
            s_out, out21, dec = graphed.out
            frames = dump_sample(s_out.shape[0], DUMP_SFORMER_FRAMES)
            dumped = {"out21": out21, "decisions": dec, "sformer_out_sample": s_out[frames.to(dev)],
                      "sformer_out_sample_frames": frames.double()}
            if gather_ok is not None:
                dumped["gathered_out21"] = tbl
            dump_outputs(args.dump_outputs, dumped)
        parity = timed_outputs_vs_oracle(model, graphed.out, host, T) if rank == 0 else None

        # ---- end to end from pinned host buffers ---------------------------------------------
        out_host = torch.empty((B, 21), dtype=torch.float32).pin_memory()
        dec_host = torch.empty((B, 12), dtype=torch.int32).pin_memory()

        def e2e_step():
            _, out21, dec = model.hot_path_from_host(host["stage3"], host["frame"], host["audio"], out_host, dec_host)
            if world > 1:
                dist.all_gather_into_tensor(gathered, out21)

        e2e_steps = max(3, min(args.steps, 20))
        for _ in range(2):
            e2e_step()
        barrier()
        e0.record()
        for _ in range(e2e_steps):
            e2e_step()
        e1.record()
        barrier()
        ms_e2e = e0.elapsed_time(e1) / e2e_steps

        # ---- per-stage breakdown + dominant-kernel roofline (timed alone, CUDA events) ---------
        vm = model.video_model.video_model

        def time_fn(fn, reps=20):
            # warm-up, synchronize, then ONE more untimed launch in front of the start event: the host enqueues the timed launches
            # while the GPU is still busy with it, so the events bracket kernel time and not the host's launch latency on an idle GPU
            for _ in range(3):
                fn()
            torch.cuda.synchronize()
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            fn()
            a.record()
            for _ in range(reps):
                fn()
            b.record()
            torch.cuda.synchronize()
            return a.elapsed_time(b) / reps

        ms_sformer = time_fn(lambda: vm.s_former.sformer(devin["stage3"]))
        ms_tformer = time_fn(lambda: vm.t_former.cls_features(devin["frame"]))
        roof = A.functional.sformer_roofline_probe(devin["stage3"], vm.s_former, time_fn) \
            if hasattr(A.functional, "sformer_roofline_probe") else None

    t = torch.tensor([ms_total, ms_e2e], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_total, ms_e2e = t.tolist()
    ms_step = ms_total / args.steps
    value = world * B / (ms_step * 1e-3)
    peaks = measured_peaks()

    if rank == 0:
        flops_sformer = B * T * FLOP_SFORMER_PER_FRAME
        if roof is None:
            roof = {"kernel": "encoder_fused_kernel<0>: the whole SFormer region (NCHW->tokens +pos, LN, QKV, attention, out-proj, MLP, tokens->NCHW) "
                              "as ONE persistent tcgen05 kernel, 1 launch per step, timed alone with CUDA events on its launch stream",
                    "achieved": flops_sformer / (ms_sformer * 1e-3) / 1e12, "launches": 1}
            tpath = os.path.join(ROOT, "profiles", "roofline_traffic.json")
            if os.path.exists(tpath):        # dram__bytes_read.sum + dram__bytes_write.sum of that kernel from the committed ncu --set full capture
                tj = json.load(open(tpath))
                roof["traffic"] = tj["dram_bytes_read"] + tj["dram_bytes_write"]
                roof["traffic_source"] = tj["source"]
                roof["algorithmic_bytes"] = tj["algorithmic_bytes"]
        roofline = {"bound": "tensor", "achieved": roof["achieved"], "peak": peaks["bf16_tflops"], "unit": "TFLOP/s",
                    "frac": roof["achieved"] / peaks["bf16_tflops"], "traffic": roof.get("traffic"),
                    "kernel": roof["kernel"], "peak_source": f"{peaks['source']} (burst: kernel timed alone)",
                    "algorithmic_flop_per_launch": flops_sformer, "traffic_source": roof.get("traffic_source"),
                    "algorithmic_bytes_per_launch": roof.get("algorithmic_bytes"), "share_of_step": ms_sformer / ms_step}
        sample = 64
        if world == 1:            # the CPU arm is timed on rank 0 at N=1 only (the other ranks' processes would share the host cores)
            cpu_v, cpu_t, cores = cpu_hot_path_clips_per_s(sample, repeats=3)
            cpu_baseline = {"value": cpu_v, "unit": "clips/s", "cores": cores, "kind": "port",
                            "sample": f"{sample} clips x {T} frames, best of 3, oracle port (torch fp32 CPU) of the same hot path"}
        else:
            cpu_baseline = None
        h2d = sum(v.numel() * v.element_size() for v in host.values())
        d2h = out_host.numel() * 4 + dec_host.numel() * 4
        line = {
            "metric": "AVFormer hot-path clips/sec (forward)", "value": value, "unit": "clips/s", "n_gpus": world,
            "steps": args.steps, "warmup": max(args.warmup, 3), "ms_per_step": ms_step, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "bf16", "data": "synthetic", "config": workload_config(),
            "clocks": clocks.summary(),
            "e2e": {"value": world * B / (ms_e2e * 1e-3), "unit": "clips/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                    "ms_per_step": ms_e2e, "note": "model.hot_path_from_host() on pinned host buffers: chunked H2D of all inputs on a copy stream overlapped with the kernels (two alternating device staging sets: the copies of step i+1 start under the kernels of step i) + D2H of logits/decisions"},
            "gpu_launches": int(launches_per_step * args.steps),
            "gpu_launches_per_step": int(launches_per_step),
            "roofline": roofline,
            "cpu_baseline": cpu_baseline,
            "gather": gather_mode, "gather_note": gather_note, "gather_checked": gather_ok, "parity_max_err": parity["logits_max_abs_err"], "decisions_match": parity["decisions_match"], "parity": parity,
            "tensor_frac_whole_step": value / world * hot_path_flops_per_clip(T) / 1e12 / peaks["bf16_tflops_sustained"],
            "breakdown_ms": {"sformer": ms_sformer, "tformer": ms_tformer, "whole_step": ms_step, "whole_step_eager_launches": ms_eager},
            "flops_per_clip": {"algorithmic": hot_path_flops_per_clip(T), "executed": hot_path_flops_per_clip(T) - tformer_skipped_flops_per_clip(T),
                               "note": "executed = algorithmic minus the last TFormer layer's out-projection and MLP on the T non-cls rows, which "
                                       "models/vformer.py:290 never reads (tensor_frac_whole_step uses the algorithmic count)"},
            "launch_mode": "one CUDA-graph replay per step (captured from the library's own kernel launches; gpu_launches counts the kernels inside it)"
                           + (f"; SFormer kernel on {sm_split[0]} SMs next to the TFormer/head chain on {sm_split[1]} SMs (avf_set_sm_cap)" if sm_split else ""),
            "train": {"see": "python bench.py --mode train (its own JSON line, reference arm and end-to-end number)"},
        }
        print(json.dumps(line), flush=True)
    if world > 1:
        graphed.release()                        # a graph holding NCCL nodes (AVF_GATHER=ingraph) goes before the communicator
        del graphed
        peer = None
        dist.barrier()
        dist.destroy_process_group()


TRAIN_CLIPS_PER_GPU = 64


def tformer_skipped_flops_per_clip(T):
    """Last TFormer layer, T non-cls rows: out-projection 2*I*D + MLP 4*D*M per row (D = I = 512, M = 1024)."""
    return T * (2 * 512 * 512 + 4 * 512 * 1024)


def timed_outputs_vs_oracle(model, outs, host, T, n_clips=8):
    """Certify what was timed: the first `n_clips` clips of the LAST timed step's outputs (the graph's static output tensors)
    against the fp64 oracle on the same inputs and weights.  Tolerances are north_star's bf16 ones."""
    import torch
    from oracle import avformer_oracle as O
    s_out, out21, dec = outs
    p = {k: v.detach().double().cpu() for k, v in model.state_dict().items()}
    ref = O.hot_path_forward(host["stage3"][: n_clips * T].double(), host["frame"][: n_clips * T].double(), host["audio"][:n_clips].double(), p, T)
    logits = out21[:n_clips, :12].double().cpu()
    err = (logits - ref["logits"]).abs().max().item()
    sure = ref["logits"].abs() > 2e-2
    dec_ok = bool((((dec[:n_clips].cpu() > 0) == (ref["logits"] > 0)) | ~sure).all())
    s_err = (s_out[: n_clips * T].double().cpu() - ref["sformer_out"]).abs()
    return {"clips_checked": n_clips, "logits_max_abs_err": err, "logits_tolerance": 2e-2, "decisions_match": dec_ok,
            "sformer_max_abs_err": s_err.max().item(), "sformer_mean_abs_err": s_err.mean().item(),
            "ok": bool(err < 2e-2 and dec_ok and s_err.max().item() < 0.2),
            "against": "oracle.hot_path_forward in fp64 on the same weights and the first clips of the timed batch"}


def _hot_params(model):
    return [p for k, p in model.named_parameters() if ".resnet." not in k and "s_former.conv1" not in k and "s_former.bn1" not in k
            and "s_former.layer" not in k]


def run_train(model, A, dev, rank, world, args):
    """The hot-path training step as the measured thing (BASELINE config 4 restricted to the transformer stack)."""
    import torch
    import torch.distributed as dist
    from avformer_b200.optim import segments_of
    T, B = N_FRAMES, TRAIN_CLIPS_PER_GPU
    g = torch.Generator(device="cpu").manual_seed(SEED + 100 + rank)
    host = {
        "stage3": torch.clamp(torch.randn(B * T, 256, 7, 7, generator=g) * 1.7 + 0.6, min=0).bfloat16().pin_memory(),
        "frame": (torch.randn(B * T, 512, generator=g).abs() * 1.2).pin_memory(),
        "audio": torch.randn(B, 512, generator=g).abs().pin_memory(),
        "labels": (torch.rand(B, 12, generator=g) < 0.3).float().pin_memory(),
    }
    stage3 = host["stage3"].to(dev).requires_grad_(True)
    frame = host["frame"].to(dev).requires_grad_(True)
    audio = host["audio"].to(dev).requires_grad_(True)
    labels = host["labels"].to(dev)
    probe = torch.randn(B * T, 256, 7, 7, generator=g).bfloat16().to(dev) * 1e-3          # stands in for d(loss)/d(sformer_out) from conv stage 4
    model.train()
    opt = A.FusedAdam(_hot_params(model), lr=5e-4, weight_decay=5e-5, segments=segments_of(model))
    L = A._lib.lib()

    def eager_step():
        opt.zero_grad()
        s_out, out21 = model.hot_path_train(stage3, frame, audio)
        loss = model.get_au_loss(out21, labels)
        torch.autograd.backward([loss, s_out], [None, probe])
        opt.step()
        return loss

    for _ in range(2):
        eager_step()
    torch.cuda.synchronize()
    n0 = L.avf_launch_count()
    eager_step()
    launches = int(L.avf_launch_count() - n0)
    graphed = A.GraphedTrainStep(model, opt, stage3, frame, audio, labels, probe)
    for _ in range(max(args.warmup, 3)):
        graphed.step()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    with ClockSampler(dev.index) as clocks:
        e0.record()
        for _ in range(args.steps):
            graphed.step()
        e1.record()
        barrier()
    ms_total = e0.elapsed_time(e1)
    if args.dump_outputs and rank == 0:
        # the last timed step: its loss, the gradients it computed and the parameters its Adam update wrote (flat buckets, sampled)
        bucket = opt._buckets[0]
        idx = dump_sample(bucket["p"].numel(), DUMP_BUCKET_ELEMENTS)
        dump_outputs(args.dump_outputs, {"loss": graphed.loss.reshape(1), "params_sample": bucket["p"][idx.to(dev)],
                                         "grads_sample": bucket["g"][idx.to(dev)], "bucket_sample_index": idx.double()})

    # end to end: inputs and labels from pinned host memory every step, the loss read back
    loss_host = torch.zeros(1, dtype=torch.float32).pin_memory()

    def e2e_step():
        loss = graphed.step(host["stage3"], host["frame"], host["audio"], host["labels"])
        loss_host.copy_(loss.reshape(1), non_blocking=True)

    e2e_steps = max(3, min(args.steps, 20))
    for _ in range(2):
        e2e_step()
    barrier()
    e0.record()
    for _ in range(e2e_steps):
        e2e_step()
    e1.record()
    barrier()
    ms_e2e = e0.elapsed_time(e1) / e2e_steps
    final_loss = float(loss_host.item())
    model.eval()

    t = torch.tensor([ms_total, ms_e2e], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_total, ms_e2e = t.tolist()
    ms_step = ms_total / args.steps
    if rank != 0:
        return
    peaks = measured_peaks()
    flops_step = 3 * B * hot_path_flops_per_clip(T)
    achieved = flops_step / (ms_step * 1e-3) / 1e12
    bucket_bytes = sum(b["g"].numel() * 4 for b in opt._buckets if b is not None)
    cpu_baseline = None
    if world == 1:
        sample = 4
        cpu_v, cpu_t, cores = cpu_train_step_clips_per_s(sample, repeats=2)
        cpu_baseline = {"value": cpu_v, "unit": "clips/s", "cores": cores, "kind": "port",
                        "sample": f"{sample} clips x {T} frames, best of 2: oracle forward + autograd backward + Adam (torch fp32 CPU) of the same step"}
    h2d = sum(v.numel() * v.element_size() for v in host.values())
    line = {
        "metric": TRAIN_METRIC, "value": world * B / (ms_step * 1e-3), "unit": "clips/s", "n_gpus": world, "steps": args.steps,
        "warmup": max(args.warmup, 3), "ms_per_step": ms_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "bf16", "data": "synthetic", "config": train_config(), "clocks": clocks.summary(),
        "e2e": {"value": world * B / (ms_e2e * 1e-3), "unit": "clips/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": 4, "ms_per_step": ms_e2e,
                "note": "GraphedTrainStep.step() fed from pinned host buffers (stage-3 maps, frame / audio features, labels) + D2H of the loss every step"},
        "gpu_launches": int(launches * args.steps), "gpu_launches_per_step": launches,
        "roofline": {"bound": "tensor", "achieved": achieved, "peak": peaks["bf16_tflops_sustained"], "unit": "TFLOP/s",
                     "frac": achieved / peaks["bf16_tflops_sustained"], "traffic": None,
                     "kernel": f"the whole training step ({launches} launches, none above 15 % of the step at 64 clips per GPU): algorithmic forward + backward "
                               "FLOPs (3 x forward) over the step time",
                     "peak_source": f"{peaks['source']} (sustained: a kernel chain timed inside a long step)", "algorithmic_flop_per_launch": flops_step},
        "cpu_baseline": cpu_baseline,
        "grad_bucket_bytes": bucket_bytes, "grad_allreduce": ("per-stack segments, asynchronous, started from the backward bridges (dp.SegmentReducer, NCCL)" if opt.overlap else
                                                               ("summed over ranks AND applied by ONE kernel over NVLink peer memory behind the backward (avf_adam_allreduce_step: two-shot all-reduce, in place, deterministic, then Adam on the replicated bucket)" if opt._buckets[0].get("peer") is not None
                                                                else "one NCCL all-reduce of the flat bucket behind the backward")) if world > 1 else None,
        "grad_allreduce_note": opt.reduce_note,
        "final_loss": final_loss,
        "launch_mode": "zero_grad + forward + AULoss + backward (+ the segment all-reduces at N>1) as ONE CUDA-graph replay, then the fused Adam launch",
    }
    print(json.dumps(line))


def run_dp_check(model, A, dev, rank, world):
    """SURVEY.md section 8(e) on hardware.  (1) evaluation: every rank runs the hot path on its own shard, the [N*b, 21] logits are
    all-gathered over NCCL; rank 0 also runs all N shards as ONE batch on its GPU and compares.  (2) training: every rank
    computes the gradients of its shard (BatchNorm1d on running statistics, no dropout: caveats 1 and 3), the bucket is
    all-reduced by FusedAdam's segment reducer and scaled by 1/N; rank 0 compares with the gradient of the mean loss over
    the concatenated batch computed on one GPU."""
    import torch
    import torch.distributed as dist
    from avformer_b200.optim import segments_of
    T, b = N_FRAMES, 48

    def inputs(r):
        g = torch.Generator(device="cpu").manual_seed(SEED + 7 + r)
        s3 = torch.clamp(torch.randn(b * T, 256, 7, 7, generator=g) * 1.7 + 0.6, min=0).bfloat16()
        fr = (torch.randn(b * T, 512, generator=g).abs() * 1.2).bfloat16()
        au = torch.randn(b, 512, generator=g).abs()
        lab = (torch.rand(b, 12, generator=g) < 0.3).float()
        return s3, fr, au, lab

    mine = [t.to(dev) for t in inputs(rank)]
    model.eval().set_dropout(0.0)
    with torch.no_grad():
        _, out21, dec = model.hot_path(mine[0], mine[1], mine[2], want_decisions=True)
    gathered = A.dp.gather_logits(out21, world * b)
    res = {"check": "dp_parity", "n_gpus": world, "clips_per_rank": b}
    if rank == 0:
        allin = [torch.cat([inputs(r)[i] for r in range(world)]).to(dev) for i in range(4)]
        with torch.no_grad():
            _, one, _ = model.hot_path(allin[0], allin[1], allin[2], want_decisions=True)
        d = (gathered - one).abs().max().item()
        res["logits_max_abs_diff"] = d
        res["logits_bit_identical"] = bool(torch.equal(gathered, one))
    # gradients
    params = _hot_params(model)
    for q in params:
        q.grad = None
    opt = A.FusedAdam(params, lr=0.0, segments=segments_of(model), overlap=True)

    def grads(s3, fr, au, lab, reduce):
        opt.zero_grad()
        s_out, o = model.hot_path_train(s3.clone().requires_grad_(True), fr.float().requires_grad_(True), au.clone().requires_grad_(True))
        loss = model.get_au_loss(o, lab) + 1e-3 * s_out.float().mean()
        loss.backward()
        if reduce:
            opt.finish_reductions()
        return loss.detach()

    grads(*mine, reduce=False)
    opt.step()                                       # lr 0: builds the flat bucket, changes nothing
    grads(*mine, reduce=True)                        # armed now: segments are all-reduced from the backward bridges
    bucket = opt._buckets[0]
    red = bucket.get("reducer")
    launched = list(red.launch_order) if red is not None else []
    avg = bucket["g"].clone() / world
    if red is not None:
        red.disarm()
    opt.overlap = False
    opt._reducer = None
    peer = bucket.get("peer")
    if peer is not None:
        # the same gradients through the one-kernel all-reduce over NVLink peer memory (FusedAdam's default): against the NCCL
        # result above (another summation order: a few ulp), and the same bits on every rank
        grads(*mine, reduce=False)
        peer.reduce_()
        res["grad_peer_reductions_completed"] = peer.check()
        avg_peer = bucket["g"].clone() / world
        res["grad_peer_vs_nccl_max_rel"] = ((avg_peer - avg).abs().max() / avg.abs().max()).item()
        hi, lo = avg_peer.clone(), avg_peer.clone()
        if world > 1:
            dist.all_reduce(hi, op=dist.ReduceOp.MAX)
            dist.all_reduce(lo, op=dist.ReduceOp.MIN)
        res["grad_peer_identical_on_all_ranks"] = bool(torch.equal(hi, lo))
        # adam_allreduce_step: reduction + Adam as one kernel against reduction, then avf_adam_step, on copies of the live buckets
        hyper = (5e-4, 0.9, 0.999, 1e-8, 5e-5)
        pa, ma, va = bucket["p"].clone(), torch.zeros_like(bucket["p"]), torch.zeros_like(bucket["p"])
        A.functional.adam_step_(pa, bucket["g"], ma, va, 1, *hyper, grad_scale=1.0 / world)
        grads(*mine, reduce=False)                   # the same local gradients again (the backward is deterministic)
        pb, mb, vb = bucket["p"].clone(), torch.zeros_like(bucket["p"]), torch.zeros_like(bucket["p"])
        peer.reduce_adam_(pb, mb, vb, 1, *hyper)
        peer.check()
        res["adam_allreduce_fused_bit_identical"] = bool(torch.equal(pa, pb) and torch.equal(ma, mb) and torch.equal(va, vb) and not torch.equal(pb, bucket["p"]))
    else:
        res["grad_peer_note"] = opt.reduce_note
    if rank == 0:
        grads(*allin, reduce=False)                  # the same loss over the concatenated batch on ONE GPU (equal shard sizes: mean of means)
        big = bucket["g"]
        worst = 0.0
        for q, o in zip(bucket["params"], bucket["offs"]):
            n = q.numel()
            ref = big[o:o + n]
            scale = ref.abs().max().item()
            if scale > 0:
                worst = max(worst, (avg[o:o + n] - ref).abs().max().item() / scale)
        res["grad_max_rel_err"] = worst
        res["grad_segments_reduced_in_order"] = launched
        res["ok"] = bool(res["logits_max_abs_diff"] <= 1e-5 and worst < 2e-3
                         and (peer is None or (res["grad_peer_vs_nccl_max_rel"] < 1e-5 and res["grad_peer_identical_on_all_ranks"]
                                              and res["adam_allreduce_fused_bit_identical"])))
        print(json.dumps(res))
    ok = torch.tensor([1 if (rank != 0 or res.get("ok")) else 0], device=dev)
    if world > 1:
        dist.all_reduce(ok, op=dist.ReduceOp.MIN)
    return bool(ok.item())


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=100)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--mode", default="fwd", choices=["fwd", "train"], help="what a step is: the evaluation hot path (default) or its training step")
    ap.add_argument("--check", action="store_true", help="data-parallel parity checks instead of timing (run under torchrun with N > 1)")
    ap.add_argument("--dump-outputs", metavar="DIR", default="",
                    help="write what the last timed step computed (rank 0) as DIR/<name>.npy, at most 64 MB in all")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl == "reference" or args.check):
        ap.error("--dump-outputs goes with the timed GPU path (--impl ours, without --check)")
    if args.impl == "reference":
        run_reference_arm(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
