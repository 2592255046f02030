"""Whole-model inference engine (SURVEY.md §8f-1): the conv backbones around the hot path — outside it by design, plain
torch / cuDNN — prepared the way a B200 wants them, without touching the model's parameters or state dict:

  * BatchNorm folded into the preceding convolution (eval statistics), weights kept as bf16 (or fp32) ``channels_last`` copies,
    so every conv is one cuDNN NHWC tensor-core kernel with a fused bias;
  * the transformer regions are the library's own kernels (fused SFormer, TFormer, AU_formers, fusion head);
  * the whole forward is captured per input shape as ONE CUDA graph (no tracing compiler: the graph replays exactly the
    cuDNN / libavformer_b200 launches of a warm-up run).

    eng = InferenceEngine(model, backbone_dtype=torch.bfloat16)
    out21 = eng({"clip": clip, "audio_features": mel})          # [B,21] like model(x), models/avformer.py:93-106

A whole video runs each frame through the video trunk once instead of once per clip that contains it (eager, no graph):

    bank = torch.cat([eng.frame_features(frames[i:i + 256]) for i in range(0, len(frames), 256)])   # [F,512]
    out21, decisions = eng.clips(bank, index, mel)              # index [n,T] frame numbers, -1 = missing; mel [n,1,64,1001]

``backbone_dtype=torch.float32`` reproduces ``model(x)`` up to the re-association of the BN fold (checked at 1e-3 in the
tests); bf16 backbones trade ~1e-1 absolute on the logits for tensor-core convolutions and are therefore opt-in.
"""
from __future__ import annotations

from typing import Dict, List, Optional, Tuple

import torch
import torch.nn.functional as F

from . import functional as AF
from .encoder import default_precision


def _fold(conv: torch.nn.Conv2d, bn: torch.nn.BatchNorm2d, dtype) -> Tuple[torch.Tensor, torch.Tensor]:
    """conv -> bn (eval) == conv with w * s and bias (beta - mean * s), s = gamma / sqrt(var + eps)."""
    s = (bn.weight.detach().float() / torch.sqrt(bn.running_var.detach().float() + bn.eps))
    w = (conv.weight.detach().float() * s[:, None, None, None]).to(dtype).contiguous(memory_format=torch.channels_last)
    b = (bn.bias.detach().float() - bn.running_mean.detach().float() * s).to(dtype)
    return w, b


class _FoldedBlock:
    def __init__(self, blk, dtype):
        self.w1, self.b1 = _fold(blk.conv1, blk.bn1, dtype)
        self.w2, self.b2 = _fold(blk.conv2, blk.bn2, dtype)
        self.stride = blk.conv1.stride
        self.down = _fold(blk.downsample[0], blk.downsample[1], dtype) if blk.downsample is not None else None
        self.down_stride = blk.downsample[0].stride if blk.downsample is not None else None

    def __call__(self, x):
        y = F.relu_(F.conv2d(x, self.w1, self.b1, self.stride, 1))
        y = F.conv2d(y, self.w2, self.b2, 1, 1)
        sc = x if self.down is None else F.conv2d(x, self.down[0], self.down[1], self.down_stride, 0)
        return F.relu_(y.add_(sc))


class _FoldedResNet:
    """conv1/bn1/relu/maxpool + layer1..4 of the ResNet-18 trunks (models/vformer.py:232-244,261-265; models/audio.py:22-39)."""

    def __init__(self, net, dtype):
        self.dtype = dtype
        self.stem = _fold(net.conv1, net.bn1, dtype)
        self.stem_stride, self.stem_pad = net.conv1.stride, net.conv1.padding
        self.layers: List[List[_FoldedBlock]] = [[_FoldedBlock(b, dtype) for b in getattr(net, f"layer{i}")] for i in range(1, 5)]

    def to_stage(self, x, first: int, last: int):
        for i in range(first, last + 1):
            for blk in self.layers[i - 1]:
                x = blk(x)
        return x

    def stem_fwd(self, img):
        x = img.to(self.dtype).contiguous(memory_format=torch.channels_last)
        x = F.relu_(F.conv2d(x, self.stem[0], self.stem[1], self.stem_stride, self.stem_pad))
        return F.max_pool2d(x, 3, 2, 1)


class InferenceEngine:
    def __init__(self, model, backbone_dtype=torch.bfloat16, use_graphs: bool = True):
        if model.training:
            raise RuntimeError("InferenceEngine folds the eval-mode BatchNorm statistics: call model.eval() first")
        self.model = model
        self.dtype = backbone_dtype
        self.use_graphs = use_graphs
        self.refolds = 0
        self._fold()

    def _fold(self) -> None:
        """(Re-)fold the BatchNorm statistics into channels_last copies of the conv weights and drop every captured graph: the
        copies, and the packed transformer weights the graphs point at, belong to ONE state of the model's parameters."""
        from .graphs import weights_signature
        model = self.model
        vm = model.video_model.video_model
        self.video = _FoldedResNet(vm.s_former, self.dtype)
        self.audio = _FoldedResNet(model.audio_model.audio_model.resnet, self.dtype)
        self.num_channels = vm.num_channels
        self._graphs: Dict[tuple, tuple] = {}
        self._sig = weights_signature(model)

    # -- eager pieces (the forward below is also what gets captured) --------------------------------------------
    def _audio_tokens_into(self, audio: torch.Tensor, fused: torch.Tensor) -> None:
        """audio [B,1,64,1001]: ResNet-18 trunk -> global average pool -> [B,512] fp32 -> AU_former into columns [0,128) of fused."""
        a = self.audio.to_stage(self.audio.stem_fwd(audio), 1, 4)
        a_feat = a.float().mean(dim=(2, 3))
        self.model.audio_model.au_head.tokens_into(a_feat, a_feat.shape[1], audio.shape[0], out=fused, ld_out=256)

    def _frame_features(self, frames: torch.Tensor) -> torch.Tensor:
        """frames [F,C,H,W] -> stem..stage 3 -> SFormer -> stage 4 -> pool -> [F,512] fp32; every step works frame by frame."""
        vm = self.model.video_model.video_model
        s3 = self.video.to_stage(self.video.stem_fwd(frames), 1, 3)
        s3 = s3.to(torch.bfloat16 if AF._mode(vm.s_former.spatial_transformer.precision or default_precision()) == AF.AVF_BF16 else torch.float32)
        s3 = vm.s_former.sformer(s3.contiguous())                      # NCHW-contiguous map in, same out (models/vformer.py:245-259)
        f = self.video.to_stage(s3.to(self.dtype).contiguous(memory_format=torch.channels_last), 4, 4)
        return f.float().mean(dim=(2, 3))                               # AdaptiveAvgPool2d((1,1)) + flatten

    @torch.no_grad()
    def _forward(self, clip: torch.Tensor, audio: torch.Tensor) -> torch.Tensor:
        m = self.model
        vm = m.video_model.video_model
        bs, _, T, H, W = clip.shape
        fused = torch.empty((bs * 12, 256), dtype=torch.float32, device=clip.device)
        self._audio_tokens_into(audio, fused)
        # video: [B,C,T,H,W] -> frames [B*T,C,H,W] -> per-frame features -> TFormer -> AU_former into columns [128,256)
        frames = clip[:, -self.num_channels:].permute(0, 2, 1, 3, 4).reshape(bs * T, self.num_channels, H, W)
        cls = vm.t_former.cls_features(self._frame_features(frames))
        m.video_model.au_head.tokens_into(cls, cls.shape[1], cls.shape[0], out=fused[:, 128:], ld_out=256)
        if m.task != "AU":
            return torch.zeros(bs, 21, device=clip.device)
        return m.au_head.logits21_(fused, bs)

    def _refresh(self) -> None:
        from .graphs import weights_signature
        if weights_signature(self.model) != self._sig:        # load_state_dict / optimizer.step() / in-place edits since the fold
            if self.model.training:
                raise RuntimeError("InferenceEngine folds the eval-mode BatchNorm statistics: call model.eval() first")
            self.refolds += 1
            self._fold()

    # -- whole videos: each frame through the video trunk once, clips gathered from the frame bank ------------------------
    @torch.no_grad()
    def frame_features(self, frames: torch.Tensor) -> torch.Tensor:
        """frames [F,C,H,W] (C = the model's num_channels) -> frame features [F,512] fp32: the per-frame part of a forward.  The rows of
        one video, concatenated over frame chunks, are the bank that ``clips`` gathers from.  Eager (no graph capture)."""
        AF._cuda(frames, "frames")
        if frames.dim() != 4 or frames.shape[1] != self.num_channels:
            raise ValueError(f"InferenceEngine.frame_features: frames must be [F, {self.num_channels}, H, W], got {tuple(frames.shape)}")
        self._refresh()
        return self._frame_features(frames)

    @torch.no_grad()
    def clips(self, bank: torch.Tensor, index: torch.Tensor, audio_features: torch.Tensor) -> Tuple[torch.Tensor, torch.Tensor]:
        """Clips described by frame indices into ``bank`` (frame_features of one video): index integer [n, T], -1 = a missing frame
        (masked out of the TFormer), audio_features [n,1,64,1001] one mel window per clip.  Returns (out21 [n,21] like model(x),
        decisions [n,12] int32 = out21[:, :12] > 0).  Eager (no graph capture)."""
        AF._cuda(audio_features, "audio_features")
        m = self.model
        if torch.is_tensor(index) and index.dim() == 2 and audio_features.shape[0] != index.shape[0]:
            raise ValueError(f"InferenceEngine.clips: {audio_features.shape[0]} audio windows for {index.shape[0]} clips: one window per clip")
        self._refresh()
        cls = m.video_model.video_model.t_former.cls_features_indexed(bank, index)      # checks the index itself
        n = cls.shape[0]
        fused = torch.empty((n * 12, 256), dtype=torch.float32, device=bank.device)
        self._audio_tokens_into(audio_features, fused)
        m.video_model.au_head.tokens_into(cls, cls.shape[1], n, out=fused[:, 128:], ld_out=256)
        if m.task != "AU":
            return torch.zeros(n, 21, device=bank.device), torch.zeros(n, 12, dtype=torch.int32, device=bank.device)
        return m.au_head.logits21_(fused, n, want_decisions=True)

    def __call__(self, x: Dict[str, torch.Tensor]) -> torch.Tensor:
        clip, audio = x["clip"], x["audio_features"]
        AF._cuda(clip, "x['clip']")
        AF._cuda(audio, "x['audio_features']")
        from .graphs import _packed_refs
        self._refresh()
        if not self.use_graphs:
            return self._forward(clip, audio)
        key = (tuple(clip.shape), clip.dtype, tuple(audio.shape), audio.dtype)
        ent = self._graphs.get(key)
        if ent is None:
            s_clip, s_audio = clip.clone(), audio.clone()
            side = torch.cuda.Stream()
            side.wait_stream(torch.cuda.current_stream())
            with torch.cuda.stream(side):
                for _ in range(2):
                    self._forward(s_clip, s_audio)
            torch.cuda.current_stream().wait_stream(side)
            torch.cuda.synchronize()
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g):
                out = self._forward(s_clip, s_audio)
            ent = self._graphs[key] = (g, s_clip, s_audio, out, _packed_refs(self.model))   # the graph reads the packed weights through raw pointers
        g, s_clip, s_audio, out, _ = ent
        s_clip.copy_(clip, non_blocking=True)
        s_audio.copy_(audio, non_blocking=True)
        g.replay()
        return out
