"""Video branch: ResNet-18 conv stages (plain torch / cuDNN — outside the hot path by design), the
SFormer token region after stage 3 and the TFormer over the clip's frames, with the reference's
constructor signatures and state-dict names (models/vformer.py:128-331).
"""
from __future__ import annotations

import torch
from torch import nn

from . import functional as AF
from .encoder import Transformer, needs_grad


class Dummy(nn.Module):
    """Identity placeholder for a removed classifier (models/avformer.py:21-26)."""

    def forward(self, input):
        return input


class BasicBlock(nn.Module):
    """Two 3x3 conv + BN with identity / 1x1-projection shortcut (standard ResNet-18 block; the
    reference's copy is models/vformer.py:128-165).  cuDNN work, not part of the hot path."""
    expansion = 1

    def __init__(self, inplanes, planes, stride=1, downsample=None, norm_layer=None):
        super().__init__()
        norm_layer = norm_layer or nn.BatchNorm2d
        self.conv1 = nn.Conv2d(inplanes, planes, 3, stride, 1, bias=False)
        self.bn1 = norm_layer(planes)
        self.relu = nn.ReLU(inplace=True)
        self.conv2 = nn.Conv2d(planes, planes, 3, 1, 1, bias=False)
        self.bn2 = norm_layer(planes)
        self.downsample = downsample
        self.stride = stride

    def forward(self, x):
        shortcut = x if self.downsample is None else self.downsample(x)
        y = self.relu(self.bn1(self.conv1(x)))
        y = self.bn2(self.conv2(y))
        return self.relu(y + shortcut)


def _stage(block, inplanes, planes, n_blocks, stride, norm_layer):
    down = None
    if stride != 1 or inplanes != planes * block.expansion:
        down = nn.Sequential(nn.Conv2d(inplanes, planes * block.expansion, 1, stride, bias=False), norm_layer(planes * block.expansion))
    mods = [block(inplanes, planes, stride, down, norm_layer=norm_layer)]
    mods += [block(planes * block.expansion, planes, norm_layer=norm_layer) for _ in range(1, n_blocks)]
    return nn.Sequential(*mods)


class ResFormer(nn.Module):
    """ResNet-18 with the S-Former after stage 3 (models/vformer.py:168-268).

    forward(x[b,t,c,h,w]) -> [b*t, 512].  Lines 245-259 of the reference (NCHW -> tokens, + pos,
    1 encoder layer, tokens -> NCHW) run as one ``avf_sformer_fwd`` call."""

    def __init__(self, block, layers, zero_init_residual=False, groups=1, width_per_group=64, replace_stride_with_dilation=None,
                 norm_layer=None, num_patches=7 * 7, dim=256, depth=1, heads=8, mlp_dim=512, dim_head=32, dropout=0.0):
        super().__init__()
        if groups != 1 or width_per_group != 64 or (replace_stride_with_dilation and any(replace_stride_with_dilation)):
            raise NotImplementedError("ResFormer: only the plain ResNet-18 configuration of the reference is supported")
        norm_layer = norm_layer or nn.BatchNorm2d
        self.conv1 = nn.Conv2d(3, 64, kernel_size=7, stride=2, padding=3, bias=False)
        self.bn1 = norm_layer(64)
        self.relu = nn.ReLU(inplace=True)
        self.maxpool = nn.MaxPool2d(kernel_size=3, stride=2, padding=1)
        self.layer1 = _stage(block, 64, 64, layers[0], 1, norm_layer)
        self.layer2 = _stage(block, 64 * block.expansion, 128, layers[1], 2, norm_layer)
        self.layer3 = _stage(block, 128 * block.expansion, 256, layers[2], 2, norm_layer)
        self.layer4 = _stage(block, 256 * block.expansion, 512, layers[3], 2, norm_layer)
        self.avgpool = nn.AdaptiveAvgPool2d((1, 1))
        self.pos_embedding = nn.Parameter(torch.randn(1, num_patches, dim))
        self.spatial_transformer = Transformer(dim, depth, heads, dim_head, mlp_dim, dropout)
        for m in self.modules():
            if isinstance(m, nn.Conv2d):
                nn.init.kaiming_normal_(m.weight, mode="fan_out", nonlinearity="relu")
            elif isinstance(m, (nn.BatchNorm2d, nn.GroupNorm)):
                nn.init.ones_(m.weight)
                nn.init.zeros_(m.bias)
        if zero_init_residual:
            for m in self.modules():
                if isinstance(m, BasicBlock):
                    nn.init.zeros_(m.bn2.weight)

    def stem_to_stage3(self, frames):
        x = self.maxpool(self.relu(self.bn1(self.conv1(frames))))
        return self.layer3(self.layer2(self.layer1(x)))

    def sformer(self, fmap, out=None):
        """The hot-path region: [F,256,7,7] -> [F,256,7,7] (``out``: optional preallocated destination, inference only)."""
        st = self.spatial_transformer
        n_tok = fmap.shape[2] * fmap.shape[3]
        if n_tok > self.pos_embedding.shape[1]:
            raise ValueError(f"stage-3 map has {n_tok} positions but pos_embedding holds {self.pos_embedding.shape[1]}")
        if needs_grad(st, fmap, self.pos_embedding) or st.dropout_state()[0] > 0.0:
            from .autograd import SFormerFn
            return SFormerFn.apply(fmap, self.pos_embedding, st, *st.param_list())
        return AF.sformer_fwd(fmap, self.pos_embedding[0, :n_tok], st.packed(), st.heads, st.dim_head, st.mlp_dim, out=out)

    def sformer_maps(self, fmap):
        """sformer() kernel by kernel with the attention maps of the spatial transformer: (fmap_out, maps [depth, F, heads, H*W, H*W]);
        fmap_out equals sformer()'s with set_fused_enabled(False) bit for bit (the same pack, layers and unpack launches)."""
        st = self.spatial_transformer
        n_tok = fmap.shape[2] * fmap.shape[3]
        if n_tok > self.pos_embedding.shape[1]:
            raise ValueError(f"stage-3 map has {n_tok} positions but pos_embedding holds {self.pos_embedding.shape[1]}")
        st.check_maps_allowed("ResFormer.sformer_maps", fmap, self.pos_embedding)
        x = AF.sformer_tokens_pack(fmap, self.pos_embedding[0, :n_tok])
        maps = st.maps_(x, fmap.shape[0], n_tok)
        return AF.sformer_tokens_unpack(x, fmap.shape, fmap.dtype), maps

    def forward(self, x, maps: bool = False):
        """x [b,t,c,h,w] -> [b*t, 512]; ``maps``: also return the SFormer's attention maps (sformer_maps)."""
        b, t, c, h, w = x.shape
        fmap = self.stem_to_stage3(x.contiguous().view(-1, c, h, w))
        fmap, smaps = self.sformer_maps(fmap) if maps else (self.sformer(fmap), None)
        feat = torch.flatten(self.avgpool(self.layer4(fmap)), 1)
        return (feat, smaps) if maps else feat


class SFormerBlock(nn.Module):
    """The spatial-transformer region alone, for any channel width: pos_embedding[1, num_patches, dim] + Transformer over the
    H*W positions of an NCHW map, transposed back (models/vformer.py:245-259).  ResFormer above is the dim-256 instantiation on the hot
    path; VGGFormer (models/vggformer.py:250-258: num_patches 49, dim 512, depth 1, 8 x 32, mlp 512) is this block behind a VGGFace2
    trunk that is not part of this package.  Inference kernels only."""

    def __init__(self, num_patches=7 * 7, dim=512, depth=1, heads=8, mlp_dim=512, dim_head=32, dropout=0.0):
        super().__init__()
        self.pos_embedding = nn.Parameter(torch.randn(1, num_patches, dim))
        self.spatial_transformer = Transformer(dim, depth, heads, dim_head, mlp_dim, dropout)

    @torch.no_grad()
    def forward(self, fmap, out=None):
        st = self.spatial_transformer
        n_tok = fmap.shape[2] * fmap.shape[3]
        if n_tok > self.pos_embedding.shape[1]:
            raise ValueError(f"map has {n_tok} positions but pos_embedding holds {self.pos_embedding.shape[1]}")
        return AF.sformer_fwd(fmap, self.pos_embedding[0, :n_tok], st.packed(), st.heads, st.dim_head, st.mlp_dim, out=out)


class TFormer(nn.Module):
    """cls + frame tokens -> 3-layer encoder -> cls row (models/vformer.py:270-293).
    ``num_patches`` is the clip length T (the reference hard-wires 16 in VideoModel)."""

    def __init__(self, num_patches=16, dim=512, depth=3, heads=8, mlp_dim=1024, dim_head=64, dropout=0.0):
        super().__init__()
        self.num_patches, self.dim = num_patches, dim
        self.cls_token = nn.Parameter(torch.randn(1, 1, dim))
        self.pos_embedding = nn.Parameter(torch.randn(1, num_patches + 1, dim))
        self.spatial_transformer = Transformer(dim, depth, heads, dim_head, mlp_dim, dropout)

    def _n_clips(self, x) -> int:
        AF._cuda(x, "x")
        if x.numel() % (self.num_patches * self.dim) != 0:
            raise ValueError(f"TFormer(num_patches={self.num_patches}): input of {tuple(x.shape)} is not a whole number of clips")
        return x.numel() // (self.num_patches * self.dim)

    def tokens(self, x, mask=None):
        """Embedded + encoded tokens [n_clips*(T+1), dim] (fp32) and n_clips; the cls rows are rows c*(T+1).  ``mask`` (optional):
        frames kept, bool [n_clips, T] (True = a real frame), the attention mask of every layer (Transformer.forward)."""
        n_clips = self._n_clips(x)
        keep = None if mask is None else AF.keep_from_mask(mask, n_clips, self.num_patches + 1)
        if needs_grad(self, x):
            from .autograd import TFormerEmbedFn
            tok = TFormerEmbedFn.apply(x, self.cls_token, self.pos_embedding, self.num_patches)
            return self.spatial_transformer.forward_train(tok, n_clips, self.num_patches + 1, keep), n_clips
        tok = AF.tformer_embed(x.detach(), self.cls_token.view(-1), self.pos_embedding[0], self.num_patches)
        self.spatial_transformer.forward_(tok, n_clips, self.num_patches + 1, keep=keep)
        return tok, n_clips

    def cls_features(self, x, mask=None):
        """Inference: cls features [n_clips, dim] fp32 in one library call; the last layer runs its post-softmax part on the cls rows
        only (the other rows never leave the module, models/vformer.py:290).  ``mask``: frames kept, as in tokens()."""
        n_clips = self._n_clips(x)
        st = self.spatial_transformer
        if st.dropout_state()[0] > 0.0:                 # train() with dropout: the tape-keeping kernels apply it
            tok, _ = self.tokens(x, mask)
            return AF.tformer_cls_extract(tok, n_clips, self.num_patches + 1)
        keep = None if mask is None else AF.keep_from_mask(mask, n_clips, self.num_patches + 1)
        return AF.tformer_fwd(x.detach(), self.cls_token.view(-1), self.pos_embedding[0], st.packed(), st.shape(n_clips, self.num_patches + 1),
                              keep)

    def cls_features_indexed(self, bank, index):
        """Inference on clips described by frame indices: cls features [n_clips, dim] fp32, equal to
        ``cls_features(bank[index.clamp(min=0)].reshape(-1, dim), mask=index >= 0)`` without the gathered copy (gather, mask and embed
        are one launch).  ``bank`` [n_bank, dim] fp32 / bf16 on CUDA: the frame features of one video, each frame computed once.
        ``index`` integer [n_clips, num_patches], on the host or the bank's device; -1 = a missing frame (masked out of every layer)."""
        AF._cuda(bank, "bank")
        st = self.spatial_transformer
        if st.dropout_state()[0] > 0.0:
            raise RuntimeError("TFormer.cls_features_indexed is inference only: this TFormer applies dropout (train() with dropout > 0), which "
                               "only the tape-keeping kernels of cls_features implement; call eval() first")
        return self._cls_indexed(bank, self.bank_index(bank.shape, bank.device, index, "cls_features_indexed"))

    def _cls_indexed(self, bank, index_i32):
        st = self.spatial_transformer
        return AF.tformer_fwd_indexed(bank.detach(), index_i32, self.cls_token.view(-1), self.pos_embedding[0], st.packed(),
                                      st.shape(index_i32.shape[0], self.num_patches + 1))

    def forward_indexed(self, bank, index):
        """forward() on clips described by frame indices: cls features [n_clips, dim], equal bit for bit to
        ``self(bank[index.clamp(min=0)].reshape(-1, dim), mask=index >= 0)`` -- with autograd, dropout and the bank's gradient -- without
        the gathered copy.  The bank's gradient sums the token gradients of every clip slot that points at a frame (ascending slot order,
        bit-reproducible), so each frame costs one backward of whatever computed the bank.  ``bank`` / ``index`` as in
        cls_features_indexed, with the same errors.  Without anything to differentiate and without dropout this is cls_features_indexed."""
        AF._cuda(bank, "bank")
        return self.forward_indexed_checked(bank, self.bank_index(bank.shape, bank.device, index, "forward_indexed"))

    def forward_indexed_checked(self, bank, index_i32):
        """forward_indexed() on an index that bank_index() returned."""
        st = self.spatial_transformer
        if not (needs_grad(self, bank) or (st.training and st.dropout > 0.0)):      # not dropout_state(): it draws the dropout seed
            return self._cls_indexed(bank, index_i32)
        from .autograd import TFormerEmbedIndexedFn
        n_clips, T = index_i32.shape[0], self.num_patches
        tok, keep = TFormerEmbedIndexedFn.apply(bank, index_i32, self.cls_token, self.pos_embedding, T)
        tok = st.forward_train(tok, n_clips, T + 1, keep)
        return tok.view(n_clips, T + 1, self.dim)[:, 0]                      # cls rows (a view: data movement only)

    def bank_index(self, bank_shape, device, index, who):
        """The checks of a bank of shape ``bank_shape`` on ``device`` and its clip table, shared by the indexed entry points (error
        messages name ``who``) -> the index as a contiguous int32 tensor on that device.  Runs no library kernel, so a caller can check
        the table before it computes the bank."""
        if len(bank_shape) != 2 or bank_shape[1] != self.dim:
            raise ValueError(f"TFormer.{who}: bank must be [n_bank, {self.dim}], got {tuple(bank_shape)}")
        if not torch.is_tensor(index):
            raise TypeError(f"TFormer.{who}: index must be an integer tensor, got {type(index).__name__}")
        if index.dtype.is_floating_point or index.dtype.is_complex or index.dtype == torch.bool:
            raise TypeError(f"TFormer.{who}: index must be an integer tensor, got {index.dtype}")
        if index.dim() != 2 or index.shape[0] == 0 or index.shape[1] != self.num_patches:
            raise ValueError(f"TFormer.{who}: index must be [n_clips, {self.num_patches}] (num_patches frames per clip), got "
                             f"{tuple(index.shape)}")
        # Checked where the table lives: on the host for free, on the device at the cost of one stream synchronisation.  While a graph
        # is captured neither that synchronisation nor a host-to-device copy is possible: the index must already be on the device, and
        # the kernel's bounds guard alone holds.
        if torch.cuda.is_current_stream_capturing():
            if not index.is_cuda:
                raise RuntimeError(f"TFormer.{who}: while a CUDA graph is being captured the index must already be on the "
                                   f"bank's device ({device}); it is on {index.device}")
        else:
            lo, hi = (int(v) for v in torch.aminmax(index))
            if lo < -1 or hi >= bank_shape[0]:
                raise ValueError(f"TFormer.{who}: index entries must lie in [-1, {bank_shape[0]}) (-1 = missing frame), got "
                                 f"[{lo}, {hi}]")
        return index.to(device=device, dtype=torch.int32).contiguous()

    def attention_maps(self, x, mask=None):
        """(cls, maps): cls equals ``cls_features(x, mask)`` bit for bit and maps fp32 [depth, n_clips, heads, T+1, T+1] holds the
        softmax probabilities of every layer; the last layer's attention runs every query row, so its map is full (which frames and
        which frames' tokens each token attended to).  Inference only: RuntimeError under autograd or in train() with dropout > 0."""
        n_clips = self._n_clips(x)
        st = self.spatial_transformer
        st.check_maps_allowed("TFormer.attention_maps", x, self.cls_token, self.pos_embedding)
        keep = None if mask is None else AF.keep_from_mask(mask, n_clips, self.num_patches + 1)
        return AF.tformer_fwd_probs(x.detach(), self.cls_token.view(-1), self.pos_embedding[0], st.packed(), st.shape(n_clips, self.num_patches + 1),
                                    keep)

    def attention_maps_indexed(self, bank, index):
        """attention_maps on clips described by frame indices, bit for bit ``attention_maps(bank[index.clamp(min=0)].reshape(-1, dim),
        mask=index >= 0)`` without the gathered copy.  ``bank`` / ``index`` as in cls_features_indexed, with the same checks and errors.
        Whole videos: ``eng.frame_features`` for the bank, then this call with the clips' index table."""
        AF._cuda(bank, "bank")
        st = self.spatial_transformer
        st.check_maps_allowed("TFormer.attention_maps_indexed", bank, self.cls_token, self.pos_embedding)
        index = self.bank_index(bank.shape, bank.device, index, "attention_maps_indexed")
        return AF.tformer_fwd_indexed_probs(bank.detach(), index, self.cls_token.view(-1), self.pos_embedding[0], st.packed(),
                                            st.shape(index.shape[0], self.num_patches + 1))

    def relevance_fwd_(self, x, keep=None):
        """The tape-keeping forward of forward() with autograd, without recording: (tokens [n_clips*(T+1), dim], tape, n_clips) for
        relevance_bwd_; the cls rows c*(T+1) of the tokens are forward()'s output bit for bit."""
        n_clips = self._n_clips(x)
        tok = AF.tformer_embed(x.detach(), self.cls_token.detach().reshape(-1), self.pos_embedding.detach()[0], self.num_patches)
        y, tape = self.spatial_transformer.relevance_fwd_(tok, n_clips, self.num_patches + 1, keep)
        return y, tape, n_clips

    def relevance_bwd_(self, tape, n_clips, d_cls, keep=None, maps=True):
        """Backward of relevance_fwd_ seeded with d_cls [n_clips, dim] on the cls rows: (dtok [n_clips*(T+1), dim] = the gradient wrt
        the embedded tokens, gradient maps [depth, n_clips, heads, T+1, T+1] or None)."""
        T1 = self.num_patches + 1
        dtok = torch.zeros((n_clips * T1, self.dim), dtype=torch.float32, device=d_cls.device)
        dtok.view(n_clips, T1, self.dim)[:, 0] = d_cls
        gmaps = self.spatial_transformer.relevance_bwd_(dtok, tape, n_clips, T1, keep, maps)
        return dtok, gmaps

    def attention_relevance(self, frame_feat, d_cls, mask=None):
        """(cls, gmaps, R) for the target whose gradient wrt the cls features is ``d_cls`` [n_clips, dim]: cls equals forward()'s with
        autograd bit for bit (the tape-keeping kernels), gmaps fp32 [depth, n_clips, heads, T+1, T+1] are the gradient maps
        G = P o dP of every layer (the last one full: the tape path runs every row) and R fp32 [n_clips, T+1, T+1] their rollout;
        R[:, 0, 1:] is the relevance of each frame for the cls token.  ``mask``: frames kept, as in forward().  No parameter gradient
        is computed or changed.  RuntimeError in train()."""
        n_clips = self._n_clips(frame_feat)
        AF._cuda(d_cls, "d_cls")
        self.spatial_transformer.check_relevance_allowed("TFormer.attention_relevance")
        if tuple(d_cls.shape) != (n_clips, self.dim):
            raise ValueError(f"TFormer.attention_relevance: d_cls must be [{n_clips}, {self.dim}], got {tuple(d_cls.shape)}")
        keep = None if mask is None else AF.keep_from_mask(mask, n_clips, self.num_patches + 1)
        with torch.no_grad():
            y, tape, _ = self.relevance_fwd_(frame_feat, keep)
            _, gmaps = self.relevance_bwd_(tape, n_clips, d_cls.detach().float(), keep)
            cls = y.view(n_clips, self.num_patches + 1, self.dim)[:, 0].contiguous()
            return cls, gmaps, AF.attention_rollout(gmaps)

    def forward(self, x, mask=None):
        """x [n_clips*T, dim] frame features -> cls features [n_clips, dim].  ``mask`` (optional): bool [n_clips, T], True = a real
        frame; clips with fewer real frames can share a batch with full ones (the padding frames' values do not matter)."""
        if needs_grad(self, x):
            tok, n_clips = self.tokens(x, mask)
            return tok.view(n_clips, self.num_patches + 1, self.dim)[:, 0]          # cls rows (a view: data movement only)
        return self.cls_features(x, mask)


class VideoModel(nn.Module):
    """models/vformer.py:295-331."""

    def __init__(self):
        super().__init__()
        self.s_former = ResFormer(BasicBlock, [2, 2, 2, 2])
        self.t_former = TFormer()
        self.fc = nn.Linear(in_features=512, out_features=7)
        self.num_channels = 3

    def forward(self, x):
        x = x[:, -self.num_channels:].permute(0, 2, 1, 3, 4)        # [B,C,T,H,W] -> [B,T,C,H,W]
        return self.fc(self.t_former(self.s_former(x)))

    def config_modality(self, modality="A;V;M"):
        if "M" not in modality:
            return
        self.num_channels = 4 if "V" in modality else 1
        old = self.s_former.conv1
        new = nn.Conv2d(self.num_channels, old.out_channels, old.kernel_size, old.stride, old.padding, bias=False)
        if "V" in modality:
            with torch.no_grad():
                new.weight[:, 0:3] = old.weight
        self.s_former.conv1 = new
