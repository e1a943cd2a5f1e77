"""DPT-Hybrid-384 (`vitb_rn50_384`) dense-prediction model, B200-native.

Drop-in for the reference's `modules/midas/dpt_depth.py::DPTDepthModel` (constructor kwargs,
`state_dict()` keys / shapes / order, `forward(x)` contract: float NCHW in, `[B,H,W]` (1 channel)
or `[B,C,H,W]` out, final ReLU when `non_negative`).  The arithmetic runs in the sm_100a kernels
of `omnidata_b200/csrc` through the C ABI (`include/omnidata_b200.h`); this file is host-side
orchestration only: weight pre-packing at load time, workspace management, launch order and
optional CUDA-graph replay.  There is no CPU / eager fallback — `forward` on a CPU tensor raises.

Reference call stack mirrored here (omnidata_tools/torch/): DPT.forward `modules/midas/dpt_depth.py:67-85`,
forward_vit / forward_flex `modules/midas/vit.py:61-155`, reassemble `vit.py:431-462`,
FeatureFusionBlock_custom / ResidualConvUnit_custom `modules/midas/blocks.py:231-341`,
head `dpt_depth.py:91-99`; encoder arithmetic is timm 0.4.12 `vit_base_resnet50_384` (`vit.py:483`).
"""
from __future__ import annotations

import math
from typing import Dict, List, Optional, Tuple

import torch
import torch.nn as nn
import torch.nn.functional as F

from . import bwd, ops
from ._capi import OdbError

_STAGES = ((256, 3), (512, 4), (1024, 9))   # timm ResNetV2(layers=(3,4,9)) widths / depths
_FEATURES = 256
_HYBRID_MAX_W = 1792    # widest input the ResNetV2 stem's im2col kernel stages (odb_stem_im2col)
# Encoders behind the same decoder (modules/midas/blocks.py:12-47 _make_encoder, dpt_depth.py:41-45 hooks):
#   vitb_rn50_384  DPT-Hybrid: ResNetV2 stages 0/1 give layer_1/2, ViT-B blocks 8/11 give layer_3/4
#   vitl16_384     DPT-Large (SURVEY 8(f) rank 3): plain ViT-L/16, blocks 5/11/17/23 give layer_1..4
#                  (vit.py:185-290: conv1x1 then ConvTranspose 4x4/s4, 2x2/s2, identity, conv3x3/s2)
_ARCH = {
    "vitb_rn50_384": dict(embed=768, heads=12, depth=12, hybrid=True, hooks=(8, 11), rn_in=(256, 512, 768, 768)),
    "vitl16_384": dict(embed=1024, heads=16, depth=24, hybrid=False, hooks=(5, 11, 17, 23),
                       rn_in=(256, 512, 1024, 1024)),
    #   vitb16_384   plain ViT-B/16, blocks 2/5/8/11, reassemble widths 96/192/384/768 (vit.py:311-318); the 96
    #                channels are carried zero-padded to 128 internally (the GEMM N tile is a multiple of 64)
    "vitb16_384": dict(embed=768, heads=12, depth=12, hybrid=False, hooks=(2, 5, 8, 11),
                       rn_in=(96, 192, 384, 768)),
}


def _pad_to(t: torch.Tensor, dim: int, size: int) -> torch.Tensor:
    """zero-pad `t` along `dim` up to `size` (weights / biases of layers whose width is not a multiple of 64)."""
    if t.shape[dim] == size:
        return t
    shape = list(t.shape)
    shape[dim] = size - t.shape[dim]
    return torch.cat([t, torch.zeros(shape, dtype=t.dtype, device=t.device)], dim=dim)
_EMBED, _HEADS, _DEPTH, _HOOKS = 768, 12, 12, (8, 11)      # the DPT-Hybrid values (module-level names kept)


def _decoder_spec(add, num_channels: int, features: int, rn_in) -> None:
    for n, c in zip((1, 2, 3, 4), rn_in):
        add(f"scratch.layer{n}_rn.weight", features, c, 3, 3)
    for n in (1, 2, 3, 4):
        p = f"scratch.refinenet{n}."
        add(p + "out_conv.weight", features, features, 1, 1)
        add(p + "out_conv.bias", features)
        for u in (1, 2):                     # refinenet4.resConfUnit1 is dead (blocks.py:328-330)
            for cv in (1, 2):
                add(f"{p}resConfUnit{u}.conv{cv}.weight", features, features, 3, 3)
                add(f"{p}resConfUnit{u}.conv{cv}.bias", features)
    add("scratch.output_conv.0.weight", features // 2, features, 3, 3)
    add("scratch.output_conv.0.bias", features // 2)
    add("scratch.output_conv.2.weight", 32, features // 2, 3, 3)
    add("scratch.output_conv.2.bias", 32)
    add("scratch.output_conv.4.weight", num_channels, 32, 1, 1)
    add("scratch.output_conv.4.bias", num_channels)


def _vit_blocks_spec(add, pm: str, embed: int, depth: int) -> None:
    for i in range(depth):
        p = f"{pm}blocks.{i}."
        add(p + "norm1.weight", embed)
        add(p + "norm1.bias", embed)
        add(p + "attn.qkv.weight", 3 * embed, embed)
        add(p + "attn.qkv.bias", 3 * embed)
        add(p + "attn.proj.weight", embed, embed)
        add(p + "attn.proj.bias", embed)
        add(p + "norm2.weight", embed)
        add(p + "norm2.bias", embed)
        add(p + "mlp.fc1.weight", 4 * embed, embed)
        add(p + "mlp.fc1.bias", 4 * embed)
        add(p + "mlp.fc2.weight", embed, 4 * embed)
        add(p + "mlp.fc2.bias", embed)
    add(pm + "norm.weight", embed)           # dead in the reference forward (vit.py:153) but present
    add(pm + "norm.bias", embed)
    add(pm + "head.weight", 1000, embed)     # dead: ImageNet classifier of the timm model
    add(pm + "head.bias", 1000)


def _plain_vit_spec(num_channels: int, features: int, arch: dict) -> List[Tuple[str, Tuple[int, ...]]]:
    """DPT with a plain ViT encoder (`vitl16_384`): keys of the reference class instantiated with timm's
    vit_large_patch16_384 (vit.py:185-318), verified against it in tests/test_boundary_cpu.py."""
    spec: List[Tuple[str, Tuple[int, ...]]] = []

    def add(key, *shape):
        spec.append((key, tuple(shape)))

    D = arch["embed"]
    pm = "pretrained.model."
    add(pm + "cls_token", 1, 1, D)
    add(pm + "pos_embed", 1, 577, D)
    add(pm + "patch_embed.proj.weight", D, 3, 16, 16)
    add(pm + "patch_embed.proj.bias", D)
    _vit_blocks_spec(add, pm, D, arch["depth"])
    for n, c in zip((1, 2, 3, 4), arch["rn_in"]):
        p = f"pretrained.act_postprocess{n}."
        add(p + "0.project.0.weight", D, 2 * D)
        add(p + "0.project.0.bias", D)
        add(p + "3.weight", c, D, 1, 1)
        add(p + "3.bias", c)
        if n == 1:
            add(p + "4.weight", c, c, 4, 4)      # ConvTranspose2d(c, c, 4, stride 4): [in, out, kh, kw]
            add(p + "4.bias", c)
        elif n == 2:
            add(p + "4.weight", c, c, 2, 2)      # ConvTranspose2d(c, c, 2, stride 2)
            add(p + "4.bias", c)
        elif n == 4:
            add(p + "4.weight", c, c, 3, 3)      # Conv2d(c, c, 3, stride 2, padding 1)
            add(p + "4.bias", c)
    _decoder_spec(add, num_channels, features, arch["rn_in"])
    return spec


def state_dict_spec(num_channels: int = 1, features: int = _FEATURES,
                    backbone: str = "vitb_rn50_384") -> List[Tuple[str, Tuple[int, ...]]]:
    """(key, shape) in reference `state_dict()` order (SURVEY.md Appendix B; verified against the
    unmodified reference class in tests/test_boundary_cpu.py)."""
    if not _ARCH[backbone]["hybrid"]:
        return _plain_vit_spec(num_channels, features, _ARCH[backbone])
    spec: List[Tuple[str, Tuple[int, ...]]] = []

    def add(key, *shape):
        spec.append((key, tuple(shape)))

    pm = "pretrained.model."
    add(pm + "cls_token", 1, 1, _EMBED)
    add(pm + "pos_embed", 1, 577, _EMBED)
    bb = pm + "patch_embed.backbone."
    add(bb + "stem.conv.weight", 64, 3, 7, 7)
    add(bb + "stem.norm.weight", 64)
    add(bb + "stem.norm.bias", 64)
    cin = 64
    for s, (cout, depth) in enumerate(_STAGES):
        mid = cout // 4
        for b in range(depth):
            p = f"{bb}stages.{s}.blocks.{b}."
            if b == 0:
                add(p + "downsample.conv.weight", cout, cin, 1, 1)
                add(p + "downsample.norm.weight", cout)
                add(p + "downsample.norm.bias", cout)
            add(p + "conv1.weight", mid, cin if b == 0 else cout, 1, 1)
            add(p + "norm1.weight", mid)
            add(p + "norm1.bias", mid)
            add(p + "conv2.weight", mid, mid, 3, 3)
            add(p + "norm2.weight", mid)
            add(p + "norm2.bias", mid)
            add(p + "conv3.weight", cout, mid, 1, 1)
            add(p + "norm3.weight", cout)
            add(p + "norm3.bias", cout)
        cin = cout
    add(pm + "patch_embed.proj.weight", _EMBED, 1024, 1, 1)
    add(pm + "patch_embed.proj.bias", _EMBED)
    _vit_blocks_spec(add, pm, _EMBED, _DEPTH)
    for n in (3, 4):
        p = f"pretrained.act_postprocess{n}."
        add(p + "0.project.0.weight", _EMBED, 2 * _EMBED)
        add(p + "0.project.0.bias", _EMBED)
        add(p + "3.weight", _EMBED, _EMBED, 1, 1)
        add(p + "3.bias", _EMBED)
        if n == 4:
            add(p + "4.weight", _EMBED, _EMBED, 3, 3)
            add(p + "4.bias", _EMBED)
    _decoder_spec(add, num_channels, features, (256, 512, _EMBED, _EMBED))
    return spec


def _std_weight(w: torch.Tensor, eps: float = 1e-8) -> torch.Tensor:
    """timm StdConv2dSame weight standardisation, folded offline for inference."""
    std, mean = torch.std_mean(w.float(), dim=[1, 2, 3], keepdim=True, unbiased=False)
    return (w.float() - mean) / (std + eps)


class _Workspace:
    """Named device buffers, allocated once and reused every forward; a name asked for with another shape (a tuple or
    torch.Size) or dtype gets a new buffer."""

    def __init__(self, device):
        self.device = device
        # name -> (buffer, shape, dtype) as requested: comparing those costs less host time than reading t.shape
        self._bufs: Dict[str, tuple] = {}

    def get(self, name: str, shape, dtype=torch.bfloat16, zero: bool = False) -> torch.Tensor:
        e = self._bufs.get(name)
        if e is None or e[1] != shape or e[2] is not dtype:
            alloc = torch.zeros if zero else torch.empty
            e = self._bufs[name] = (alloc(shape, device=self.device, dtype=dtype), shape, dtype)
        return e[0]


class DPTDepthModel(nn.Module):
    """B200-native DPT-Hybrid; same constructor as the reference (`dpt_depth.py:27-35,88`)."""

    def __init__(self, path: Optional[str] = None, non_negative: bool = True, num_channels: int = 1,
                 backbone: str = "vitb_rn50_384", features: int = 256, readout: str = "project",
                 channels_last: bool = False, use_bn: bool = False, **kwargs):
        super().__init__()
        if backbone not in _ARCH:
            # reference: print + assert False (modules/midas/blocks.py:42-44)
            print(f"Backbone '{backbone}' not implemented")
            raise AssertionError(f"Backbone '{backbone}' not implemented")
        self.backbone = backbone
        self.arch = _ARCH[backbone]
        self._rn_pad = tuple((c + 63) // 64 * 64 for c in self.arch["rn_in"])
        if features != 256 or readout != "project" or use_bn:
            raise NotImplementedError("only features=256, readout='project', use_bn=False (the Omnidata DPT-Hybrid)")
        self.non_negative = bool(non_negative)
        self.num_channels = int(num_channels)
        self.channels_last = channels_last        # a no-op in the reference as well (dpt_depth.py:68-69)
        self.use_cuda_graph = False
        self.keep_taps = False                    # tests: keep named intermediate activations
        self.taps: Dict[str, torch.Tensor] = {}
        # "bf16": tcgen05 tensor-core path (bf16 operands / storage, fp32 accumulation, fp32 ViT residual stream);
        # "fp32": correctness mode — every operand and activation fp32, contractions on the FP32 pipe with fp64
        #         combination of partial sums (the reference is fp32-only: requirements.txt:4, no autocast anywhere)
        self._precision = "bf16"
        self._packed = None
        self._packed_sig = None
        self._workspaces: Dict[Tuple[int, int, int], _Workspace] = {}
        self._graphs: Dict[Tuple[int, int, int], tuple] = {}
        self._build_parameters()
        self.register_load_state_dict_post_hook(lambda module, incompatible: module._invalidate())
        if path is not None:
            self.load(path)

    # ------------------------------------------------------------------ parameters / state_dict
    def _build_parameters(self):
        gen = torch.Generator().manual_seed(0)
        for key, shape in state_dict_spec(self.num_channels, backbone=self.backbone):
            *path, leaf = key.split(".")
            mod = self
            for name in path:
                child = mod._modules.get(name)
                if child is None:
                    child = nn.Module()
                    mod.add_module(name, child)
                mod = child
            if key.endswith("cls_token") or key.endswith("pos_embed"):
                t = torch.randn(shape, generator=gen) * 0.02
            elif leaf == "bias":
                t = torch.zeros(shape)
            elif len(shape) == 1:
                t = torch.ones(shape)
            else:
                fan_in = math.prod(shape[1:])
                t = torch.randn(shape, generator=gen) / math.sqrt(fan_in)
            mod.register_parameter(leaf, nn.Parameter(t))

    def load(self, path: str):
        """reference BaseModel.load (modules/midas/base_model.py:5-16)."""
        parameters = torch.load(path, map_location=torch.device("cpu"))
        if "optimizer" in parameters:
            parameters = parameters["model"]
        self.load_state_dict(parameters)

    @property
    def precision(self) -> str:
        return self._precision

    @precision.setter
    def precision(self, value: str):
        if value not in ("bf16", "fp32"):
            raise ValueError("precision must be 'bf16' or 'fp32'")
        if value != self._precision:
            self._precision = value
            self._invalidate()
            self._workspaces.clear()

    def _invalidate(self):
        self._packed = None
        self._packed_sig = None
        self._graphs.clear()

    def refresh_weights(self):
        """Re-derive the packed kernel weights (and drop captured CUDA graphs) after the parameters changed.
        `forward` also detects in-place updates by itself (parameter version counters and storage pointers)."""
        self._invalidate()

    def _weights_signature(self):
        # in-place updates (optimizer steps on a flat buffer, broadcast copy_, EMA) bump `_version`;
        # re-pointed storage (flatten_parameters, .data = ...) changes `data_ptr`
        sig = 0
        for p in self.parameters():
            sig = (sig * 1000003 + p._version * 31 + p.data_ptr()) & 0xFFFFFFFFFFFFFFFF
        return sig

    def _apply(self, fn, *args, **kwargs):
        out = super()._apply(fn, *args, **kwargs)
        self._invalidate()
        self._workspaces.clear()
        return out

    # ------------------------------------------------------------------ weight pre-pack (one-time)
    @torch.no_grad()
    def _prepack(self, device) -> dict:
        sd = {k: v.detach().to(device) for k, v in self.state_dict().items()}
        f32 = lambda k: sd[k].float().clone().contiguous()      # own storage: packed state never aliases a parameter
        wdt = torch.float32 if self._precision == "fp32" else torch.bfloat16
        bf = lambda t: t.to(wdt).contiguous()                      # operand storage type of the GEMM weights
        _pack = ops.pack_conv_weight
        pack_w = lambda w: _pack(w, wdt)
        pk: dict = {}
        pm = "pretrained.model."
        D, depth = self.arch["embed"], self.arch["depth"]
        if self.arch["hybrid"]:
            bb = pm + "patch_embed.backbone."
            # stem 7x7: [64,3,7,7] -> [64, (ky,kx,c)=147] padded to 160 columns
            w = _std_weight(sd[bb + "stem.conv.weight"]).permute(0, 2, 3, 1).reshape(64, 147)
            pk["stem_w"] = bf(F.pad(w, (0, 13)))
            pk["stem_g"], pk["stem_b"] = f32(bb + "stem.norm.weight"), f32(bb + "stem.norm.bias")
            blocks = []
            for s, (cout, dep) in enumerate(_STAGES):
                for b in range(dep):
                    p = f"{bb}stages.{s}.blocks.{b}."
                    e = {"stride": 2 if (b == 0 and s > 0) else 1, "cout": cout, "mid": cout // 4}
                    if b == 0:
                        e["wd"] = pack_w(_std_weight(sd[p + "downsample.conv.weight"]))
                        e["gd"], e["bd"] = f32(p + "downsample.norm.weight"), f32(p + "downsample.norm.bias")
                    for i in (1, 2, 3):
                        e[f"w{i}"] = pack_w(_std_weight(sd[p + f"conv{i}.weight"]))
                        e[f"g{i}"], e[f"b{i}"] = f32(p + f"norm{i}.weight"), f32(p + f"norm{i}.bias")
                    blocks.append((s, b, e))
            pk["rn_blocks"] = blocks
            pk["proj_w"] = pack_w(sd[pm + "patch_embed.proj.weight"])
        else:
            # PatchEmbed conv [D,3,16,16]: its row-major flattening is the GEMM weight for odb_patchify's columns
            pk["proj_w"] = bf(sd[pm + "patch_embed.proj.weight"].reshape(D, -1))
        pk["proj_b"] = f32(pm + "patch_embed.proj.bias")
        pk["cls"] = f32(pm + "cls_token").reshape(-1)
        pk["pos"] = f32(pm + "pos_embed")                       # [1,577,D] fp32 master copy
        vit = []
        for i in range(depth):
            p = f"{pm}blocks.{i}."
            vit.append({
                "ln1": (f32(p + "norm1.weight"), f32(p + "norm1.bias")),
                "qkv": (bf(sd[p + "attn.qkv.weight"]), f32(p + "attn.qkv.bias")),
                "proj": (bf(sd[p + "attn.proj.weight"]), f32(p + "attn.proj.bias")),
                "ln2": (f32(p + "norm2.weight"), f32(p + "norm2.bias")),
                "fc1": (bf(sd[p + "mlp.fc1.weight"]), f32(p + "mlp.fc1.bias")),
                "fc2": (bf(sd[p + "mlp.fc2.weight"]), f32(p + "mlp.fc2.bias")),
            })
        pk["vit"] = vit
        for n in ((3, 4) if self.arch["hybrid"] else (1, 2, 3, 4)):
            p = f"pretrained.act_postprocess{n}."
            wfull = bf(sd[p + "0.project.0.weight"])               # [D, 2D]
            pk[f"ro{n}_wfull"] = wfull
            pk[f"ro{n}_wtok"] = wfull[:, :D].contiguous()          # token half of the split Linear
            pk[f"ro{n}_b"] = f32(p + "0.project.0.bias")
            cp = self._rn_pad[n - 1]
            pk[f"pp{n}_w"] = pack_w(_pad_to(sd[p + "3.weight"], 0, cp))
            pk[f"pp{n}_b"] = _pad_to(f32(p + "3.bias"), 0, cp)
        pk["pp4s_w"] = pack_w(sd["pretrained.act_postprocess4.4.weight"])
        pk["pp4s_b"] = f32("pretrained.act_postprocess4.4.bias")
        if not self.arch["hybrid"]:
            # ConvTranspose2d(c, c, k, stride k) (vit.py:216-225, 240-249): k*k independent 1x1 convolutions,
            # one per output phase (dy, dx): W_phase[out][in] = weight[in][out][dy][dx]
            for n, k in ((1, 4), (2, 2)):
                cp = self._rn_pad[n - 1]
                w = _pad_to(_pad_to(sd[f"pretrained.act_postprocess{n}.4.weight"].float(), 0, cp), 1, cp)
                pk[f"pp{n}t_w"] = [[bf(w[:, :, dy, dx].t()) for dx in range(k)] for dy in range(k)]
                pk[f"pp{n}t_b"] = _pad_to(f32(f"pretrained.act_postprocess{n}.4.bias"), 0, cp)
        for n in (1, 2, 3, 4):
            pk[f"rn{n}_w"] = pack_w(_pad_to(sd[f"scratch.layer{n}_rn.weight"], 1, self._rn_pad[n - 1]))
            p = f"scratch.refinenet{n}."
            pk[f"ff{n}_out"] = (pack_w(sd[p + "out_conv.weight"]), f32(p + "out_conv.bias"))
            for u in (1, 2):
                pk[f"ff{n}_rcu{u}"] = tuple(
                    (pack_w(sd[f"{p}resConfUnit{u}.conv{cv}.weight"]),
                     f32(f"{p}resConfUnit{u}.conv{cv}.bias")) for cv in (1, 2))
        pk["head0"] = (pack_w(sd["scratch.output_conv.0.weight"]), f32("scratch.output_conv.0.bias"))
        pk["head2"] = (pack_w(sd["scratch.output_conv.2.weight"]), f32("scratch.output_conv.2.bias"))
        pk["head4"] = (sd["scratch.output_conv.4.weight"].float().reshape(self.num_channels, 32).contiguous(),
                       f32("scratch.output_conv.4.bias"))
        pk["pos_cache"] = {}
        return pk

    def _pos_for_grid(self, pk, gh: int, gw: int):
        """(pos0 fp32 [D], grid fp32 [gh*gw, D]); bilinear resize as vit.py:102-116 if needed."""
        key = (gh, gw)
        if key not in pk["pos_cache"]:
            pos = pk["pos"]
            grid = pos[0, 1:]
            if (gh, gw) != (24, 24):
                g = grid.reshape(1, 24, 24, -1).permute(0, 3, 1, 2)
                g = F.interpolate(g, size=(gh, gw), mode="bilinear")
                grid = g.permute(0, 2, 3, 1).reshape(gh * gw, -1)
            pk["pos_cache"][key] = (pos[0, 0].contiguous(), grid.float().contiguous())
        return pk["pos_cache"][key]

    # ------------------------------------------------------------------ forward
    def forward(self, x: torch.Tensor) -> torch.Tensor:
        if not x.is_cuda:
            raise OdbError("omnidata_b200.DPTDepthModel runs on a CUDA (sm_100a) device only; "
                           "there is no CPU fallback — move the model and input to cuda")
        if x.dim() != 4 or x.shape[1] != 3:
            raise ValueError(f"expected input [B,3,H,W], got {tuple(x.shape)}")
        B, _, H, W = x.shape
        if H < 32 or W < 32 or H % 32 or W % 32:
            raise ValueError(f"H and W must be positive multiples of 32, got {H}x{W}")
        if self.arch["hybrid"] and W > _HYBRID_MAX_W:
            raise ValueError(f"the hybrid backbone's stem supports input widths up to {_HYBRID_MAX_W}, got {W}")
        if self.training and torch.is_grad_enabled():
            # train() mode under autograd: the differentiable forward (activations kept for the backward kernels);
            # eval() mode, or any call under torch.no_grad(), is the inference path below and returns a tensor
            # that is not attached to an autograd graph
            return self._forward_autograd(x)
        x = x.detach().float().contiguous()
        sig = self._weights_signature()
        if self._packed is None or sig != self._packed_sig:
            self._invalidate()
            self._packed = self._prepack(x.device)
            self._packed_sig = sig
        if self.use_cuda_graph and not self.keep_taps:
            out = self._forward_graph(x)
        else:
            out = self._forward_impl(x)
        return out.squeeze(dim=1)                     # dpt_depth.py:107

    def _forward_autograd(self, x: torch.Tensor) -> torch.Tensor:
        """Differentiable forward (train_depth.py:183-190 training_step): implemented by omnidata_b200.train."""
        from . import train
        return train.differentiable_forward(self, x)

    def _forward_graph(self, x: torch.Tensor) -> torch.Tensor:
        key = tuple(x.shape[i] for i in (0, 2, 3))
        entry = self._graphs.get(key)
        if entry is None:
            static_in = x.clone()
            side = torch.cuda.Stream()
            side.wait_stream(torch.cuda.current_stream())
            with torch.cuda.stream(side):
                for _ in range(2):                    # warm-up: allocate workspaces, configure kernels
                    self._forward_impl(static_in)
            torch.cuda.current_stream().wait_stream(side)
            graph = torch.cuda.CUDAGraph()
            with torch.cuda.graph(graph):
                static_out = self._forward_impl(static_in)
            entry = (graph, static_in, static_out)
            self._graphs[key] = entry
        graph, static_in, static_out = entry
        static_in.copy_(x)
        graph.replay()
        return static_out.clone()

    @torch.no_grad()
    def _forward_impl(self, x: torch.Tensor) -> torch.Tensor:
        pk = self._packed
        B, _, H, W = x.shape
        key = (B, H, W)
        ws = self._workspaces.get(key)
        if ws is None:
            ws = self._workspaces[key] = _Workspace(x.device)
        taps = self.taps if self.keep_taps else None
        if taps is not None:
            taps.clear()
        gh, gw = H // 16, W // 16
        pos0, pos_grid = self._pos_for_grid(pk, gh, gw)
        pos_b = pk["pos_cache"].get((gh, gw, B))           # derived from the weights: lives with the packed weights
        if pos_b is None:                                  # pos[1:] replicated per image: the GEMM's fp32 residual operand
            pos_b = pk["pos_cache"][(gh, gw, B)] = pos_grid.unsqueeze(0).expand(B, -1, -1).contiguous()
        out = network_forward(pk, x, ws, self.arch, self._precision == "fp32", (pos0, pos_b), self.non_negative, taps=taps)
        if taps is not None:
            self.taps = {k: v.clone() for k, v in taps.items()}
        return out if (self.use_cuda_graph and not self.keep_taps) else out.clone()


def _debug_upsample(z: torch.Tensor) -> torch.Tensor:
    o = torch.empty((z.shape[0], 2 * z.shape[1], 2 * z.shape[2], z.shape[3]), device=z.device, dtype=z.dtype)
    ops.upsample2x_add(z, o)
    return o


def _resnet_features(pk, x, ws, fp32, taps, save):
    """ResNetV2 stem + stages of the hybrid encoder -> (layer_1, layer_2, stage-2 features)."""
    B, _, H, W = x.shape
    adt = torch.float32 if fp32 else torch.bfloat16
    buf = lambda name, shape, dtype=adt: ws.get(name, shape, dtype)
    # ---------------- ResNetV2 stem + stages (timm; hooks at vit.py:363-368)
    h2, w2 = H // 2, W // 2
    n_gn = 1 + sum(3 * d + 1 for _, d in _STAGES)
    stats_pool = buf("gn_stats", (n_gn, B, 32, 2), torch.float32)
    # the kernel leaves it zeroed.  The most it needs is for the stem conv (64 channels at H/2) and stage 0's
    # 256-channel outputs (at H/4), which come to the same size; 4 MiB covers 384x384 up to batch 56
    gn_need = ops.lib().odb_groupnorm_scratch_bytes(B, h2 * w2, 64, 32)
    gn_scratch = ws.get("gn_scratch", (max(4 << 20, gn_need),), torch.uint8, zero=True)
    stat_i = iter(range(n_gn))
    # fused statistics: the conv epilogue writes per-warp partial sums here (largest layer:
    # stage 0 at 96x96 -> 72 tiles x 4 quadrants x 32 groups x 2 per image)
    gn_part = buf("gn_partial", (B * ((H // 4) * (W // 4) // 32 + 64) * 4 * 32 * 2,), torch.float32)

    def conv_stats(fn, *args, out, **kw):
        """conv + GroupNorm statistics of its (unrounded) output.  Tensor-core path: partial sums in the conv
        epilogue + finalize; fp32 mode: the deterministic standalone statistics kernel."""
        st = stats_pool[next(stat_i)]
        if fp32:
            fn(*args, out, **kw)
            ops.groupnorm_stats(out, st, scratch=gn_scratch)
        else:
            fn(*args, out, gn_stats=(gn_part, st), **kw)
        return st

    cols = buf("stem_cols", (B * h2 * w2, 160))
    ops.stem_im2col(x, cols)
    s0 = buf("stem_conv", (B, h2, w2, 64))
    st = conv_stats(ops.conv1x1, cols.view(B, h2, w2, 160), pk["stem_w"], out=s0)
    t = buf("stem_pool", (B, h2 // 2, w2 // 2, 64))
    ops.stem_gn_relu_maxpool(s0, st, pk["stem_g"], pk["stem_b"], t)
    if taps is not None:
        taps["stem_conv"], taps["stem_pool"] = s0, t
    if save is not None:
        save["stem"], save["blocks"] = (cols, s0, st, t), []
    feats = []
    hh, ww = h2 // 2, w2 // 2
    for s, b, e in pk["rn_blocks"]:
        stride, cout, mid = e["stride"], e["cout"], e["mid"]
        ho, wo = hh // stride, ww // stride
        tag = f"s{s}b{b}"
        shortcut, sc_stats = t, None
        if b == 0:
            d = buf(tag + "_ds", (B, ho, wo, cout))
            sc_stats = conv_stats(ops.conv1x1, t[:, ::stride, ::stride, :] if stride > 1 else t, e["wd"], out=d)
            shortcut = d
        y1 = buf(tag + "_y1", (B, hh, ww, mid))
        st1 = conv_stats(ops.conv1x1, t, e["w1"], out=y1)
        a1 = buf(tag + "_a1", (B, hh, ww, mid))
        ops.groupnorm_apply(y1, st1, e["g1"], e["b1"], a1, relu=True)
        y2 = buf(tag + "_y2", (B, ho, wo, mid))
        if stride == 1:
            st2 = conv_stats(ops.conv3x3, a1, e["w2"], out=y2)
        else:
            st2 = conv_stats(lambda a, w_, o, **kw: ops.conv3x3_s2(a, w_, o, "same", **kw), a1, e["w2"], out=y2)
        a2 = buf(tag + "_a2", (B, ho, wo, mid))
        ops.groupnorm_apply(y2, st2, e["g2"], e["b2"], a2, relu=True)
        y3 = buf(tag + "_y3", (B, ho, wo, cout))
        st3 = conv_stats(ops.conv1x1, a2, e["w3"], out=y3)
        out = buf(tag + "_out", (B, ho, wo, cout))
        if b == 0:
            ops.groupnorm_apply(y3, st3, e["g3"], e["b3"], out, relu=True, res=shortcut,
                                res_stats=sc_stats, res_gamma=e["gd"], res_beta=e["bd"])
        else:
            ops.groupnorm_apply(y3, st3, e["g3"], e["b3"], out, relu=True, res=shortcut)
        if save is not None:
            rec = dict(tag=tag, p=f"pretrained.model.patch_embed.backbone.stages.{s}.blocks.{b}.", stride=stride, t_in=t,
                       b=b, s=s, y1=y1, st1=st1, a1=a1, y2=y2, st2=st2, a2=a2, y3=y3, st3=st3, out=out)
            if b == 0:
                rec.update(d=shortcut, std=sc_stats)
            save["blocks"].append(rec)
        t, hh, ww = out, ho, wo
        if taps is not None:
            taps[f"{tag}_out"] = out
        if b == _STAGES[s][1] - 1:
            feats.append(t)
    return feats


def network_forward(pk: dict, x: torch.Tensor, ws: _Workspace, arch: dict, fp32: bool, pos, non_negative: bool,
                    taps: Optional[dict] = None, save: Optional[dict] = None) -> torch.Tensor:
    """One forward of the network: packed weights `pk` (the structure of `DPTDepthModel._prepack`), input x fp32
    [B,3,H,W], activation buffers from `ws`, `arch` an `_ARCH` entry, `fp32` the correctness mode, pos = (pos0 fp32
    [D], pos[1:] fp32 [B, gh*gw, D]).  Returns the output buffer [B,C,H,W] fp32 of `ws`.

    `taps` receives named intermediate activations (tests).  With `save` (DPT-Hybrid only) this is the train-mode
    forward: every activation the backward of omnidata_b200.train reads gets a buffer of its own and is recorded in
    `save`; the MLP GELU, the readout GELU and the head tail keep their inputs."""
    if save is not None and not arch["hybrid"]:
        raise NotImplementedError("the train-mode forward is built for the DPT-Hybrid model (vitb_rn50_384)")
    B, _, H, W = x.shape
    f32 = torch.float32
    adt = f32 if fp32 else torch.bfloat16                       # activation storage type
    buf = lambda name, shape, dtype=adt: ws.get(name, shape, dtype)
    if save is not None:
        save.update(x=x, B=B, H=H, W=W)

    D, heads = arch["embed"], arch["heads"]
    hooks = arch["hooks"]
    if arch["hybrid"]:
        layer_1, layer_2, f3 = _resnet_features(pk, x, ws, fp32, taps, save)
        gh, gw = f3.shape[1], f3.shape[2]
    else:
        gh, gw = H // 16, W // 16
    ntok = gh * gw + 1
    rows = B * ntok
    if save is not None:
        save.update(gh=gh, gw=gw, ntok=ntok, f3=f3)

    # ---------------- tokens: patch proj + cls + pos (vit.py:131-147).  The residual stream is fp32 in BOTH
    # precisions (timm Block.forward adds every branch to an fp32 `x`; SURVEY.md C.1): the proj / fc2 epilogues
    # read and write fp32, LayerNorm reads fp32.
    pos0, pos_b = pos
    if save is None:
        # the residual stream lives in one buffer per hooked block: the block after a hook writes its first
        # residual add into the next buffer, which leaves the hooked activation intact
        tok_bufs = [buf(f"tok_{i}", (B, ntok, D), f32) for i in range(len(hooks))]
        tok = tok_bufs[0]
    else:
        # the stream before every block (xs) and between its two residual adds (xm)
        xs = [buf(f"vit_x{i}", (B, ntok, D), f32) for i in range(len(pk["vit"]) + 1)]
        xm = [buf(f"vit_m{i}", (B, ntok, D), f32) for i in range(len(pk["vit"]))]
        tok = xs[0]
    ops.write_cls_row(tok, pk["cls"], pos0)
    if arch["hybrid"]:
        ops.linear(f3.view(B, 1, gh * gw, 1024), pk["proj_w"], tok[:, 1:, :].unsqueeze(1), bias=pk["proj_b"],
                   residual=pos_b.unsqueeze(1))
    else:
        cols = buf("patch_cols", (B, 1, gh * gw, 3 * 16 * 16))
        ops.patchify(x, cols.view(B * gh * gw, -1), 16)
        ops.linear(cols, pk["proj_w"], tok[:, 1:, :].unsqueeze(1), bias=pk["proj_b"], residual=pos_b.unsqueeze(1))

    if taps is not None:
        taps["tokens_in"] = tok.clone()
    # ---------------- ViT blocks (vit.py:150-151); final norm is dead compute and skipped
    if save is None:                                   # scratch shared by all blocks
        h1 = h2 = buf("vit_h", (B, ntok, D))
        qkv = buf("vit_qkv", (B, ntok, 3 * D))
        att = buf("vit_att", (B, ntok, D))
        mlp = buf("vit_mlp", (B, ntok, 4 * D))
        lse = None
    else:
        vit = []
    cur = tok
    hooked = []
    for i, blk in enumerate(pk["vit"]):
        if save is None:
            x_in = cur
            x_mid = x_out = tok_bufs[len(hooked)] if (i - 1) in hooks else cur
        else:
            x_in, x_mid, x_out = xs[i], xm[i], xs[i + 1]
            h1, h2 = buf(f"vit_h1_{i}", (B, ntok, D)), buf(f"vit_h2_{i}", (B, ntok, D))
            qkv = buf(f"vit_qkv_{i}", (B, ntok, 3 * D))
            att = buf(f"vit_att_{i}", (B, ntok, D))
            lse = None if fp32 else buf(f"vit_lse_{i}", (B, heads, ntok), f32)
            u, mlp = buf(f"vit_u_{i}", (B, ntok, 4 * D)), buf(f"vit_mlp_{i}", (B, ntok, 4 * D))
        ops.layernorm(x_in, blk["ln1"][0], blk["ln1"][1], h1)
        ops.linear(h1.view(rows, -1), blk["qkv"][0], qkv.view(rows, -1), bias=blk["qkv"][1])
        ops.attention(qkv, att, heads=heads, scale=0.125, lse=lse)
        ops.linear(att.view(rows, -1), blk["proj"][0], x_mid.view(rows, -1), bias=blk["proj"][1],
                   residual=x_in.view(rows, -1))
        ops.layernorm(x_mid, blk["ln2"][0], blk["ln2"][1], h2)
        if save is None:
            ops.linear(h2.view(rows, -1), blk["fc1"][0], mlp.view(rows, -1), bias=blk["fc1"][1], act=ops.ACT_GELU)
        elif fp32:                                     # the fp32 conv kernel has no GELU out2
            ops.linear(h2.view(rows, -1), blk["fc1"][0], u.view(rows, -1), bias=blk["fc1"][1])
            bwd.gelu_fwd(u, mlp)
        else:       # one pass: the pre-activation (kept for the backward) and gelu of the same fp32 value
            ops.linear(h2.view(rows, -1), blk["fc1"][0], u.view(rows, -1), bias=blk["fc1"][1],
                       out2=mlp.view(rows, -1), out2_act=ops.ACT_GELU)
        ops.linear(mlp.view(rows, -1), blk["fc2"][0], x_out.view(rows, -1), bias=blk["fc2"][1],
                   residual=x_mid.view(rows, -1))
        cur = x_out
        if i in hooks:
            hooked.append(cur)
        if save is not None:
            vit.append(dict(h1=h1, qkv=qkv, att=att, lse=lse, h2=h2, u=u, mlp=mlp))
        if taps is not None:
            taps[f"tokens_{i}"] = cur.clone()
    if save is not None:
        save.update(xs=xs, xm=xm, vit=vit)

    # ---------------- reassemble (vit.py:66-97, 185-290 / 431-462); outputs carried zero-padded to the GEMM's N
    # granularity
    def readout(tk32, n):
        tk = tk32
        if not fp32:                                   # the hooked activation leaves the fp32 stream as a bf16 operand
            tk = buf(f"ro{n}_tok", (B, ntok, D))
            ops.cast_f32_bf16(tk32, tk)
        cb = buf(f"ro{n}_cb", (B, D), f32)
        ops.readout_cls_bias(pk[f"ro{n}_wfull"], pk[f"ro{n}_b"], tk, cb)
        r = buf(f"ro{n}_r", (B, 1, gh * gw, D))
        if save is None:
            ops.linear(tk[:, 1:, :].unsqueeze(1), pk[f"ro{n}_wtok"], r, bias=cb, bias_per_image=True, act=ops.ACT_GELU)
        else:
            pre = buf(f"ro{n}_pre", (B, 1, gh * gw, D))
            ops.linear(tk[:, 1:, :].unsqueeze(1), pk[f"ro{n}_wtok"], pre, bias=cb, bias_per_image=True)
            bwd.gelu_fwd(pre, r)
        w, bias = pk[f"pp{n}_w"], pk[f"pp{n}_b"]
        o = buf(f"pp{n}", (B, gh, gw, w.shape[0]))
        ops.conv1x1(r.view(B, gh, gw, D), w, o, bias=bias)
        if save is not None:
            save[f"ro{n}"] = dict(tk=tk, tk32=tk32, pre=pre, r=r, o=o)
        return o

    def conv_transpose(t, n, k):
        """ConvTranspose2d(c, c, k, stride k): phase (dy, dx) of the output is a 1x1 convolution of the
        input, stored through a strided view of the output (no scatter kernel)."""
        c = t.shape[3]
        o = buf(f"pp{n}t", (B, gh * k, gw * k, c))
        for dy in range(k):
            for dx in range(k):
                ops.conv1x1(t, pk[f"pp{n}t_w"][dy][dx], o[:, dy::k, dx::k, :], bias=pk[f"pp{n}t_b"])
        return o

    if arch["hybrid"]:
        tokens_8, tokens_11 = hooked
        layer_3 = readout(tokens_8, 3)
        u4 = readout(tokens_11, 4)
    else:
        layer_1 = conv_transpose(readout(hooked[0], 1), 1, 4)
        layer_2 = conv_transpose(readout(hooked[1], 2), 2, 2)
        layer_3 = readout(hooked[2], 3)
        u4 = readout(hooked[3], 4)
    layer_4 = buf("pp4s", (B, gh // 2, gw // 2, pk["pp4s_w"].shape[0]))
    ops.conv3x3_s2(u4, pk["pp4s_w"], layer_4, "sym1", bias=pk["pp4s_b"])

    # ---------------- scratch.layerN_rn (dpt_depth.py:73-76): raw + relu copies feed the RCUs
    rn_raw, rn_relu = [], []
    for n, l in zip((1, 2, 3, 4), (layer_1, layer_2, layer_3, layer_4)):
        shp = (B, l.shape[1], l.shape[2], _FEATURES)
        raw, rl = buf(f"rn{n}_raw", shp), buf(f"rn{n}_relu", shp)
        ops.conv3x3(l, pk[f"rn{n}_w"], raw, out2=rl)
        rn_raw.append(raw)
        rn_relu.append(rl)
    if save is not None:
        save.update(layers=(layer_1, layer_2, layer_3, layer_4), rn_raw=rn_raw, rn_relu=rn_relu)

    # ---------------- RefineNet fusion (dpt_depth.py:78-81; blocks.py:263-341)
    def rcu(n, u, x_raw, x_relu, out, out2=None):
        (w1, b1), (w2, b2) = pk[f"ff{n}_rcu{u}"]
        tmid = buf(f"ff{n}_rcu{u}_t", x_raw.shape)
        ops.conv3x3(x_relu, w1, tmid, bias=b1, act=ops.ACT_RELU)       # relu(conv1(relu(x)))
        ops.conv3x3(tmid, w2, out, bias=b2, residual=x_raw, out2=out2)  # conv2(.) + x
        if save is not None:
            save[f"ff{n}.rcu{u}"] = dict(x_raw=x_raw, x_relu=x_relu, tmid=tmid)

    def fusion_tail(n, s_raw, s_relu):
        """RCU2, then the 1x1 out_conv at the input resolution (it commutes with the bilinear
        upsample: the interpolation weights sum to one)."""
        y = buf(f"ff{n}_y", s_raw.shape)
        rcu(n, 2, s_raw, s_relu, y)
        z = buf(f"ff{n}_z", s_raw.shape)
        w, bias = pk[f"ff{n}_out"]
        ops.conv1x1(y, w, z, bias=bias)
        if save is not None:
            save[f"ff{n}"] = dict(y=y, z=z)
        return z

    z = fusion_tail(4, rn_raw[3], rn_relu[3])
    if taps is not None:
        taps["path_4"] = _debug_upsample(z)
    for n in (3, 2, 1):
        l_raw, l_relu = rn_raw[n - 1], rn_relu[n - 1]
        res = buf(f"ff{n}_res", l_raw.shape)
        rcu(n, 1, l_raw, l_relu, res)
        s_raw, s_relu = buf(f"ff{n}_s", l_raw.shape), buf(f"ff{n}_s_relu", l_raw.shape)
        ops.upsample2x_add(z, s_raw, res=res, out_relu=s_relu)         # up(path) + RCU1(layer_rn)
        z = fusion_tail(n, s_raw, s_relu)
        if taps is not None and n > 1:
            taps[f"path_{n}"] = _debug_upsample(z)
    path_1 = buf("path_1", (B, z.shape[1] * 2, z.shape[2] * 2, _FEATURES))
    ops.upsample2x_add(z, path_1)

    # ---------------- head (dpt_depth.py:91-99)
    w0, b0 = pk["head0"]
    h1 = buf("head_h1", (B, path_1.shape[1], path_1.shape[2], _FEATURES // 2))
    ops.conv3x3(path_1, w0, h1, bias=b0)
    h1u = buf("head_h1u", (B, H, W, _FEATURES // 2))
    ops.upsample2x_add(h1, h1u)
    w2, b2 = pk["head2"]
    w4, b4 = pk["head4"]
    out = buf("out", (B, w4.shape[0], H, W), f32)
    if save is None and not fp32:
        ops.conv3x3(h1u, w2, None, bias=b2, head=(w4, b4, out, non_negative))
    else:
        # the 128 -> 32 conv (+ReLU) on its own (training: carried zero-padded to 64 channels), then the 1x1 conv
        # (+ReLU) to NCHW
        h2 = buf("head_h2", (B, H, W, w2.shape[0]))
        ops.conv3x3(h1u, w2, h2, bias=b2, act=ops.ACT_RELU)
        if save is not None:
            bwd.head_tail_fwd(h2, w4, b4, out, non_negative)
            save["head"] = dict(path_1=path_1, h1=h1, h1u=h1u, a=h2, out=out, w4=w4)
        else:
            pre = buf("head_pre", (B, w4.shape[0], H, W), f32) if taps is not None else None
            ops.head_tail_f32(h2, w4, b4, out, relu=non_negative, pre=pre)
            if taps is not None:
                taps["head_pre_relu"] = pre

    if taps is not None:
        for hk, tk in zip(hooks, hooked):
            taps[f"tokens_{hk}"] = tk
        taps.update(layer_1=layer_1, layer_2=layer_2, layer_3=layer_3, layer_4=layer_4, path_1=path_1,
                    layer_1_rn=rn_raw[0], layer_2_rn=rn_raw[1], layer_3_rn=rn_raw[2],
                    layer_4_rn=rn_raw[3])
    return out
