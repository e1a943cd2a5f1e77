"""Train step of the DPT-Hybrid depth model (train_depth.py:183-190 training_step, :261-279 _shared_step, :381-383 Adam,
:424-426 DDP): differentiable forward + hand-written backward over the kernels of this package.

`TrainEngine(model)` owns flat fp32 parameter / gradient buffers (the model's nn.Parameters become views), re-packs the
GEMM operands from the fp32 master weights every step (odb_pack_weight: cast, ResNetV2 weight standardisation, dgrad
layout), runs the model's forward (`model.network_forward`, the one inference runs) with every activation the backward
needs kept, and the backward:
  * dgrad of every conv / linear layer = odb_conv_gemm with the re-packed (in/out swapped, 180-degree rotated) weight;
    stride-2 convolutions scatter through parity-plane output views;
  * wgrad = odb_conv_wgrad (tcgen05, both operands MN-major straight from the channels-last tensors; fp32 twin);
  * attention backward = odb_attention_bwd; LayerNorm / GroupNorm / GELU / ReLU / bilinear / max-pool / head backward and
    bias gradients = the kernels of csrc/bwd_ops.cu.
`precision="fp32"` runs the same orchestration on the FP32-pipe twins: the mode the gradient-parity tests use against
torch.autograd of the reference arithmetic.  `differentiable_forward(model, x)` wraps the engine in a
torch.autograd.Function so that `loss(model(x)).backward()` fills `p.grad` like the reference module would.
"""
from __future__ import annotations

from typing import Dict, List, Optional, Tuple

import numpy as np
import torch

from . import bwd, ops
from ._capi import OdbError
from .model import _STAGES, DPTDepthModel, _Workspace, network_forward


def _parity_dgrad_plan(mode: str):
    """Stride-2 3x3 convolution, gradient w.r.t. the input: for input parity plane (py, px) the list of
    (tap index t = ky*3+kx, dy, dx): dX[2p + py, 2q + px] += W_t^T dY[p + dy, q + dx]."""
    def axis(par):
        if mode == "same":          # i = 2o + k
            return [(0, 0), (2, -1)] if par == 0 else [(1, 0)]
        if mode == "sym1":          # i = 2o + k - 1
            return [(1, 0)] if par == 0 else [(0, 1), (2, 0)]
        raise ValueError(mode)
    plan = {}
    for py in (0, 1):
        for px in (0, 1):
            plan[(py, px)] = [(ky * 3 + kx, dy, dx) for ky, dy in axis(py) for kx, dx in axis(px)]
    return plan


class TrainEngine:
    def __init__(self, model: DPTDepthModel, precision: str = "bf16"):
        if model.backbone != "vitb_rn50_384":
            raise NotImplementedError("the train step is built for the DPT-Hybrid depth / normal model (vitb_rn50_384)")
        if precision not in ("bf16", "fp32"):
            raise ValueError("precision must be 'bf16' or 'fp32'")
        self.model = model
        self.fp32 = precision == "fp32"
        self.adt = torch.float32 if self.fp32 else torch.bfloat16
        p0 = next(model.parameters())
        if not p0.is_cuda:
            raise OdbError("TrainEngine: the model must live on a CUDA device (no CPU path)")
        self.device = p0.device
        self.C = model.num_channels
        self.non_negative = model.non_negative
        # ---- flat fp32 master parameters / gradients (16-byte aligned slices, state_dict order)
        names, params = zip(*model.named_parameters())
        sizes = [(p.numel() + 3) // 4 * 4 for p in params]
        self.flat = torch.zeros(sum(sizes), device=self.device, dtype=torch.float32)
        self.flat_grad = torch.zeros_like(self.flat)
        self.P: Dict[str, torch.Tensor] = {}
        self.G: Dict[str, torch.Tensor] = {}
        off = 0
        with torch.no_grad():
            for name, p, n in zip(names, params, sizes):
                self.flat[off:off + p.numel()].copy_(p.data.reshape(-1).float())
                p.data = self.flat[off:off + p.numel()].view_as(p.data)
                self.P[name] = p.data
                self.G[name] = self.flat_grad[off:off + p.numel()].view_as(p.data)
                off += n
        self.param_names = list(names)
        self.ws = _Workspace(self.device)          # weight operands, activations and gradients
        self._build_layer_table()
        self.pk = self._packed_weights()
        self.saved = None

    # ------------------------------------------------------------------ weight table / per-step packing
    def _build_layer_table(self):
        """(key, param name, n, c, taps, n_pad, standardize) for every GEMM weight; fwd [n_pad][taps*c],
        bwd [c][taps*n_pad] operand buffers are allocated once and re-filled every step."""
        T = []
        bb = "pretrained.model.patch_embed.backbone."
        cin = 64
        for s, (cout, depth) in enumerate(_STAGES):
            mid = cout // 4
            for b in range(depth):
                p = f"{bb}stages.{s}.blocks.{b}."
                if b == 0:
                    T.append((f"s{s}b{b}.wd", p + "downsample.conv.weight", cout, cin, 1, cout, True))
                T.append((f"s{s}b{b}.w1", p + "conv1.weight", mid, cin if b == 0 else cout, 1, mid, True))
                T.append((f"s{s}b{b}.w2", p + "conv2.weight", mid, mid, 9, mid, True))
                T.append((f"s{s}b{b}.w3", p + "conv3.weight", cout, mid, 1, cout, True))
            cin = cout
        pm = "pretrained.model."
        T.append(("proj", pm + "patch_embed.proj.weight", 768, 1024, 1, 768, False))
        for i in range(12):
            p = f"{pm}blocks.{i}."
            T.append((f"blk{i}.qkv", p + "attn.qkv.weight", 2304, 768, 1, 2304, False))
            T.append((f"blk{i}.proj", p + "attn.proj.weight", 768, 768, 1, 768, False))
            T.append((f"blk{i}.fc1", p + "mlp.fc1.weight", 3072, 768, 1, 3072, False))
            T.append((f"blk{i}.fc2", p + "mlp.fc2.weight", 768, 3072, 1, 768, False))
        for n in (3, 4):
            T.append((f"pp{n}", f"pretrained.act_postprocess{n}.3.weight", 768, 768, 1, 768, False))
        T.append(("pp4s", "pretrained.act_postprocess4.4.weight", 768, 768, 9, 768, False))
        for n, c in zip((1, 2, 3, 4), (256, 512, 768, 768)):
            T.append((f"rn{n}", f"scratch.layer{n}_rn.weight", 256, c, 9, 256, False))
        for n in (1, 2, 3, 4):
            p = f"scratch.refinenet{n}."
            T.append((f"ff{n}.out", p + "out_conv.weight", 256, 256, 1, 256, False))
            for u in ((2,) if n == 4 else (1, 2)):
                for cv in (1, 2):
                    T.append((f"ff{n}.rcu{u}.c{cv}", f"{p}resConfUnit{u}.conv{cv}.weight", 256, 256, 9, 256, False))
        T.append(("head0", "scratch.output_conv.0.weight", 128, 256, 9, 128, False))
        T.append(("head2", "scratch.output_conv.2.weight", 32, 128, 9, 64, False))     # carried zero-padded to 64
        self.layers = T
        self.W: Dict[str, Tuple[torch.Tensor, torch.Tensor]] = {}
        for key, pname, n, c, taps, n_pad, std in T:
            fwd = torch.zeros((n_pad, taps * c), device=self.device, dtype=self.adt)
            bwd_ = torch.zeros((c, taps * n_pad), device=self.device, dtype=self.adt)
            self.W[key] = (fwd, bwd_)
        self.meta = {key: (pname, n, c, taps, n_pad, std) for key, pname, n, c, taps, n_pad, std in T}
        self.gp = torch.empty(768 * 9 * 768, device=self.device, dtype=torch.float32)     # packed-layout wgrad scratch
        # one-launch packing of all layers; packed-layout gradient buffers of the layers that need the unpack pass
        # (3x3 taps or weight standardisation), converted by ONE launch per all-reduce bucket
        self.pack_table = bwd.PackTable([(self.P[pn], self.W[k][0], self.W[k][1], n, c, taps, n_pad, c, std)
                                         for k, pn, n, c, taps, n_pad, std in T], self.adt)
        self.gp_layer: Dict[str, torch.Tensor] = {}
        groups = {"decoder": [], "resnet": []}
        for k, pn, n, c, taps, n_pad, std in T:
            if taps == 1 and not std and n_pad == n:
                continue                                           # written straight into the flat gradient
            gp = torch.zeros((n_pad, taps * c), device=self.device, dtype=torch.float32)
            self.gp_layer[k] = gp
            tag = "resnet" if "backbone" in pn else "decoder"
            groups[tag].append((gp, self.P[pn], self.G[pn], n, c, taps, c, std))
        self.unpack_tables = {t: bwd.UnpackTable(v) for t, v in groups.items() if v}
        self.zb = torch.zeros(4096, device=self.device, dtype=torch.float32)               # zero "bias" of the dgrad convs:
        #   selects the straight-line (bias / bias + residual) epilogues of the tensor-core kernel

    def _packed_weights(self) -> dict:
        """The forward's weights, in the structure of DPTDepthModel._prepack, over the engine's persistent operands: the
        forward GEMM operands of the layer table, views of the fp32 master parameters and the buffers pack() fills."""
        P, W, get = self.P, {k: w[0] for k, w in self.W.items()}, self.ws.get
        pm, bb = "pretrained.model.", "pretrained.model.patch_embed.backbone."
        pk = {"stem_w": get("w.stem", (64, 160), self.adt),
              "stem_g": P[bb + "stem.norm.weight"], "stem_b": P[bb + "stem.norm.bias"], "rn_blocks": []}
        for s, (cout, depth) in enumerate(_STAGES):
            for b in range(depth):
                p, tag = f"{bb}stages.{s}.blocks.{b}.", f"s{s}b{b}"
                e = {"stride": 2 if (b == 0 and s > 0) else 1, "cout": cout, "mid": cout // 4}
                if b == 0:
                    e.update(wd=W[tag + ".wd"], gd=P[p + "downsample.norm.weight"], bd=P[p + "downsample.norm.bias"])
                for i in (1, 2, 3):
                    e[f"w{i}"], e[f"g{i}"], e[f"b{i}"] = W[f"{tag}.w{i}"], P[p + f"norm{i}.weight"], P[p + f"norm{i}.bias"]
                pk["rn_blocks"].append((s, b, e))
        pk["proj_w"], pk["proj_b"] = W["proj"], P[pm + "patch_embed.proj.bias"]
        pk["cls"], pk["pos"] = P[pm + "cls_token"].reshape(-1), P[pm + "pos_embed"]
        pk["vit"] = []
        for i in range(12):
            p = f"{pm}blocks.{i}."
            pk["vit"].append({"ln1": (P[p + "norm1.weight"], P[p + "norm1.bias"]),
                              "qkv": (W[f"blk{i}.qkv"], P[p + "attn.qkv.bias"]),
                              "proj": (W[f"blk{i}.proj"], P[p + "attn.proj.bias"]),
                              "ln2": (P[p + "norm2.weight"], P[p + "norm2.bias"]),
                              "fc1": (W[f"blk{i}.fc1"], P[p + "mlp.fc1.bias"]),
                              "fc2": (W[f"blk{i}.fc2"], P[p + "mlp.fc2.bias"])})
        for n in (3, 4):
            p = f"pretrained.act_postprocess{n}."
            pk[f"ro{n}_wfull"] = get(f"w.ro{n}.full", (768, 1536), self.adt)
            pk[f"ro{n}_wtok"] = get(f"w.ro{n}.tok", (768, 768), self.adt)
            pk[f"ro{n}_b"] = P[p + "0.project.0.bias"]
            pk[f"pp{n}_w"], pk[f"pp{n}_b"] = W[f"pp{n}"], P[p + "3.bias"]
        pk["pp4s_w"], pk["pp4s_b"] = W["pp4s"], P["pretrained.act_postprocess4.4.bias"]
        for n in (1, 2, 3, 4):
            p = f"scratch.refinenet{n}."
            pk[f"rn{n}_w"] = W[f"rn{n}"]
            pk[f"ff{n}_out"] = (W[f"ff{n}.out"], P[p + "out_conv.bias"])
            for u in ((2,) if n == 4 else (1, 2)):
                pk[f"ff{n}_rcu{u}"] = tuple((W[f"ff{n}.rcu{u}.c{cv}"], P[f"{p}resConfUnit{u}.conv{cv}.bias"]) for cv in (1, 2))
        pk["head0"] = (W["head0"], P["scratch.output_conv.0.bias"])
        pk["head2"] = (W["head2"], get("w.head2.bias", (64,), torch.float32))        # zero-padded to 64 like the weight
        pk["head4"] = (P["scratch.output_conv.4.weight"].reshape(self.C, 32), P["scratch.output_conv.4.bias"])
        return pk

    @torch.no_grad()
    def pack(self, batch: int):
        """fp32 master weights -> GEMM operands (every step: the optimizer just changed them).  Returns the position
        embedding as the forward takes it for `batch` images: (pos0 [D], pos[1:] replicated per image [batch, 576, D])."""
        self.pack_table.run()
        P, pk = self.P, self.pk
        bb = "pretrained.model.patch_embed.backbone."
        # stem 7x7 (3 input channels): [64,3,7,7] -> standardise -> [64, (ky,kx,c)=147] padded to 160 columns
        w = P[bb + "stem.conv.weight"]
        std_, mean = torch.std_mean(w, dim=[1, 2, 3], keepdim=True, unbiased=False)
        ws = ((w - mean) / (std_ + 1e-8)).permute(0, 2, 3, 1).reshape(64, 147)
        pk["stem_w"].zero_()
        pk["stem_w"][:, :147].copy_(ws)
        # ProjectReadout Linear(1536 -> 768): token half as a GEMM operand (fwd / bwd), whole matrix for the cls kernel
        for n in (3, 4):
            wfull = P[f"pretrained.act_postprocess{n}.0.project.0.weight"]
            pk[f"ro{n}_wfull"].copy_(wfull)
            pk[f"ro{n}_wtok"].copy_(wfull[:, :768])
            self.ws.get(f"w.ro{n}.tokT", (768, 768), self.adt).copy_(wfull[:, :768].t())
            self.ws.get(f"w.ro{n}.clsT", (768, 768), torch.float32).copy_(wfull[:, 768:].t())
        # stride-2 3x3 convolutions: per-parity-plane dgrad operands cut out of the rotated dgrad weight
        self.plane_w = {}
        for key, mode in (("s1b0.w2", "same"), ("s2b0.w2", "same"), ("pp4s", "sym1")):
            _, n, c, taps, n_pad, _ = self.meta[key]
            wb = self.W[key][1]                                    # [c][9 * n], tap slot 8 - t holds W_t^T
            for plane, taps_ in _parity_dgrad_plan(mode).items():
                cat = torch.cat([wb[:, (8 - t) * n_pad:(9 - t) * n_pad] for t, _, _ in taps_], dim=1).contiguous()
                self.plane_w[(key, plane)] = (cat, [(0, dx, dy) for _, dy, dx in taps_])
        b2 = pk["head2"][1]
        b2.zero_()
        b2[:32].copy_(P["scratch.output_conv.2.bias"])
        pos = P["pretrained.model.pos_embed"]
        pos_b = self.ws.get("pos_expanded", (batch, pos.shape[1] - 1, pos.shape[2]), torch.float32)
        pos_b.copy_(pos[0, 1:].unsqueeze(0).expand(batch, -1, -1))
        return pos[0, 0], pos_b

    # ------------------------------------------------------------------ small helpers
    def _wgrad(self, key: str, views, taps, dy, n_rows: Optional[int] = None):
        """weight gradient of layer `key` into the flat gradient buffer (through the weight standardisation)."""
        pname, n, c, ntaps, n_pad, std = self.meta[key]
        if ntaps == 1 and not std and n_pad == n:
            # linear / 1x1 layer without weight standardisation: the packed gradient layout IS the parameter layout
            bwd.conv_wgrad(views, taps, dy, self.G[pname].view(n, c))
            return
        bwd.conv_wgrad(views, taps, dy, self.gp_layer[key])        # converted to parameter layout by the bucket's unpack launch

    def _bias_grad(self, pname: str, dy, n: Optional[int] = None):
        g = self.G[pname]
        if n is None or dy.shape[-1] == g.numel():
            bwd.colsum(dy.reshape(-1, dy.shape[-1]), g.view(1, -1))
        else:                                                   # padded output channels (head conv2)
            tmp = self.ws.get("tmp.bias", (1, dy.shape[-1]), torch.float32)
            bwd.colsum(dy.reshape(-1, dy.shape[-1]), tmp)
            g.copy_(tmp[0, :g.numel()])

    def _zb(self, w: torch.Tensor):
        """zero bias vector for a dgrad convolution with weight `w` [n_out][K] (tensor-core path only)."""
        return None if self.fp32 else self.zb[: w.shape[0]]

    # ------------------------------------------------------------------ forward (activations kept)
    @torch.no_grad()
    def forward(self, x: torch.Tensor) -> torch.Tensor:
        if not x.is_cuda or x.dim() != 4 or x.shape[1] != 3:
            raise OdbError("TrainEngine.forward: CUDA input [B,3,H,W] required")
        x = x.detach().float().contiguous()
        B, _, H, W = x.shape
        if H % 32 or W % 32 or (H // 16) * (W // 16) + 1 > 640:
            raise ValueError("H and W must be multiples of 32 with at most 639 patches")
        if (H // 16, W // 16) != (24, 24):
            raise NotImplementedError("train step: 384x384 inputs (24x24 patch grid)")
        pos = self.pack(B)
        self.saved = {}
        return network_forward(self.pk, x, self.ws, self.model.arch, self.fp32, pos, self.non_negative, save=self.saved)

    # ------------------------------------------------------------------ backward
    def _dgrad_s2(self, key: str, dy, dx):
        """gradient w.r.t. the input of a stride-2 3x3 convolution: one small convolution per input parity plane,
        stored through a strided view of dx."""
        for (py, px) in ((0, 0), (0, 1), (1, 0), (1, 1)):
            w, taps = self.plane_w[(key, (py, px))]
            ops.conv_gemm([dy], taps, w, dx[:, py::2, px::2, :], bias=self._zb(w))

    @torch.no_grad()
    def backward(self, dout: torch.Tensor, on_ready=None):
        """dout: gradient w.r.t. the forward's output [B,C,H,W] fp32.  Fills self.flat_grad (all 368 tensors).
        on_ready(tag) is called when a contiguous range of the flat gradient is final (plan_grad_buckets): the
        data-parallel train step launches that range's all-reduce while the rest of the backward runs."""
        ready = on_ready if on_ready is not None else (lambda tag: None)
        S, P, G, Wt = self.saved, self.P, self.G, self.W
        buf = lambda name, shape, dtype=self.adt: self.ws.get(name, shape, dtype)
        if S is None:
            raise OdbError("TrainEngine.backward: call forward first")
        B, H, W = S["B"], S["H"], S["W"]
        f32 = torch.float32
        dout = dout.detach().float().contiguous().view(B, self.C, H, W)
        hd = S["head"]
        # ---- head
        da = buf("g.head_a", hd["a"].shape)
        bwd.head_tail_bwd(dout, hd["out"], hd["a"], hd["w4"], da, G["scratch.output_conv.4.weight"].view(self.C, 32),
                          G["scratch.output_conv.4.bias"], self.non_negative)
        dh1u = buf("g.head_h1u", hd["h1u"].shape)
        ops.conv3x3(da, Wt["head2"][1], dh1u, bias=self._zb(Wt["head2"][1]))
        self._wgrad("head2", [hd["h1u"]], bwd.TAPS_3X3, da)
        self._bias_grad("scratch.output_conv.2.bias", da, n=32)
        dh1 = buf("g.head_h1", hd["h1"].shape)
        bwd.upsample2x_bwd(dh1u, dh1)
        dpath = buf("g.path_1", hd["path_1"].shape)
        ops.conv3x3(dh1, Wt["head0"][1], dpath, bias=self._zb(Wt["head0"][1]))
        self._wgrad("head0", [hd["path_1"]], bwd.TAPS_3X3, dh1)
        self._bias_grad("scratch.output_conv.0.bias", dh1)

        # ---- RefineNet fusion blocks
        def rcu_bwd(n, u_, d_out, dx):
            """d_out: gradient w.r.t. the RCU output; dx <- gradient w.r.t. its (pre-ReLU) input."""
            r = S[f"ff{n}.rcu{u_}"]
            p = f"scratch.refinenet{n}.resConfUnit{u_}."
            dt = buf(f"g.ff{n}_rcu{u_}_t", r["tmid"].shape)
            ops.conv3x3(d_out, Wt[f"ff{n}.rcu{u_}.c2"][1], dt, bias=self._zb(Wt[f"ff{n}.rcu{u_}.c2"][1]))
            self._wgrad(f"ff{n}.rcu{u_}.c2", [r["tmid"]], bwd.TAPS_3X3, d_out)
            self._bias_grad(p + "conv2.bias", d_out)
            bwd.mask_add(dt, dt, mask=r["tmid"])                        # through relu(conv1 + b1)
            dxr = buf(f"g.ff{n}_rcu{u_}_x", r["x_raw"].shape)
            ops.conv3x3(dt, Wt[f"ff{n}.rcu{u_}.c1"][1], dxr, bias=self._zb(Wt[f"ff{n}.rcu{u_}.c1"][1]))
            self._wgrad(f"ff{n}.rcu{u_}.c1", [r["x_relu"]], bwd.TAPS_3X3, dt)
            self._bias_grad(p + "conv1.bias", dt)
            bwd.mask_add(dx, dxr, a=d_out, mask=r["x_relu"])            # skip + through relu(x)

        dz = buf("g.ff1_z", S["ff1"]["z"].shape)
        bwd.upsample2x_bwd(dpath, dz)
        d_rn = [None] * 4
        for n in (1, 2, 3, 4):
            f = S[f"ff{n}"]
            dy = buf(f"g.ff{n}_y", f["y"].shape)
            ops.conv1x1(dz, Wt[f"ff{n}.out"][1], dy, bias=self._zb(Wt[f"ff{n}.out"][1]))
            self._wgrad(f"ff{n}.out", [f["y"]], bwd.TAPS_1, dz)
            self._bias_grad(f"scratch.refinenet{n}.out_conv.bias", dz)
            ds_ = buf(f"g.ff{n}_s", f["y"].shape)
            rcu_bwd(n, 2, dy, ds_)
            if n == 4:
                d_rn[3] = ds_
            else:
                dr = buf(f"g.rn{n}_raw", f["y"].shape)
                rcu_bwd(n, 1, ds_, dr)                                  # res = RCU1(layer_rn): d res = d s
                d_rn[n - 1] = dr
                dz = buf(f"g.ff{n + 1}_z", S[f"ff{n + 1}"]["z"].shape)
                bwd.upsample2x_bwd(ds_, dz)
        # ---- scratch.layerN_rn
        d_layers = []
        for n in (1, 2, 3, 4):
            l = S["layers"][n - 1]
            dl = buf(f"g.layer_{n}", l.shape)
            ops.conv3x3(d_rn[n - 1], Wt[f"rn{n}"][1], dl, bias=self._zb(Wt[f"rn{n}"][1]))
            self._wgrad(f"rn{n}", [l], bwd.TAPS_3X3, d_rn[n - 1])
            d_layers.append(dl)
        # ---- reassemble: act_postprocess4.4 (stride 2), then the two readouts
        gh, gw, ntok, D = S["gh"], S["gw"], S["ntok"], 768
        u4 = S["ro4"]["o"]
        du4 = buf("g.pp4", u4.shape)
        self._dgrad_s2("pp4s", d_layers[3], du4)
        planes = [u4[:, py::2, px::2, :] for py in range(2) for px in range(2)]
        self._wgrad("pp4s", planes, ops._parity_taps("sym1"), d_layers[3])
        self._bias_grad("pretrained.act_postprocess4.4.bias", d_layers[3])

        def readout_bwd(n, do):
            """-> gradient w.r.t. the hooked tokens, activation type [B, ntok, D]."""
            r = S[f"ro{n}"]
            pp = f"pretrained.act_postprocess{n}."
            dr = buf(f"g.ro{n}_r", r["r"].shape)
            ops.conv1x1(do, Wt[f"pp{n}"][1], dr.view(B, gh, gw, D), bias=self._zb(Wt[f"pp{n}"][1]))
            self._wgrad(f"pp{n}", [r["r"].view(B, gh, gw, D)], bwd.TAPS_1, do)
            self._bias_grad(pp + "3.bias", do)
            bwd.gelu_bwd(dr, r["pre"], dr)
            dtk = buf(f"g.ro{n}_tok", (B, ntok, D))
            ops.linear(dr, self.ws.get(f"w.ro{n}.tokT", (D, D), self.adt), dtk[:, 1:, :].unsqueeze(1))
            gw_ = G[pp + "0.project.0.weight"]
            gp = self.gp[: D * D].view(D, D)
            bwd.conv_wgrad([r["tk"][:, 1:, :].unsqueeze(1)], bwd.TAPS_1, dr, gp)
            gw_[:, :D].copy_(gp)
            # cls half: cb[b] = W[:, D:] tok[b, 0] + bias, added to every token of image b
            dcb = buf(f"g.ro{n}_cb", (B, D), f32)
            bwd.colsum(dr.view(B, gh * gw, D), dcb, batches=B)
            bwd.colsum(dcb, G[pp + "0.project.0.bias"].view(1, -1))
            tok0 = buf(f"ro{n}_tok0", (B, D), f32)
            tok0.copy_(r["tk"][:, 0, :])
            bwd.conv_wgrad([tok0.view(1, 1, B, D)], bwd.TAPS_1, dcb.view(1, 1, B, D), gp)
            gw_[:, D:].copy_(gp)
            dt0 = buf(f"g.ro{n}_tok0", (B, D), f32)
            ops.linear(dcb, self.ws.get(f"w.ro{n}.clsT", (D, D), f32), dt0)
            dtk[:, 0, :].copy_(dt0)
            return dtk

        dtk4 = readout_bwd(4, du4)
        dtk3 = readout_bwd(3, d_layers[2])
        self.unpack_tables["decoder"].run()
        ready("decoder")
        # ---- ViT blocks (fp32 stream gradient ds, activation-type copy ds16 for the GEMMs)
        pm = "pretrained.model."
        rows = B * ntok
        xs, xm, vit = S["xs"], S["xm"], S["vit"]
        ds = buf("g.vit_ds", (B, ntok, D), f32)
        ds_b = buf("g.vit_ds_b", (B, ntok, D), f32)
        ds16 = buf("g.vit_ds16", (B, ntok, D)) if not self.fp32 else None
        bwd.add_cast(None, dtk4, ds, ds16)
        hooked = (8, 11)                                             # blocks whose output gradient gets a readout gradient
        for i in range(11, -1, -1):
            p = f"{pm}blocks.{i}."
            v = vit[i]
            if i == 5:
                ready("vit_hi")
            if i == 8:                                               # hook after block 8: tokens_8 also feed readout 3
                bwd.add_cast(ds, dtk3, ds, ds16)
            g16 = ds if self.fp32 else ds16
            # mlp: x_{i+1} = xm + fc2(gelu(fc1(LN2(xm))))
            dmlp = buf("g.vit_mlp", v["mlp"].shape)
            ops.linear(g16.view(rows, -1), Wt[f"blk{i}.fc2"][1], dmlp.view(rows, -1), bias=self._zb(Wt[f"blk{i}.fc2"][1]))
            self._wgrad(f"blk{i}.fc2", [v["mlp"].view(rows, -1)], bwd.TAPS_1, g16.view(rows, -1))
            if i in hooked:                                          # else: written by block i+1's norm1 backward
                bwd.colsum(ds.view(rows, -1), G[p + "mlp.fc2.bias"].view(1, -1))
            bwd.gelu_bwd(dmlp, v["u"], dmlp)
            dh = buf("g.vit_h", v["h2"].shape)
            ops.linear(dmlp.view(rows, -1), Wt[f"blk{i}.fc1"][1], dh.view(rows, -1), bias=self._zb(Wt[f"blk{i}.fc1"][1]))
            self._wgrad(f"blk{i}.fc1", [v["h2"].view(rows, -1)], bwd.TAPS_1, dmlp.view(rows, -1))
            self._bias_grad(p + "mlp.fc1.bias", dmlp.view(rows, -1))
            # ds_b = gradient at attn.proj's output: its column sums are proj's bias gradient (same pass)
            bwd.layernorm_bwd(dh, xm[i], P[p + "norm2.weight"], ds, ds_b, ds16, G[p + "norm2.weight"], G[p + "norm2.bias"],
                              dcolsum=G[p + "attn.proj.bias"])
            g16 = ds_b if self.fp32 else ds16
            # attention: xm = x_i + proj(attn(qkv(LN1(x_i))))
            datt = buf("g.vit_att", v["att"].shape)
            ops.linear(g16.view(rows, -1), Wt[f"blk{i}.proj"][1], datt.view(rows, -1), bias=self._zb(Wt[f"blk{i}.proj"][1]))
            self._wgrad(f"blk{i}.proj", [v["att"].view(rows, -1)], bwd.TAPS_1, g16.view(rows, -1))
            dqkv = buf("g.vit_qkv", v["qkv"].shape)
            bwd.attention_bwd(v["qkv"], v["att"], datt, v["lse"], dqkv, heads=12, scale=0.125)
            ops.linear(dqkv.view(rows, -1), Wt[f"blk{i}.qkv"][1], dh.view(rows, -1), bias=self._zb(Wt[f"blk{i}.qkv"][1]))
            self._wgrad(f"blk{i}.qkv", [v["h1"].view(rows, -1)], bwd.TAPS_1, dqkv.view(rows, -1))
            self._bias_grad(p + "attn.qkv.bias", dqkv.view(rows, -1))
            # ds = gradient at block i-1's output = at its mlp.fc2 output, unless a hook adds to it first
            fc2_bias = G[f"{pm}blocks.{i - 1}.mlp.fc2.bias"] if i >= 1 and (i - 1) not in hooked else None
            bwd.layernorm_bwd(dh, xs[i], P[p + "norm1.weight"], ds_b, ds, ds16, G[p + "norm1.weight"], G[p + "norm1.bias"],
                              dcolsum=fc2_bias)
        # ---- tokens: cls / pos_embed, patch projection
        gpos = G[pm + "pos_embed"]
        bwd.colsum(ds.view(B, ntok * D), gpos.view(1, -1))
        G[pm + "cls_token"].view(-1).copy_(gpos[0, 0])
        g16 = ds if self.fp32 else ds16
        f3 = S["f3"]
        dtok = g16[:, 1:, :].unsqueeze(1)
        df3 = buf("g.f3", f3.shape)
        ops.linear(dtok, Wt["proj"][1], df3.view(B, 1, gh * gw, 1024), bias=self._zb(Wt["proj"][1]))
        self._wgrad("proj", [f3.view(B, 1, gh * gw, 1024)], bwd.TAPS_1, dtok)
        tmpb = buf("tmp.projbias", (B, D), f32)
        bwd.colsum(ds[:, 1:, :], tmpb, batches=B)
        bwd.colsum(tmpb, G[pm + "patch_embed.proj.bias"].view(1, -1))
        ready("vit_lo")

        # ---- ResNetV2 bottlenecks, last to first
        d_out = df3
        for rec in reversed(S["blocks"]):
            tag, p, stride = rec["tag"], rec["p"], rec["stride"]
            s, b = rec["s"], rec["b"]
            # stage outputs also feed the decoder
            if (s, b) == (1, _STAGES[1][1] - 1):
                bwd.mask_add(d_out, d_layers[1], a=d_out)
            if (s, b) == (0, _STAGES[0][1] - 1):
                bwd.mask_add(d_out, d_layers[0], a=d_out)
            out, t_in = rec["out"], rec["t_in"]
            g = buf(f"g.{tag}_g", out.shape)
            bwd.mask_add(g, d_out, mask=out)                             # through the block's final ReLU
            dy3 = buf(f"g.{tag}_y3", out.shape)
            bwd.groupnorm_bwd(g, rec["y3"], rec["st3"], P[p + "norm3.weight"], dy3, G[p + "norm3.weight"], G[p + "norm3.bias"])
            da2 = buf(f"g.{tag}_a2", rec["a2"].shape)
            ops.conv1x1(dy3, Wt[tag + ".w3"][1], da2, bias=self._zb(Wt[tag + ".w3"][1]))
            self._wgrad(tag + ".w3", [rec["a2"]], bwd.TAPS_1, dy3)
            dy2 = buf(f"g.{tag}_y2", rec["y2"].shape)
            bwd.groupnorm_bwd(da2, rec["y2"], rec["st2"], P[p + "norm2.weight"], dy2, G[p + "norm2.weight"], G[p + "norm2.bias"],
                              mask=rec["a2"])
            da1 = buf(f"g.{tag}_a1", rec["a1"].shape)
            a1 = rec["a1"]
            if stride == 1:
                ops.conv3x3(dy2, Wt[tag + ".w2"][1], da1, bias=self._zb(Wt[tag + ".w2"][1]))
                self._wgrad(tag + ".w2", [a1], bwd.TAPS_3X3, dy2)
            else:
                self._dgrad_s2(tag + ".w2", dy2, da1)
                planes = [a1[:, py::2, px::2, :] for py in range(2) for px in range(2)]
                self._wgrad(tag + ".w2", planes, ops._parity_taps("same"), dy2)
            dy1 = buf(f"g.{tag}_y1", rec["y1"].shape)
            bwd.groupnorm_bwd(da1, rec["y1"], rec["st1"], P[p + "norm1.weight"], dy1, G[p + "norm1.weight"], G[p + "norm1.bias"],
                              mask=a1)
            dt_in = buf(f"g.{tag}_in", t_in.shape)
            if b == 0:
                dd = buf(f"g.{tag}_ds", rec["d"].shape)
                bwd.groupnorm_bwd(g, rec["d"], rec["std"], P[p + "downsample.norm.weight"], dd,
                                  G[p + "downsample.norm.weight"], G[p + "downsample.norm.bias"])
                if stride > 1:
                    dt_in.zero_()
                    ops.conv1x1(dd, Wt[tag + ".wd"][1], dt_in[:, ::stride, ::stride, :], bias=self._zb(Wt[tag + ".wd"][1]))
                    self._wgrad(tag + ".wd", [t_in[:, ::stride, ::stride, :]], bwd.TAPS_1, dd)
                else:
                    ops.conv1x1(dd, Wt[tag + ".wd"][1], dt_in, bias=self._zb(Wt[tag + ".wd"][1]))
                    self._wgrad(tag + ".wd", [t_in], bwd.TAPS_1, dd)
                ops.conv1x1(dy1, Wt[tag + ".w1"][1], dt_in, residual=dt_in, bias=self._zb(Wt[tag + ".w1"][1]))
            else:
                ops.conv1x1(dy1, Wt[tag + ".w1"][1], dt_in, residual=g, bias=self._zb(Wt[tag + ".w1"][1]))
            self._wgrad(tag + ".w1", [t_in], bwd.TAPS_1, dy1)
            d_out = dt_in
        # ---- stem
        bb = "pretrained.model.patch_embed.backbone."
        cols, s0, st0, t = S["stem"]
        g_s0 = buf("g.stem_gn", s0.shape)
        bwd.stem_pool_bwd(d_out, s0, st0, P[bb + "stem.norm.weight"], P[bb + "stem.norm.bias"], g_s0)
        ds0 = buf("g.stem_conv", s0.shape)
        bwd.groupnorm_bwd(g_s0, s0, st0, P[bb + "stem.norm.weight"], ds0, G[bb + "stem.norm.weight"], G[bb + "stem.norm.bias"])
        gp = self.gp[: 64 * 160].view(64, 160)
        h2, w2 = H // 2, W // 2
        bwd.conv_wgrad([cols.view(B, h2, w2, 160)], bwd.TAPS_1, ds0, gp)
        g147 = buf("tmp.stem_g", (64, 147), f32)
        g147.copy_(gp[:, :147])
        bwd.unpack_wgrad(g147, P[bb + "stem.conv.weight"], G[bb + "stem.conv.weight"], 64, 3, 49, 3, True)
        self.unpack_tables["resnet"].run()
        ready("resnet")
        return self.flat_grad


class _DptFunction(torch.autograd.Function):
    @staticmethod
    def forward(ctx, engine, x, *params):
        out = engine.forward(x)
        ctx.engine = engine
        return out.clone()

    @staticmethod
    def backward(ctx, grad_out):
        eng = ctx.engine
        eng.backward(grad_out)
        grads = tuple(eng.G[n].clone() for n in eng.param_names)
        return (None, None) + grads


def differentiable_forward(model: DPTDepthModel, x: torch.Tensor) -> torch.Tensor:
    """model(x) under autograd in train() mode: returns a tensor whose backward fills p.grad of every parameter
    (the gradient w.r.t. the input image is not produced: the reference never asks for it either)."""
    eng = getattr(model, "_train_engine", None)
    if eng is None or eng.fp32 != (model.precision == "fp32"):
        eng = TrainEngine(model, precision=model.precision)
        object.__setattr__(model, "_train_engine", eng)
    params = [p for _, p in model.named_parameters()]
    out = _DptFunction.apply(eng, x, *params)
    return out.squeeze(dim=1)


# ====================================================================================== the train step
def plan_grad_buckets(names: List[str], sizes: List[int]) -> List[Tuple[int, int, str]]:
    """Contiguous [start, end) ranges of the flat gradient buffer (state_dict order, padded sizes) in the order the
    backward COMPLETES them, so that each range can be all-reduced while the rest of the backward still runs:
      decoder + reassemble (scratch.*, act_postprocess*) -> ViT blocks 6..11 -> ViT blocks 0..5 + patch projection ->
      cls / pos_embed + the ResNetV2 stem and stages.
    Returns (start, end, ready_after) with ready_after in {"decoder", "vit_hi", "vit_lo", "resnet"}."""
    offs, off = {}, 0
    for n, s in zip(names, sizes):
        offs[n] = (off, off + s)
        off += s
    total = off

    def first(pred):
        return min(offs[n][0] for n in names if pred(n))
    b_blocks = first(lambda n: n.startswith("pretrained.model.blocks."))
    b_proj = first(lambda n: n.startswith("pretrained.model.patch_embed.proj."))
    b_blk6 = first(lambda n: n.startswith("pretrained.model.blocks.6."))
    b_tail = first(lambda n: n.startswith("pretrained.model.norm.") or n.startswith("pretrained.act_postprocess") or
                   n.startswith("scratch."))
    assert b_proj < b_blocks < b_blk6 < b_tail
    return [(b_tail, total, "decoder"), (b_blk6, b_tail, "vit_hi"), (b_proj, b_blk6, "vit_lo"), (0, b_proj, "resnet")]


class DepthTrainStep:
    """One process per GPU.  step(rgb, depth_gt, mask_float): forward -> clamp + MiDaS SSI + gradient-matching + virtual
    normal loss -> backward -> gradient all-reduce (data parallel, as the reference's PL DDP, train_depth.py:424-426:
    mean over ranks, bucketed, overlapped with the rest of the backward on a communication stream) -> clip_grad_norm_(10)
    -> Adam(lr) on the flat fp32 master weights (train_depth.py:381-383, Trainer(gradient_clip_val=10))."""

    def __init__(self, model: DPTDepthModel, lr: float = 1e-5, clip: Optional[float] = 10.0, precision: str = "bf16",
                 input_size=(384, 384)):
        import torch.distributed as dist
        from .losses import DepthStepLoss
        from .optim import FlatAdam
        self.engine = TrainEngine(model, precision)
        self.loss = DepthStepLoss(input_size)
        self.opt = FlatAdam(self.engine.flat, lr=lr)
        self.clip = clip
        self.dist = dist if (dist.is_available() and dist.is_initialized() and dist.get_world_size() > 1) else None
        self.world = self.dist.get_world_size() if self.dist else 1
        eng = self.engine
        sizes = [(eng.P[n].numel() + 3) // 4 * 4 for n in eng.param_names]
        self.buckets = plan_grad_buckets(eng.param_names, sizes)
        self.comm_stream = torch.cuda.Stream(eng.device) if self.dist else None
        self.global_step = 0
        self.allreduce_bytes = sum(e - s for s, e, _ in self.buckets) * 4 if self.dist else 0
        self._hooks_done: Dict[str, torch.cuda.Event] = {}
        # The eager step issues ~1150 launches from Python and is host-bound at batch 16; with use_cuda_graph the whole
        # launch sequence (forward, loss, backward, clip, Adam) is captured once per (shape, loss mix) and replayed.
        # Single-process by default; graph_collectives=True also captures the NCCL all-reduces (fork / join of the
        # communication stream inside the capture).
        self.use_cuda_graph = False
        self.graph_collectives = False
        self._graphs: Dict[tuple, dict] = {}

    def _allreduce_bucket(self, tag: str):
        """called by the backward when the range `tag` of the flat gradient is final"""
        if self.dist is None:
            return
        s, e = next((s, e) for s, e, t in self.buckets if t == tag)
        ev = torch.cuda.Event()
        ev.record(torch.cuda.current_stream(self.engine.device))
        with torch.cuda.stream(self.comm_stream):
            self.comm_stream.wait_event(ev)
            self.dist.all_reduce(self.engine.flat_grad[s:e], op=self.dist.ReduceOp.AVG)

    @torch.no_grad()
    def step(self, rgb: torch.Tensor, depth_gt: torch.Tensor, mask_float: torch.Tensor, points=None,
             full_mix: Optional[bool] = None) -> torch.Tensor:
        """-> fp32 [5] on the device: (loss, ssi, reg, vn, gradient norm before clipping); no host synchronisation."""
        if full_mix is None:
            full_mix = self.global_step >= 15000                     # train_depth.py:274-279
        if self.use_cuda_graph and (self.dist is None or self.graph_collectives):
            with torch.cuda.device(self.engine.device):             # capture / replay on the engine's device and stream
                return self._step_graph(rgb, depth_gt, mask_float, points, bool(full_mix))
        res = self._launch_sequence(rgb, depth_gt, mask_float, points, bool(full_mix), scalars_on_device=False)
        self.global_step += 1
        return res

    def _launch_sequence(self, rgb, depth_gt, mask_float, points, full_mix: bool, scalars_on_device: bool) -> torch.Tensor:
        eng = self.engine
        out = eng.forward(rgb)                                        # [B,1,H,W]
        losses, dpred = self.loss(out, depth_gt, mask_float, full_mix=full_mix, points=points)
        eng.backward(dpred, on_ready=self._allreduce_bucket)
        if self.dist is not None:
            torch.cuda.current_stream(eng.device).wait_stream(self.comm_stream)
        norm = self.opt.step(eng.flat_grad, max_norm=self.clip, scalars_on_device=scalars_on_device)
        res = torch.empty(5, device=eng.device, dtype=torch.float32)
        res[:4].copy_(losses)
        res[4:5].copy_(norm.reshape(1) if norm is not None else torch.zeros(1, device=eng.device))
        return res

    # ------------------------------------------------------------------ captured step
    _RING = 4           # host staging slots: the CPU may run at most _RING - 1 replays ahead of the GPU

    def _capture(self, key, rgb, depth_gt, mask_float, points, full_mix: bool) -> dict:
        eng, dev = self.engine, self.engine.device
        g = {"rgb": rgb.detach().float().contiguous().clone(), "gt": depth_gt.detach().float().contiguous().clone(),
             "mask": mask_float.detach().float().contiguous().clone(), "pts": None, "slot": 0,
             "host": [dict(scal=torch.zeros(2, dtype=torch.float32).pin_memory(), pts=None, done=None)
                      for _ in range(self._RING)]}
        if full_mix:
            arrs = [np.ascontiguousarray(q, dtype=np.int32) for q in points]
            g["pts"] = [torch.from_numpy(a).to(dev) for a in arrs]
            for h in g["host"]:
                h["pts"] = [torch.empty(a.shape, dtype=torch.int32).pin_memory() for a in arrs]
        # one eager step first (workspaces, kernel attributes, NCCL channels): a training step changes the weights and
        # the optimizer state, so both are put back before the capture
        snap = (eng.flat.clone(), self.opt.exp_avg.clone(), self.opt.exp_avg_sq.clone(), self.opt.step_count)
        cur = torch.cuda.current_stream(dev)
        side = torch.cuda.Stream(dev)
        side.wait_stream(cur)
        with torch.cuda.stream(side):
            self.opt.stage_step_scalars(g["host"][0]["scal"])
            self._launch_sequence(g["rgb"], g["gt"], g["mask"], g["pts"], full_mix, scalars_on_device=True)
        cur.wait_stream(side)
        torch.cuda.synchronize(dev)
        eng.flat.copy_(snap[0]); self.opt.exp_avg.copy_(snap[1]); self.opt.exp_avg_sq.copy_(snap[2])
        self.opt.step_count = snap[3]
        del snap
        graph = torch.cuda.CUDAGraph()
        # with NCCL in the capture, other threads of the process (the process group's watchdog) keep making CUDA calls:
        # restrict the capture's error checking to this thread
        mode = "thread_local" if self.dist is not None else "global"
        with torch.cuda.graph(graph, capture_error_mode=mode):
            g["res"] = self._launch_sequence(g["rgb"], g["gt"], g["mask"], g["pts"], full_mix, scalars_on_device=True)
        g["graph"] = graph
        g["scratch"] = bwd._SCRATCH.buf        # the shared kernel workspace the captured launches point into stays alive
        return g

    def _step_graph(self, rgb, depth_gt, mask_float, points, full_mix: bool) -> torch.Tensor:
        if full_mix and points is None:
            points = self.loss.vnl.select_index()                   # host NumPy RNG, the reference's call sequence
        key = (tuple(rgb.shape), tuple(depth_gt.shape), tuple(mask_float.shape), full_mix)
        g = self._graphs.get(key)
        if g is None:
            # the engine's activation buffers are re-allocated when the input shape changes: graphs of other shapes
            # would replay into freed memory
            for k in [k for k in self._graphs if k[:3] != key[:3]]:
                del self._graphs[k]
            g = self._graphs[key] = self._capture(key, rgb, depth_gt, mask_float, points, full_mix)
        h = g["host"][g["slot"]]
        g["slot"] = (g["slot"] + 1) % self._RING
        if h["done"] is not None:
            h["done"].synchronize()                                 # the replay that last read this staging slot has run
        g["rgb"].copy_(rgb); g["gt"].copy_(depth_gt); g["mask"].copy_(mask_float)
        if full_mix:
            for dst, hp, q in zip(g["pts"], h["pts"], points):
                hp.copy_(torch.from_numpy(np.ascontiguousarray(q, dtype=np.int32)))
                dst.copy_(hp, non_blocking=True)
        self.opt.stage_step_scalars(h["scal"])
        g["graph"].replay()
        h["done"] = torch.cuda.Event()
        h["done"].record(torch.cuda.current_stream(self.engine.device))
        self.global_step += 1
        return g["res"].clone()
