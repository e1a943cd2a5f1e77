"""Inputs above 640 tokens (512x512 and up): the key-streaming attention kernels and the whole model at high
resolution.

Kernels: the bf16 tcgen05 streaming kernel against the bf16-rounding oracle (oracle/dpt_oracle.py::_attention_bf16)
and exact softmax, with the bounds of tests/test_kernels_gpu.py::test_attention; the fp32-mode streaming kernel
against float64, with the bound of tests/test_fp32_mode_gpu.py.  Model: DPT-Hybrid depth and normal at four sizes
against the CPU fp32 oracle (fp32 mode 1e-5 at every tap; bf16 mode no worse than stock torch.autocast(bfloat16) of
the oracle on the same GPU and input), the plain-ViT backbones against their own fp32 mode and HuggingFace's DPT
port, CUDA-graph replay and batch independence at 1024x1024, and demo.py --image_size."""
import subprocess
import sys
from pathlib import Path

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

ROOT = Path(__file__).resolve().parents[1]
KERNEL_TOL = 2e-6             # tests/test_fp32_mode_gpu.py: one op in fp32 with fp64 sums
FP32_TOL = 1e-5
# The post-ReLU depth output in fp32 mode at 448x768 and 1024x1024 measured 1.16e-5 and 1.04e-5 against the CPU fp32
# oracle on one NVIDIA B200 (1000 W power limit); every tap, the pre-ReLU head included, stays <= 7.8e-6.  That is
# what two fp32 evaluations in different summation orders give there: the oracle's own fp32 output is 7.6e-6 and
# 8.7e-6 away from its float64 evaluation at those sizes (5.6e-6 at 384x384).  Bound = 1.16e-5 x 1.2.
FP32_DEPTH_OUTPUT_TOL = 1.4e-5
BF16_OUTPUT_CEILING = 6e-2    # tests/test_entrypoints_gpu.py
# fp32 mode of the plain-ViT models vs HuggingFace's DPT port (fp32, on the CPU) at 512x512 (vitl16_384) and 768x768
# (vitb16_384).  Measured on one NVIDIA B200 (1000 W power limit): 8.1e-7 and 1.66e-6; bound = measured x 1.2, rounded
# up.  (HF's own fp32 result is 5.0e-7 and 1.1e-6 from its float64 evaluation.)
HF_TOL = {"vitl16_384": 1.0e-6, "vitb16_384": 2.0e-6}
TAPS = ["layer_1", "layer_2", "tokens_8", "tokens_11", "layer_3", "layer_4", "layer_1_rn", "layer_2_rn", "layer_3_rn",
        "layer_4_rn", "path_4", "path_3", "path_2", "path_1"]


def dev():
    return torch.device("cuda:0")


def rnd(*shape, scale=1.0, seed=0):
    g = torch.Generator(device="cpu").manual_seed(seed + sum(shape))
    return (torch.randn(*shape, generator=g) * scale).to(dev())


def rel(a, b):
    a, b = a.double(), b.double()
    return float((a - b).norm() / (b.norm() + 1e-30))


@pytest.fixture(scope="module", autouse=True)
def _setup(lib_built):
    torch.backends.cuda.matmul.allow_tf32 = False
    torch.backends.cudnn.allow_tf32 = False
    yield


# ---------------------------------------------------------------------------------------------------- kernels
@pytest.mark.parametrize("heads", [12, 16])
@pytest.mark.parametrize("tokens", [641, 1025, 1345, 2305, 4097])
def test_attention_bf16_streaming(tokens, heads):
    from omnidata_b200 import ops
    from oracle.dpt_oracle import _attention_bf16
    b, d = 3, heads * 64
    qkv = rnd(b, tokens, 3 * d)
    qkv[..., :2 * d] *= 2.0           # peaky softmax, as in a trained ViT
    qkv = qkv.to(torch.bfloat16)
    out = torch.full((b, tokens, d), float("nan"), device=dev(), dtype=torch.bfloat16)
    ops.attention(qkv, out, heads=heads)
    again = torch.full_like(out, float("nan"))
    ops.attention(qkv, again, heads=heads)
    alone = []
    for i in range(b):
        o1 = torch.full((1, tokens, d), float("nan"), device=dev(), dtype=torch.bfloat16)
        ops.attention(qkv[i:i + 1].contiguous(), o1, heads=heads)
        alone.append(o1)
    torch.cuda.synchronize()
    assert torch.equal(out, again)                                  # bit-reproducible
    for i in range(b):
        assert torch.equal(out[i:i + 1], alone[i]), i               # independent of the rest of the batch
    q, k, v = qkv.float().view(b, tokens, 3, heads, 64).permute(2, 0, 3, 1, 4)
    ref = _attention_bf16(q, k, v).transpose(1, 2).reshape(b, tokens, d)
    err = rel(out.float(), ref.to(torch.bfloat16).float())
    assert err <= 1e-3, err
    exact = (torch.softmax(q @ k.transpose(-1, -2) * 0.125, dim=-1) @ v).transpose(1, 2).reshape(b, tokens, d)
    err = rel(out.float(), exact)
    assert err < 4e-3, err


def test_attention_bf16_streaming_rejects_lse():
    from omnidata_b200 import ops
    from omnidata_b200._capi import OdbError
    qkv = rnd(1, 641, 2304).to(torch.bfloat16)
    out = torch.empty(1, 641, 768, device=dev(), dtype=torch.bfloat16)
    lse = torch.empty(1, 12, 641, device=dev())
    with pytest.raises(OdbError):
        ops.attention(qkv, out, lse=lse)


@pytest.mark.parametrize("tokens", [641, 2305, 4097])
def test_attention_fp32_streaming(tokens):
    from omnidata_b200 import ops
    b = 2 if tokens < 4000 else 1
    qkv = rnd(b, tokens, 2304)
    qkv[..., :1536] *= 2.0
    out = torch.full((b, tokens, 768), float("nan"), device=dev())
    ops.attention(qkv, out)
    torch.cuda.synchronize()
    q, k, v = qkv.double().view(b, tokens, 3, 12, 64).permute(2, 0, 3, 1, 4)
    ref = (torch.softmax(q @ k.transpose(-1, -2) * 0.125, dim=-1) @ v).transpose(1, 2).reshape(b, tokens, 768)
    err = rel(out, ref)
    assert err < KERNEL_TOL, err


# ---------------------------------------------------------------------------------------------------- DPT-Hybrid
SIZES = [(512, 320), (512, 512), (448, 768), (1024, 1024)]


def _nchw(name, t):
    t = t.float().cpu()
    return t if (name.startswith("tokens") or t.dim() != 4 or name == "head_pre_relu") else t.permute(0, 3, 1, 2)


@pytest.fixture(scope="module", params=SIZES, ids=lambda s: f"{s[0]}x{s[1]}")
def hybrid_run(lib_built, request):
    from omnidata_b200.model import DPTDepthModel
    from oracle import dpt_oracle, weights
    H, W = request.param
    g = torch.Generator().manual_seed(H + W)
    x = torch.rand(1, 3, H, W, generator=g) * 2 - 1
    res = {}
    for c in (1, 3):
        sd = weights.make_state_dict(0, c)
        model = DPTDepthModel(backbone="vitb_rn50_384", num_channels=c)
        model.load_state_dict(sd, strict=True)
        model = model.cuda().eval()
        model.keep_taps = True
        r = {}
        with torch.no_grad():
            for prec in ("bf16", "fp32"):
                model.precision = prec
                y = model(x.cuda())
                torch.cuda.synchronize()
                r[prec] = (y.float().cpu(), {k: _nchw(k, v) for k, v in model.taps.items()})
            t32, tac = {}, {}
            y32 = dpt_oracle.forward_fp32(sd, x, t32)
            sdg = {k: v.cuda() for k, v in sd.items()}
            with torch.autocast("cuda", dtype=torch.bfloat16):
                yac = dpt_oracle.forward_fp32(sdg, x.cuda(), tac).float().cpu()
        r.update(y32=y32, t32=t32, yac=yac, tac={k: v.float().cpu() for k, v in tac.items()})
        res[c] = r
        del model, sdg
        torch.cuda.empty_cache()
    return (H, W), res


@pytest.mark.parametrize("c", [1, 3])
def test_hybrid_fp32_mode_matches_oracle_at_every_tap(hybrid_run, c):
    (H, W), res = hybrid_run
    r = res[c]
    y, taps = r["fp32"]
    assert tuple(y.shape) == ((1, H, W) if c == 1 else (1, 3, H, W))
    report = {k: rel(taps[k], r["t32"][k]) for k in TAPS + ["head_pre_relu"]}
    report["output"] = rel(y, r["y32"])
    print("\n".join(f"{H}x{W} c{c} {k}: {v:.2e}" for k, v in report.items()))
    for k, v in report.items():
        assert v <= (FP32_DEPTH_OUTPUT_TOL if (k, c) == ("output", 1) else FP32_TOL), (k, v, report)


@pytest.mark.parametrize("c", [1, 3])
def test_hybrid_bf16_not_worse_than_stock_autocast(hybrid_run, c):
    (H, W), res = hybrid_run
    r = res[c]
    y, taps = r["bf16"]
    assert tuple(y.shape) == ((1, H, W) if c == 1 else (1, 3, H, W))
    report = {k: (rel(taps[k], r["t32"][k]), rel(r["tac"][k], r["t32"][k])) for k in TAPS}
    report["output"] = (rel(y, r["y32"]), rel(r["yac"], r["y32"]))
    print("\n".join(f"{H}x{W} c{c} {k}: {m:.3e} (autocast {s:.3e})" for k, (m, s) in report.items()))
    for k, (mine, stock) in report.items():
        assert mine <= 1.10 * stock, (k, mine, stock)


def test_hybrid_rejects_inputs_the_stem_cannot_take():
    from omnidata_b200.model import DPTDepthModel
    from omnidata_b200 import synthetic
    m = DPTDepthModel()
    m.load_state_dict(synthetic.make_state_dict(0, 1))
    m = m.cuda().eval()
    with torch.no_grad(), pytest.raises(ValueError, match="1792"):
        m(torch.zeros(1, 3, 64, 1824, device=dev()))
    with torch.no_grad(), pytest.raises(ValueError, match="multiples of 32"):
        m(torch.zeros(1, 3, 64, 80, device=dev()))


def test_hybrid_graph_replay_and_batch_independence_at_1024():
    from omnidata_b200.model import DPTDepthModel
    from omnidata_b200 import synthetic
    m = DPTDepthModel()
    m.load_state_dict(synthetic.make_state_dict(0, 1))
    m = m.cuda().eval()
    g = torch.Generator().manual_seed(3)
    x = (torch.rand(2, 3, 1024, 1024, generator=g) * 2 - 1).cuda()
    with torch.no_grad():
        eager = m(x)
        singles = [m(x[i:i + 1]) for i in range(2)]
        m.use_cuda_graph = True
        graphed = m(x)
        graphed2 = m(x)
    torch.cuda.synchronize()
    assert eager.shape == (2, 1024, 1024)
    assert torch.equal(eager, graphed) and torch.equal(graphed, graphed2)
    for i in range(2):
        assert torch.equal(eager[i:i + 1], singles[i]), i


# ---------------------------------------------------------------------------------------------------- plain ViT
@pytest.mark.parametrize("backbone,size", [("vitl16_384", 512), ("vitb16_384", 768)])
def test_plain_vit_high_resolution(backbone, size):
    from omnidata_b200 import synthetic
    from omnidata_b200.model import DPTDepthModel, state_dict_spec
    from oracle import make_golden
    sd = synthetic.make_state_dict(0, 1, spec=state_dict_spec(1, backbone=backbone))
    m = DPTDepthModel(backbone=backbone)
    m.load_state_dict(sd, strict=True)
    m = m.cuda().eval()
    x = make_golden.golden_input(1, seed=0, size=size)
    with torch.no_grad():
        y16 = m(x.cuda()).float().cpu()
        m.precision = "fp32"
        y32 = m(x.cuda()).float().cpu()
    assert y16.shape == (1, size, size)
    err16 = rel(y16, y32)
    print(f"{backbone} {size}: bf16 vs fp32 mode {err16:.3e}")
    assert err16 <= BF16_OUTPUT_CEILING, err16
    pytest.importorskip("transformers")
    from transformers import DPTConfig, DPTForDepthEstimation
    from test_timm_shim_vs_hf_cpu import remap_plain_vit
    dim, depth, heads, hooks, neck = {
        "vitl16_384": (1024, 24, 16, [5, 11, 17, 23], [256, 512, 1024, 1024]),
        "vitb16_384": (768, 12, 12, [2, 5, 8, 11], [96, 192, 384, 768])}[backbone]
    cfg = DPTConfig(is_hybrid=False, image_size=384, patch_size=16, hidden_size=dim, num_hidden_layers=depth,
                    num_attention_heads=heads, intermediate_size=4 * dim, backbone_out_indices=hooks,
                    readout_type="project", neck_hidden_sizes=neck, reassemble_factors=[4, 2, 1, 0.5],
                    fusion_hidden_size=256, qkv_bias=True, hidden_act="gelu", layer_norm_eps=1e-6,
                    hidden_dropout_prob=0.0, attention_probs_dropout_prob=0.0)
    hf = DPTForDepthEstimation(cfg).eval()
    hf.load_state_dict(remap_plain_vit(sd, depth, dim), strict=False)
    with torch.no_grad():
        y_hf = hf(pixel_values=x).predicted_depth
    err = rel(y32, y_hf)
    print(f"{backbone} {size}: fp32 mode vs HF port {err:.3e}")
    assert err <= HF_TOL[backbone], err


# ---------------------------------------------------------------------------------------------------- demo
@pytest.mark.parametrize("task", ["normal", "depth"])
def test_demo_image_size(tmp_path, task):
    from PIL import Image
    rng = np.random.default_rng(1)
    src = tmp_path / "test1.png"
    Image.fromarray(rng.integers(0, 256, size=(900, 1000, 3), dtype=np.uint8)).save(src)
    out = tmp_path / "out"
    r = subprocess.run([sys.executable, str(ROOT / "demo.py"), "--task", task, "--img_path", str(src),
                        "--output_path", str(out), "--synthetic_weights", "--weights_dir", str(tmp_path / "none"),
                        "--image_size", "768"], capture_output=True, text=True, cwd=str(ROOT), timeout=600)
    assert r.returncode == 0, r.stderr[-2000:]
    res = Image.open(out / f"test1_{task}.png")
    assert Image.open(out / "test1_rgb.png").size == (512, 512)
    assert res.size == ((768, 768) if task == "normal" else (512, 512))
    assert np.asarray(res).std() > 0
