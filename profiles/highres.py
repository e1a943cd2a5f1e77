"""High-resolution inference on one GPU: images/s of the depth model (CUDA graph, CUDA events) and the attention
kernels at each size against torch's scaled_dot_product_attention on the same bf16 qkv.

    python profiles/highres.py OUT_DIR          -> OUT_DIR/highres.json

Attention work is counted algorithmically, 4 * B * heads * N^2 * 64 FLOP per launch (QK^T and PV): the streaming
kernel's second QK^T pass (above 640 tokens) is recompute and is not counted.  Up to 640 tokens odb_attention runs
the resident-K/V kernel, above it the key-streaming kernel.  Each timing window is at least two seconds after a
warm-up of the same shape.  qkv is the same buffer on every launch, so where it fits (< 126 MB) it is read from L2."""
import json
import statistics
import subprocess
import sys
from pathlib import Path

import torch
import torch.nn.functional as F

sys.path.insert(0, str(Path(__file__).resolve().parents[1]))
from omnidata_b200 import ops, synthetic  # noqa: E402
from omnidata_b200.model import _ARCH, DPTDepthModel, state_dict_spec  # noqa: E402

MODEL_CASES = [("vitb_rn50_384", 32, 384, 384), ("vitb_rn50_384", 8, 512, 512), ("vitb_rn50_384", 4, 768, 768),
               ("vitb_rn50_384", 2, 1024, 1024), ("vitl16_384", 4, 768, 768)]
MIN_WINDOW_MS = 2000.0


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    name, power, clock = [s.strip() for s in q.stdout.strip().splitlines()[0].split(",")]
    return {"name": name, "power_limit": power, "max_sm_clock": clock, "torch_name": torch.cuda.get_device_name()}


def timed(fn, min_ms=MIN_WINDOW_MS):
    """ms per call of fn over a window of at least min_ms, after a warm-up."""
    for _ in range(3):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(3):
        fn()
    e1.record()
    torch.cuda.synchronize()
    n = max(10, int(min_ms / max(e0.elapsed_time(e1) / 3, 1e-3)) + 1)
    e0.record()
    for _ in range(n):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / n, n


def attention_case(b, tokens, heads):
    g = torch.Generator(device="cpu").manual_seed(tokens)
    qkv = torch.randn(b, tokens, 3 * heads * 64, generator=g)
    qkv[..., :2 * heads * 64] *= 2.0
    qkv = qkv.to(torch.bfloat16).cuda()
    out = torch.empty(b, tokens, heads * 64, device="cuda", dtype=torch.bfloat16)
    flop = 4.0 * b * heads * tokens * tokens * 64
    ours, _ = timed(lambda: ops.attention(qkv, out, heads=heads))     # warm-up and window length
    n = max(20, int(MIN_WINDOW_MS / ours))
    with ops.LaunchTimer() as lt:
        for _ in range(n):
            ops.attention(qkv, out, heads=heads)
    per_launch = [t for _, _, t in lt.results()]
    ms = statistics.median(per_launch)
    q, k, v = qkv.view(b, tokens, 3, heads, 64).permute(2, 0, 3, 1, 4)
    sdpa_ms, _ = timed(lambda: F.scaled_dot_product_attention(q, k, v, scale=0.125))
    return {"batch": b, "tokens": tokens, "heads": heads, "kernel": "resident" if tokens <= 640 else "streaming",
            "launches_timed": n, "median_ms": ms, "min_ms": min(per_launch), "max_ms": max(per_launch),
            "tflops": flop / ms / 1e9, "ns_per_query_key_pair_per_head": ms * 1e6 / (b * heads * tokens * tokens),
            "sdpa_ms": sdpa_ms, "sdpa_tflops": flop / sdpa_ms / 1e9, "qkv_mb": qkv.numel() * 2 / 1e6}


def model_case(backbone, b, h, w):
    spec = state_dict_spec(1, backbone=backbone)
    model = DPTDepthModel(backbone=backbone)
    model.load_state_dict(synthetic.make_state_dict(0, 1, spec=spec))
    model = model.cuda().eval()
    x = torch.rand(b, 3, h, w, device="cuda") * 2 - 1
    with torch.no_grad():
        model.use_cuda_graph = True
        ms, n = timed(lambda: model(x))
    del model
    torch.cuda.empty_cache()
    return {"backbone": backbone, "batch": b, "height": h, "width": w, "steps_timed": n, "ms_per_step": ms,
            "images_per_s": b / ms * 1e3}


def main():
    if len(sys.argv) != 2:
        raise SystemExit("usage: python profiles/highres.py OUT_DIR")
    out_dir = Path(sys.argv[1])
    out_dir.mkdir(parents=True, exist_ok=True)
    if not torch.cuda.is_available():
        raise SystemExit("profiles/highres.py measures on a CUDA device; none is visible")
    res = {"gpu": gpu_info(), "method": __doc__, "models": [], "attention": []}
    for backbone, b, h, w in MODEL_CASES:
        r = model_case(backbone, b, h, w)
        print(json.dumps(r), flush=True)
        res["models"].append(r)
    for backbone, b, h, w in MODEL_CASES:
        heads = _ARCH[backbone]["heads"]
        r = attention_case(b, (h // 16) * (w // 16) + 1, heads)
        r["backbone"] = backbone
        print(json.dumps(r), flush=True)
        res["attention"].append(r)
    res["gpu_after"] = gpu_info()
    (out_dir / "highres.json").write_text(json.dumps(res, indent=1) + "\n")


if __name__ == "__main__":
    main()
