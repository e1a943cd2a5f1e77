"""Diagnostic (not a test): the bf16 train-step gradient of the benchmark regime against the fp32 correctness mode (the
reference arithmetic), same batch.  Prints global and per-bucket gradient norms and their relative differences.  How
much a one-ulp change of the forward (GELU of the bf16-rounded fc1 pre-activation) moves the gradient is on record in
profiles/r02_gradient_sensitivity.json.

    python tests/diag_gradnorm_gpu.py [batch] > gpurun_out/diag_gradnorm.json
"""
import json
import sys
from pathlib import Path

import numpy as np
import torch

sys.path.insert(0, str(Path(__file__).resolve().parents[1]))
from omnidata_b200 import synthetic  # noqa: E402
from omnidata_b200.losses import DepthStepLoss  # noqa: E402
from omnidata_b200.model import DPTDepthModel  # noqa: E402
from omnidata_b200.train import TrainEngine, plan_grad_buckets  # noqa: E402

IMG = 384


def main():
    B = int(sys.argv[1]) if len(sys.argv) > 1 else 4
    dev = torch.device("cuda:0")

    def make_model():
        model = DPTDepthModel(backbone="vitb_rn50_384")
        model.load_state_dict(synthetic.make_state_dict(0, 1), strict=True)
        model = model.to(dev)
        probe = (torch.rand(4, 3, IMG, IMG, generator=torch.Generator().manual_seed(77)) * 2 - 1).to(dev)
        sd = model.state_dict(keep_vars=True)
        w4, b4 = sd["scratch.output_conv.4.weight"], sd["scratch.output_conv.4.bias"]
        with torch.no_grad():                                   # the regime of omnidata_b200/train_bench.py
            b4.add_(100.0)
            model.eval()
            pre = model(probe).float() - 100.0
            b4.sub_(100.0)
            lo, hi = float(pre.min()), float(pre.max())
            sc = 0.8 / max(hi - lo, 1e-6)
            w4.mul_(sc)
            b4.copy_((b4 - lo) * sc + 0.1)
        return model

    gen = torch.Generator(device="cpu").manual_seed(2000)
    model = make_model()
    rgb = (torch.rand(B, 3, IMG, IMG, generator=gen) * 2 - 1).to(dev)
    with torch.no_grad():
        model.eval()
        p0 = model(rgb).float().unsqueeze(1).cpu()
    gt = (p0 * (0.8 + 0.4 * torch.rand(B, 1, IMG, IMG, generator=gen)) + 0.05 * torch.rand(B, 1, IMG, IMG, generator=gen)).clamp(0, 1).to(dev)
    mask = (torch.rand(B, 1, IMG, IMG, generator=gen) > 0.1).float().to(dev)
    np.random.seed(1234)
    loss = DepthStepLoss((IMG, IMG))
    points = loss.vnl.select_index()

    grads, outs = {}, {}
    for name, precision in (("bf16", "bf16"), ("fp32_mode", "fp32")):
        m = make_model().train()
        eng = TrainEngine(m, precision)
        out = eng.forward(rgb)
        losses, dpred = loss(out, gt, mask, full_mix=True, points=points)
        eng.backward(dpred)
        torch.cuda.synchronize()
        grads[name] = eng.flat_grad.double().clone()
        outs[name] = (out.double().clone(), [float(v) for v in losses.cpu()])
        names = eng.param_names
        sizes = [(eng.P[n].numel() + 3) // 4 * 4 for n in names]
        del eng, m
        torch.cuda.empty_cache()
    buckets = plan_grad_buckets(names, sizes)
    rep = {"batch": B, "losses": {k: v[1] for k, v in outs.items()},
           "prediction_rel_diff_vs_fp32": float((outs["bf16"][0] - outs["fp32_mode"][0]).norm() / outs["fp32_mode"][0].norm()),
           "grad_norm": {k: float(g.norm()) for k, g in grads.items()}, "buckets": {}}

    def rel(a, b):
        return float((a - b).norm() / (b.norm() + 1e-300))
    rep["rel_diff_bf16_vs_fp32"] = rel(grads["bf16"], grads["fp32_mode"])
    for s, e, tag in buckets:
        rep["buckets"][tag] = {"norm": {k: float(g[s:e].norm()) for k, g in grads.items()},
                               "bf16_vs_fp32": rel(grads["bf16"][s:e], grads["fp32_mode"][s:e])}
    print(json.dumps(rep, indent=1))


if __name__ == "__main__":
    main()
