#!/usr/bin/env python
"""CLI with the reference's flags and outputs (omnidata_tools/torch/demo.py:23-36,125-163):

    python demo.py --task {normal,depth} --img_path FILE-or-DIR --output_path DIR

writes <name>_<task>.png and <name>_rgb.png.  Weights: ./pretrained_models/omnidata_dpt_{normal,depth}_v2.ckpt
(reference checkpoint names, demo.py:62,80); `--synthetic_weights` substitutes seeded random weights
when no checkpoint is available (offline).  Inference runs on cuda:0 through the sm_100a kernels —
there is no CPU path.
"""
from __future__ import annotations

import argparse
import glob
import os
import sys
from pathlib import Path

import numpy as np
import torch
from PIL import Image

_VIRIDIS = np.array([[68, 1, 84], [72, 40, 120], [62, 74, 137], [49, 104, 142], [38, 130, 142], [31, 158, 137],
                     [53, 183, 121], [109, 205, 89], [180, 222, 44], [253, 231, 37]], dtype=np.float32)


def viridis(a: np.ndarray) -> np.ndarray:
    """Depth colouring of demo.py:147 `plt.imsave(path, depth, cmap='viridis')`: normalise to the data range, map through
    viridis.  With matplotlib installed its own 256-entry LUT and quantisation are used (the reference's exact RGB
    values; the reference writes RGBA, this writes RGB).  matplotlib is absent from this image and its table is not
    reproducible offline: the fallback interpolates ten anchor colours of the map and is off by a few levels between
    anchors — a visual approximation, not a bit-exact one."""
    lo, hi = float(a.min()), float(a.max())
    t = (a - lo) / (hi - lo) if hi > lo else np.zeros_like(a)
    try:
        from matplotlib import cm
        return (cm.get_cmap("viridis")(t, bytes=True)[..., :3]).astype(np.uint8)
    except Exception:
        pass
    pos = t * (len(_VIRIDIS) - 1)
    i0 = np.clip(np.floor(pos).astype(int), 0, len(_VIRIDIS) - 2)
    w = (pos - i0)[..., None]
    rgb = _VIRIDIS[i0] * (1 - w) + _VIRIDIS[i0 + 1] * w
    return rgb.round().astype(np.uint8)


def resize_center_crop(img: Image.Image, size: int) -> Image.Image:
    """transforms.Resize(size, BILINEAR) + CenterCrop(size) on a PIL image (demo.py:74-76)."""
    w, h = img.size
    if w <= h:
        nw, nh = size, int(size * h / w)
    else:
        nw, nh = int(size * w / h), size
    img = img.resize((nw, nh), Image.BILINEAR)
    left, top = int(round((nw - size) / 2.0)), int(round((nh - size) / 2.0))
    return img.crop((left, top, left + size, top + size))


def to_tensor(img: Image.Image) -> torch.Tensor:
    a = np.asarray(img, dtype=np.float32) / 255.0
    if a.ndim == 2:
        a = a[..., None]
    return torch.from_numpy(a).permute(2, 0, 1).contiguous()


def build_model(task: str, root_dir: str, synthetic: bool, device):
    import hubconf
    model = hubconf.dpt_hybrid_384(pretrained=False, task=task)
    ckpt = os.path.join(root_dir, hubconf._CKPT[task])
    if os.path.exists(ckpt):
        hubconf._load_checkpoint(model, ckpt)
    elif synthetic:
        from omnidata_b200 import synthetic as syn
        model.load_state_dict(syn.make_state_dict(0, model.num_channels))
        print(f"[demo] {ckpt} not found: using seeded synthetic weights")
    else:
        raise FileNotFoundError(f"{ckpt} not found (pass --synthetic_weights to run without a checkpoint)")
    return model.to(device).eval()


def main(argv=None):
    parser = argparse.ArgumentParser(description="Visualize output for depth or surface normals")
    parser.add_argument("--task", dest="task", default="NONE", help="normal or depth")
    parser.add_argument("--img_path", dest="img_path", help="path to rgb image")
    parser.add_argument("--output_path", dest="output_path", help="path to where output image should be stored")
    parser.add_argument("--synthetic_weights", action="store_true")
    parser.add_argument("--weights_dir", default="./pretrained_models/")
    parser.add_argument("--image_size", type=int, default=384,
                        help="side of the square network input (a multiple of 32); above 384 gives sharper maps")
    args = parser.parse_args(argv)
    if args.task not in ("normal", "depth"):
        print("task should be one of the following: normal, depth")
        sys.exit()
    if args.image_size < 32 or args.image_size % 32:
        parser.error("--image_size must be a positive multiple of 32")
    if not torch.cuda.is_available():
        print("demo.py: a CUDA (sm_100a) device is required; this implementation has no CPU path")
        sys.exit(1)
    device = torch.device("cuda:0")
    os.makedirs(args.output_path, exist_ok=True)
    model = build_model(args.task, args.weights_dir, args.synthetic_weights, device)
    image_size = args.image_size
    from omnidata_b200 import imageproc
    preprocess = imageproc.DevicePreprocessor(args.task, image_size, device)

    def save_outputs(img_path, name):
        with torch.no_grad():
            save_path = os.path.join(args.output_path, f"{name}_{args.task}.png")
            print(f"Reading input {img_path} ...")
            img = Image.open(img_path)
            if img.mode in ("RGB", "L"):
                # Resize(image_size, BILINEAR) + CenterCrop + ToTensor [+ Normalize] on the device: the decoded
                # 8-bit image is uploaded once, the kernels reproduce Pillow's fixed-point resize exactly
                t = preprocess(np.array(img)).unsqueeze(0)
            else:
                # RGBA / palette / 16-bit: Pillow converts or premultiplies before resizing — keep its path
                t = to_tensor(resize_center_crop(img, image_size))[:3]
                if args.task == "depth":
                    t = (t - 0.5) / 0.5                               # Normalize(0.5, 0.5), demo.py:92-95
                t = t.unsqueeze(0).to(device)
                if t.shape[1] == 1:
                    t = t.repeat_interleave(3, 1)
            resize_center_crop(img, 512).save(os.path.join(args.output_path, f"{name}_rgb.png"))
            output = model(t)
            if args.task == "depth":
                # clamp(0,1) -> bicubic 512 -> clamp(0,1) -> 1 - x in one kernel (demo.py:140-145)
                output = imageproc.bicubic_resize(output.float(), (512, 512), clamp_in=True, clamp_out=True, invert=True)
                Image.fromarray(viridis(output.detach().cpu().squeeze().numpy())).save(save_path)
            else:
                # clamp(0,1) + ToPILImage: uint8 HWC = trunc(x * 255) (demo.py:140,150)
                arr = imageproc.to_uint8_hwc(output[0].float(), clamp01=True)
                Image.fromarray(arr.cpu().numpy()).save(save_path)
            print(f"Writing output {save_path} ...")

    p = Path(args.img_path)
    if p.is_file():
        save_outputs(args.img_path, os.path.splitext(os.path.basename(args.img_path))[0])
    elif p.is_dir():
        for f in sorted(glob.glob(args.img_path + "/*")):
            save_outputs(f, os.path.splitext(os.path.basename(f))[0])
    else:
        print("invalid file path!")
        sys.exit()


if __name__ == "__main__":
    main()
