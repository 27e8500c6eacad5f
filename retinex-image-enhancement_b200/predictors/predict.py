"""Drop-in for the reference's ``predictors/predict.py`` inference drivers (:144-235) and CLI (:238-310).

The reference unpacks two values from a model that returns three (predict.py:163 vs models/model.py:455) and
raises ``ValueError``; this module unpacks ``(enhanced, reflectance, illu)``.  Output names and flags are the
reference's: ``--checkpoint --input --output --max_size --no_comparison --device``.
"""
from __future__ import annotations

import argparse
import os
import time

import numpy as np
import torch

from ..enhancers.adaptive_params import cnn_maps
from ..enhancers.simple_enhance import AMP_DTYPES, _to_u8_hwc, amp_context, list_images, load_image, save_image, shard_for_rank
from ..models.model import UP_Retinex


def create_comparison(img_low, img_enhanced, illu_map, save_path):
    """Three-panel strip input | enhanced | illumination (predict.py:100-141)."""
    from PIL import Image
    Image.fromarray(np.concatenate([_to_u8_hwc(img_low), _to_u8_hwc(img_enhanced), _to_u8_hwc(illu_map)], axis=1)).save(save_path)
    print(f"Saved comparison: {save_path}")


def predict_single_image(model, image_path, output_dir, device, max_size=None, save_comparison=True, amp=None):
    """amp: "fp16" / "bf16" runs the model under torch.autocast("cuda") (None: f32)."""
    img_low, _ = load_image(image_path, max_size, device=device)
    img_low = img_low.to(device)
    start = time.time()
    with torch.no_grad(), amp_context(amp):
        img_enhanced, _reflectance, illu_map = model(img_low)
    if img_enhanced.is_cuda:
        torch.cuda.synchronize(img_enhanced.device)
    print(f"Inference time: {time.time() - start:.4f}s")
    os.makedirs(output_dir, exist_ok=True)
    stem = os.path.splitext(os.path.basename(image_path))[0]
    save_image(img_enhanced, os.path.join(output_dir, f"{stem}_enhanced.png"))
    save_image(illu_map, os.path.join(output_dir, f"{stem}_illumination.png"))
    if save_comparison:
        create_comparison(img_low, img_enhanced, illu_map, os.path.join(output_dir, f"{stem}_comparison.png"))


def predict_batch(model, input_dir, output_dir, device, max_size=None, save_comparison=True, batch_size=16, amp=None):
    """predict.py:186-235 over the batch pipeline of enhancers/simple_enhance.py (SURVEY 8f row N1): files are decoded ahead of
    the GPU, same-shaped frames run as one device batch (uint8 up, uint8 enhanced + illumination down), PNGs are encoded on a
    thread pool.  Same three files per image as predict_single_image."""
    from ..enhancers.simple_enhance import resolve_device, run_batch_pipeline
    from .. import native
    amp_context(amp)   # an unknown amp fails before any file is read
    files = [f for f in list_images(input_dir) if os.path.splitext(f)[1].lower() in {".jpg", ".jpeg", ".png", ".bmp"}]
    if not files:
        print(f"No images found in {input_dir}")
        return
    device = resolve_device(device)
    mine = shard_for_rank(files)
    print(f"Found {len(files)} images ({len(mine)} on this rank)")
    t0 = time.time()

    def frame_fn(low):
        with torch.no_grad(), amp_context(amp):
            maps = cnn_maps(model, low)
            if maps is not None:
                # both stored frames in one pass over x and the maps: R and enhanced are never written
                return native.retinex_quantize_u8(low.contiguous(), *maps, autocast=torch.is_autocast_enabled("cuda"))
            enhanced, _reflectance, illu = model(low)
        # a map from a CNN under autocast is widened first, as _to_u8_hwc does
        return native.quantize_u8(enhanced.contiguous()), native.quantize_u8(illu.to(torch.float32).contiguous())

    def write_files(stem, low8, enh8, illu8):
        save_image(enh8, os.path.join(output_dir, f"{stem}_enhanced.png"))
        save_image(illu8, os.path.join(output_dir, f"{stem}_illumination.png"))
        if save_comparison:
            create_comparison(low8, enh8, illu8, os.path.join(output_dir, f"{stem}_comparison.png"))

    def host_fn(path, _arr):
        predict_single_image(model, path, output_dir, device, max_size, save_comparison, amp)

    run_batch_pipeline(mine, output_dir, device, max_size, batch_size, frame_fn, write_files, host_fn)
    total = time.time() - t0
    print(f"Total images processed: {len(mine)}\nTotal time: {total:.2f}s")
    if mine:
        print(f"Average time per image: {total / len(mine):.4f}s")


def load_checkpoint(model, checkpoint_path, device):
    """Checkpoints of the reference trainer (trainers/train.py:134-162): {'epoch', 'model_state_dict', 'optimizer_state_dict'};
    a bare state_dict is accepted too.  The module tree of models/model.py mirrors the reference's, so its keys load strictly;
    a checkpoint trained with other ``use_preact`` / ``use_aspp`` flags than the model was built with is reported as such."""
    if not os.path.exists(checkpoint_path):
        raise FileNotFoundError(f"Checkpoint not found: {checkpoint_path}")
    ckpt = torch.load(checkpoint_path, map_location=device)
    state = ckpt["model_state_dict"] if isinstance(ckpt, dict) and "model_state_dict" in ckpt else ckpt
    try:
        model.load_state_dict(state)
    except RuntimeError as e:
        has_aspp = any(".bottleneck.1.aspp_branches." in k for k in state)
        has_preact = any(k.endswith("enc1.bn1.weight") and state[k].shape[0] == 32 for k in state)
        raise RuntimeError(f"checkpoint {checkpoint_path} does not match the model's architecture flags: it looks like "
                           f"use_preact={has_preact}, use_aspp={has_aspp} (pass --use_preact / --use_aspp accordingly). "
                           f"Original error: {e}") from e
    if isinstance(ckpt, dict) and "epoch" in ckpt:
        print(f"Loaded checkpoint from epoch {ckpt['epoch']}")
    return model


def main(argv=None):
    p = argparse.ArgumentParser(description="UP-Retinex Inference")
    p.add_argument("--checkpoint", type=str, required=True)
    p.add_argument("--input", type=str, required=True)
    p.add_argument("--output", type=str, default="./results")
    p.add_argument("--max_size", type=int, default=None)
    p.add_argument("--no_comparison", action="store_true")
    p.add_argument("--device", type=str, default=None)
    p.add_argument("--amp", type=str, default=None, choices=sorted(AMP_DTYPES), help="run the CNN under CUDA autocast")
    args = p.parse_args(argv)
    from ..enhancers.simple_enhance import bind_rank_to_gpu
    device = args.device or ("cuda" if torch.cuda.is_available() else "cpu")
    if device == "cuda" and torch.cuda.is_available():
        device = bind_rank_to_gpu()
    model = UP_Retinex()
    load_checkpoint(model, args.checkpoint, "cpu")       # predict.py:282-288: a missing checkpoint is an error
    model = model.to(device).eval()
    if not os.path.exists(args.input):
        raise ValueError(f"Invalid input path: {args.input}")
    if os.path.isdir(args.input):
        predict_batch(model, args.input, args.output, device, args.max_size, not args.no_comparison, amp=args.amp)
    else:
        predict_single_image(model, args.input, args.output, device, args.max_size, not args.no_comparison, amp=args.amp)


if __name__ == "__main__":
    main()
