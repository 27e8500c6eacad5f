"""Command lines of the reference, same flags: ``main.py --mode {train,predict,enhance}`` (main.py:25-117) and the
root ``simple_enhance.py`` (:17-42).  Only the enhance / predict modes are on the hot path; ``--mode train`` is the
reference's stock PyTorch trainer (out of scope) and is refused with a pointer to it."""
from __future__ import annotations

import argparse
import os

import torch


def _device(arg):
    """Device string of this process.  One process per GPU (torchrun): rank r of a node works on cuda:LOCAL_RANK -- the file
    list is sharded by RANK (enhancers/simple_enhance.py: shard_for_rank), so every rank must also sit on its own GPU."""
    dev = arg or ("cuda" if torch.cuda.is_available() else "cpu")
    if dev == "cuda" and torch.cuda.is_available():
        from .enhancers.simple_enhance import bind_rank_to_gpu
        return bind_rank_to_gpu()
    return dev


def _model(device, use_preact=False, use_aspp=False):
    from .models.model import UP_Retinex
    return UP_Retinex(use_preact=use_preact, use_aspp=use_aspp).to(device).eval()


def main_enhance(args):
    from .enhancers.adaptive_params import AdaptiveParameterAdjuster
    from .enhancers.simple_enhance import enhance_batch_images, enhance_single_image
    device = _device(args.device)
    if not args.input_path or not os.path.exists(args.input_path):
        raise SystemExit(f"错误: 输入路径 '{args.input_path}' 不存在")
    if os.path.isdir(args.input_path):
        enhance_batch_images(args.input_path, args.output_dir, device, args.max_size, args.multi_scale, args.content_aware,
                             model=_model(device, args.use_preact, args.use_aspp), amp=args.amp)
    else:
        enhance_single_image(_model(device, args.use_preact, args.use_aspp), args.input_path, args.output_dir, device,
                             args.max_size, args.multi_scale, args.content_aware, adjuster=AdaptiveParameterAdjuster(), amp=args.amp)


def main_predict(args):
    """main.py:150-206: refuses to run without a checkpoint file (a randomly initialised network would write plausible-looking
    *_enhanced.png files), then file or directory."""
    from .predictors import predict as P
    if not args.checkpoint or not os.path.exists(args.checkpoint):
        print(f"错误: 找不到模型检查点文件 '{args.checkpoint}'")
        print("请先训练模型或提供有效的检查点文件")
        return 1
    if not args.input_path or not os.path.exists(args.input_path):
        print(f"错误: 输入路径 '{args.input_path}' 不存在")
        return 1
    device = _device(args.device)
    os.makedirs(args.output_dir, exist_ok=True)
    print("正在加载模型...")
    model = _model("cpu", args.use_preact, args.use_aspp)
    P.load_checkpoint(model, args.checkpoint, "cpu")
    model = model.to(device).eval()
    print("模型加载完成")
    if os.path.isdir(args.input_path):
        P.predict_batch(model, args.input_path, args.output_dir, device, args.max_size, not args.no_comparison, amp=args.amp)
    else:
        P.predict_single_image(model, args.input_path, args.output_dir, device, args.max_size, not args.no_comparison, amp=args.amp)
    return 0


def build_main_parser():
    p = argparse.ArgumentParser(description="UP-Retinex (B200 hot path)")
    # defaults of the reference's main.py:29-44
    p.add_argument("--mode", type=str, default="predict", choices=["train", "predict", "enhance"])
    p.add_argument("--input_path", type=str, default="./data/test")
    p.add_argument("--output_dir", type=str, default="./results")
    p.add_argument("--checkpoint", type=str, default="./checkpoints/best_model.pth")
    p.add_argument("--max_size", type=int, default=None)
    p.add_argument("--device", type=str, default=None)
    p.add_argument("--multi_scale", action="store_true")
    p.add_argument("--content_aware", action="store_true")
    p.add_argument("--use_preact", action="store_true")
    p.add_argument("--use_aspp", action="store_true")
    p.add_argument("--no_comparison", action="store_true")
    p.add_argument("--amp", type=str, default=None, choices=["bf16", "fp16"], help="run the CNN under CUDA autocast")
    return p


def main(argv=None):
    args, _unknown = build_main_parser().parse_known_args(argv)   # training flags of main.py:31-75 are tolerated
    if args.mode == "train":
        raise SystemExit("--mode train is the reference's stock PyTorch trainer (out of scope of upretinex-b200); "
                         "its dynamic smoothness statistic lives in retinex_image_enhancement_b200.losses.loss")
    return main_predict(args) if args.mode == "predict" else main_enhance(args)


def simple_enhance_main(argv=None):
    p = argparse.ArgumentParser(description="UP-Retinex simple enhance (B200 hot path)")
    p.add_argument("--input", type=str, required=True)
    p.add_argument("--output", type=str, default="./results")
    p.add_argument("--max_size", type=int, default=None)
    p.add_argument("--device", type=str, default=None)
    p.add_argument("--multi_scale", action="store_true")
    p.add_argument("--content_aware", action="store_true")     # parsed AND forwarded (the reference drops it, :70-77)
    p.add_argument("--amp", type=str, default=None, choices=["bf16", "fp16"], help="run the CNN under CUDA autocast")
    a = p.parse_args(argv)
    ns = argparse.Namespace(input_path=a.input, output_dir=a.output, max_size=a.max_size, device=a.device,
                            multi_scale=a.multi_scale, content_aware=a.content_aware, use_preact=False, use_aspp=False, amp=a.amp)
    return main_enhance(ns)
