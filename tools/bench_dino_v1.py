"""Times the DINOv1 workload d1 -- ViTExtractor('dino_vits8', stride 4) at 224 x 298 (a 55 x 73 patch grid,
T = 4016 tokens), layer 11, facet 'key', then VLAD with K = 128 -- at batch 32 and batch 1, and prints one JSON
document (also written to --out):

  * device-timed images/s of extract_descriptors and of extract + VLAD.generate_multi, per-category device times
    from anyloc_profile_*, achieved TFLOP/s against 430.6 GFLOP/img (11 blocks + the key projection) and the
    attention share of time and FLOPs;
  * the log-bin kernel (bin=True): achieved bytes/s (read + 17x write) against 7.7 TB/s;
  * the reference's GPU path on the same card: the restated DINOv1 model in fp32 PyTorch at batch 1 (full
    forward + hook, as dino_extractor.py runs it), descriptors copied to the host, VLAD on the CPU;
  * parity of the timed outputs against the CPU oracle on 2 images;
  * the card name and its power limit, read in the same run.

    python tools/bench_dino_v1.py --steps 10 --warmup 3 --out profiles/r03_bench_dino_v1_d1.json
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from anyloc_b200 import _lib, dino_v1, utilities as u, vit  # noqa: E402
from oracle import anyloc_oracle as ao                     # noqa: E402
from oracle import dino_v1_restated as d1                  # noqa: E402

NAME, STRIDE, H, W, LAYER, FACET, K = "dino_vits8", 4, 224, 298, 11, "key", 128
HBM_PEAK = 7.7e12


def flops_per_image():
    """GEMM + attention FLOPs of blocks 0..10 plus the key projection of block 11 (multiply-add = 2)"""
    D, heads = 384, 6
    gh, gw = 1 + (H - 8) // STRIDE, 1 + (W - 8) // STRIDE
    T = gh * gw + 1
    patch = 2.0 * gh * gw * 192 * D
    block_gemm = 2.0 * T * D * (3 * D + D + 4 * D + 4 * D)
    attn = 4.0 * T * T * D
    return patch + LAYER * (block_gemm + attn) + 2.0 * T * D * D, LAYER * attn


def timed(fn, steps):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for i in range(steps):
        fn(i)
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / steps


def card():
    info = {"name": torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,power.max_limit,clocks.max.sm",
                            "--format=csv,noheader", "-i", str(torch.cuda.current_device())],
                           capture_output=True, text=True, timeout=30).stdout.strip()
        info["power_limit, power_max_limit, sm_clock_max"] = q
    except Exception as e:          # the query is informational; the numbers stand without it
        info["query_error"] = f"{type(e).__name__}: {e}"
    return info


def profile(fn, n=3):
    _lib.profile_enable(True)
    ms = timed(fn, n)
    prof = _lib.profile_read()
    _lib.profile_enable(False)
    return ms, {c: {"ms_per_step": v[0] / n, "groups_per_step": v[1] / n, "work_per_step": v[2] / n}
                for c, v in prof.items() if v[1]}


def run_batch(ext, vlad, B, steps, warmup, gflop, attn_gflop):
    img = torch.randn(B, 3, H, W, generator=torch.Generator().manual_seed(B)).cuda()
    extract = lambda i: ext.extract_descriptors(img, LAYER, FACET)
    pipeline = lambda i: vlad.generate_multi(ext.extract_descriptors(img, LAYER, FACET).squeeze(1))
    for _ in range(warmup):
        pipeline(0)
    torch.cuda.synchronize()
    ms_ext = timed(extract, steps)
    ms_pipe = timed(pipeline, steps)
    _, prof = profile(extract)
    attn_ms = prof.get("attention", {}).get("ms_per_step", 0.0)
    dev_ms = sum(v["ms_per_step"] for v in prof.values())
    ext.raise_if_overflowed()
    return img, {
        "batch": B,
        "extract_ms": ms_ext, "extract_img_per_s": B * 1e3 / ms_ext,
        "extract_vlad_ms": ms_pipe, "extract_vlad_img_per_s": B * 1e3 / ms_pipe,
        "achieved_tflops": B * gflop / ms_ext,                      # GFLOP / ms = TFLOP/s
        "attention": {"flop_share": attn_gflop / gflop, "time_share_of_profiled_device_time": attn_ms / dev_ms,
                      "achieved_tflops": B * attn_gflop / attn_ms if attn_ms else None},
        "profile": prof,
    }


def log_bin_rate(ext, steps):
    img = torch.randn(32, 3, H, W, generator=torch.Generator().manual_seed(3)).cuda()
    ext.extract_descriptors(img, LAYER, FACET, bin=True)
    _, prof = profile(lambda i: ext.extract_descriptors(img, LAYER, FACET, bin=True))
    lb = prof["log_bin"]
    gh, gw = ext.num_patches
    x = torch.randn(32, gh * gw, 384, device="cuda")
    ms = timed(lambda i: dino_v1.log_bin(x, gh, gw), steps)
    nbytes = 18.0 * 4 * x.numel()
    return {"batch": 32, "out_shape": [32, 1, gh * gw, 17 * 384],
            "in_pipeline_ms": lb["ms_per_step"], "in_pipeline_bytes_per_s": lb["work_per_step"] / lb["ms_per_step"] * 1e3,
            "alone_ms": ms, "alone_bytes_per_s": nbytes / ms * 1e3, "fraction_of_7.7TB/s": nbytes / ms * 1e3 / HBM_PEAK}


def reference_gpu_path(sd, centers, n_img):
    """restated fp32 model on the GPU at batch 1 with the reference's key hook, .cpu(), CPU VLAD"""
    model = d1.from_state_dict(sd, NAME).cuda()
    model.patch_embed.proj.stride = (STRIDE, STRIDE)
    model.interpolate_pos_encoding = lambda x, w, h: d1.pos_encoding(model, 1 + (w - 8) // STRIDE,
                                                                     1 + (h - 8) // STRIDE, w, h)
    feats = []

    def hook(mod, inp, out):
        x = inp[0]
        B, N, C = x.shape
        feats.append(mod.qkv(x).reshape(B, N, 3, mod.num_heads, C // mod.num_heads).permute(2, 0, 3, 1, 4)[1])
    h = model.blocks[LAYER].attn.register_forward_hook(hook)
    imgs = torch.randn(n_img, 3, H, W, generator=torch.Generator().manual_seed(9))
    times = []
    with torch.no_grad():
        for i in range(n_img + 1):
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            feats.clear()
            model(imgs[i % n_img][None].cuda())
            desc = feats[0][:, :, 1:].permute(0, 2, 3, 1).flatten(-2).cpu()[0]
            ao.vlad_generate(desc, centers)
            if i:
                times.append(time.perf_counter() - t0)
    h.remove()
    return {"img_per_s": 1.0 / float(np.mean(times)), "ms_per_img": 1e3 * float(np.mean(times)), "images": n_img,
            "what": "restated DINOv1 fp32 (torch.backends tf32 off) batch 1, full forward + key hook, .cpu(), "
                    "oracle VLAD on the host"}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--precision", default="f16x3", choices=["f16x3", "tf32x3"])
    ap.add_argument("--ref-images", type=int, default=4)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    torch.cuda.set_device(0)
    gflop, attn_gflop = (f / 1e9 for f in flops_per_image())
    sd = vit.random_state_dict(NAME, seed=0, device="cuda")
    ext = dino_v1.ViTExtractor(NAME, STRIDE, device="cuda", weights=sd, precision=args.precision)
    ext.check_finite = "deferred"
    # vocabulary from 4 images' descriptors (what VLAD.fit would leave; fit itself is not timed)
    voc = torch.randn(4, 3, H, W, generator=torch.Generator().manual_seed(1)).cuda()
    np.random.seed(0)
    vlad = u.VLAD(K)
    vlad.fit(ext.extract_descriptors(voc, LAYER, FACET).reshape(-1, 384))
    res = {"workload": "d1: dino_vits8 stride 4, 224x298 (55x73 grid, T=4016), layer 11 key, VLAD K=128",
           "precision": args.precision, "gflop_per_img": gflop, "attention_gflop_per_img": attn_gflop,
           "card": card()}
    img32, res["b32"] = run_batch(ext, vlad, 32, args.steps, args.warmup, gflop, attn_gflop)
    _, res["b1"] = run_batch(ext, vlad, 1, args.steps, args.warmup, gflop, attn_gflop)
    res["log_bin"] = log_bin_rate(ext, args.steps)
    # parity of the timed outputs (batch 32, images 0 and 31) against the CPU oracle
    out = ext.extract_descriptors(img32, LAYER, FACET)[[0, 31]].cpu()
    model = d1.from_state_dict(sd, NAME)
    ref = d1.extract_descriptors(model, img32[[0, 31]].cpu(), STRIDE, LAYER, FACET)
    res["parity_rel_inf_vs_oracle_2img"] = float((out - ref).abs().max() / ref.abs().max())
    res["reference_gpu_path_b1"] = reference_gpu_path(sd, vlad.c_centers.cpu(), args.ref_images)
    res["speedup_b32_extract_vlad_vs_reference"] = res["b32"]["extract_vlad_img_per_s"] / \
        res["reference_gpu_path_b1"]["img_per_s"]
    res["card_after"] = card()
    text = json.dumps(res, indent=1)
    print(text)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
