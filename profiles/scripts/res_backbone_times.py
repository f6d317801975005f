"""BaseBEVResBackbone on a B200: ms per 16 x 64 x 512^2 batch (pillar rows + index map of synthetic nuScenes sweeps, as
PillarVFEFromPoints(EMIT_INDEX_MAP) leaves them), algorithmic TFLOP/s from the shapes and the share of the 701 TFLOP/s
sustained tf32 figure of DESIGN.md 4e; the restatement (oracle/bev_res_oracle.py) eager with cuDNN TF32 on the same
input; and BaseBEVBackbone of this tree against an older tree (--base-tree), alternated process by process.

Every working set is far above the 126 MB of L2 (a level-0 activation alone is 1 GiB).  Times are CUDA events around one
forward, median of --calls after --warmup.  Writes one JSON file (--out).

    python profiles/scripts/res_backbone_times.py --out out/r05_res_backbone.json [--base-tree DIR]
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))

RES_CFG = dict(LAYER_NUMS=[1, 2, 2, 2], LAYER_STRIDES=[1, 2, 2, 2], NUM_FILTERS=[64, 128, 256, 256],
               UPSAMPLE_STRIDES=[0.5, 1, 2, 4], NUM_UPSAMPLE_FILTERS=[128, 128, 128, 128])
# the BaseBEVBackbone of bench.py's f-3 measurement (cbgs_pp_multihead.yaml)
PLAIN_CFG = dict(LAYER_NUMS=[3, 5, 5], LAYER_STRIDES=[2, 2, 2], NUM_FILTERS=[64, 128, 256], UPSAMPLE_STRIDES=[0.5, 1, 2],
                 NUM_UPSAMPLE_FILTERS=[128, 128, 128])
NB, C_IN, GRID = 16, 64, 512
SUSTAINED_TF32 = 701e12


def res_backbone_flops(cfg, c_in, h, w, nb):
    """Multiply-adds x 2 of every convolution of BaseBEVResBackbone on an h x w input: per level the first BasicBlock's
    1x1 projection and two 3x3 convolutions, LAYER_NUMS more blocks of two 3x3, then the up-sampling branch."""
    total, c, outs = 0.0, c_in, []
    for n, s, f in zip(cfg["LAYER_NUMS"], cfg["LAYER_STRIDES"], cfg["NUM_FILTERS"]):
        h, w = (h - 1) // s + 1, (w - 1) // s + 1
        px = nb * h * w
        total += 2.0 * px * f * c + 2.0 * px * f * c * 9 + 2.0 * px * f * f * 9
        total += n * 2 * (2.0 * px * f * f * 9)
        c = f
        outs.append((h, w, f))
    for (hh, ww, f), us, uf in zip(outs, cfg["UPSAMPLE_STRIDES"], cfg["NUM_UPSAMPLE_FILTERS"]):
        if us >= 1:
            total += 2.0 * nb * hh * ww * f * uf * us * us
        else:
            k = int(round(1 / us))
            total += 2.0 * nb * (hh // k) * (ww // k) * f * uf * k * k
    return total


def _inputs(torch, dev):
    import numpy as np

    from lidar_vision_vqa_b200 import synth
    from lidar_vision_vqa_b200.modules import PillarVFEFromPoints

    rng, vs = [-51.2, -51.2, -5.0, 51.2, 51.2, 3.0], [0.2, 0.2, 8.0]
    pts, offs = synth.make_batch(NB, synth.NUSCENES_32, 5, seed0=0)
    b = np.repeat(np.arange(NB), np.diff(offs)).astype(np.float32)[:, None]
    points = torch.from_numpy(np.concatenate([b, pts], axis=1)).to(dev)
    base = dict(USE_NORM=True, WITH_DISTANCE=False, USE_ABSLOTE_XYZ=True, NUM_FILTERS=[C_IN], MAX_POINTS_PER_VOXEL=32,
                MAX_NUMBER_OF_VOXELS=30000)
    torch.manual_seed(0)
    vfe = PillarVFEFromPoints(dict(base, EMIT_INDEX_MAP=True), 5, vs, rng, [GRID, GRID, 1]).eval().to(dev)
    vfe_c = PillarVFEFromPoints(dict(base, FUSE_SCATTER=True), 5, vs, rng, [GRID, GRID, 1]).eval().to(dev)
    vfe_c.load_state_dict(vfe.state_dict())
    with torch.inference_mode():
        d = vfe({"points": points, "batch_size": NB})
        canvas = vfe_c({"points": points, "batch_size": NB})["spatial_features"]
    return {"pillar_features": d["pillar_features"], "bev_index_map": d["bev_index_map"]}, canvas


def _median_ms(torch, fn, warmup, calls):
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    times = []
    for _ in range(calls):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        b.synchronize()
        times.append(a.elapsed_time(b))
    return statistics.median(times), min(times), max(times)


def _randomise_bn(torch, m, seed):
    g = torch.Generator().manual_seed(seed)
    with torch.no_grad():
        for mod in m.modules():
            if isinstance(mod, torch.nn.BatchNorm2d):
                mod.weight.copy_(0.5 + torch.rand(mod.weight.shape, generator=g))
                mod.bias.copy_(0.2 * torch.randn(mod.bias.shape, generator=g))
                mod.running_mean.copy_(0.2 * torch.randn(mod.bias.shape, generator=g))
                mod.running_var.copy_(0.5 + 1.5 * torch.rand(mod.bias.shape, generator=g))
    return m


def plain_child(tree, warmup, calls):
    """One BaseBEVBackbone timing with the package of ``tree`` (printed as JSON): run in a process of its own."""
    sys.path.insert(0, tree)
    from lidar_vision_vqa_b200 import build as _b

    _b.needs_build = lambda: False  # time the library that is there
    import torch

    from lidar_vision_vqa_b200.backbone import BaseBEVBackbone

    dev = torch.device("cuda:0")
    rows_map, _ = _inputs(torch, dev)
    torch.manual_seed(0)
    bb = _randomise_bn(torch, BaseBEVBackbone(PLAIN_CFG, C_IN), 1).eval().to(dev)
    with torch.inference_mode():
        med, lo, hi = _median_ms(torch, lambda: bb(dict(rows_map)), warmup, calls)
        out = bb(dict(rows_map))["spatial_features_2d"]
    torch.cuda.synchronize()
    import hashlib

    digest = hashlib.sha256(out.cpu().numpy().tobytes()).hexdigest()[:16]
    print(json.dumps(dict(tree=tree, ms_median=med, ms_min=lo, ms_max=hi, output_sha256_16=digest)))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--calls", type=int, default=25)
    ap.add_argument("--base-tree", default=None, help="an older checkout: BaseBEVBackbone before / after, alternated")
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--plain-child", default=None, help=argparse.SUPPRESS)
    args = ap.parse_args()
    if args.plain_child:
        plain_child(args.plain_child, args.warmup, args.calls)
        return
    sys.path.insert(0, ROOT)
    import torch

    from lidar_vision_vqa_b200 import BaseBEVResBackbone
    from oracle import bev_res_oracle as ro

    if not torch.cuda.is_available():
        raise SystemExit("no CUDA device: nothing measured")
    dev = torch.device("cuda:0")
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                         capture_output=True, text=True).stdout.strip()
    rec = dict(card=torch.cuda.get_device_name(dev), nvidia_smi=smi, batch=f"{NB} x {C_IN} x {GRID}^2", cfg=RES_CFG,
               warmup=args.warmup, calls=args.calls)
    rows_map, canvas = _inputs(torch, dev)
    rec["pillars"] = int(rows_map["pillar_features"].shape[0])
    rec["occupancy"] = rec["pillars"] / (NB * GRID * GRID)

    torch.manual_seed(0)
    ref = ro.randomise(ro.BaseBEVResBackbone(RES_CFG, C_IN), 1).eval().to(dev)
    mine = BaseBEVResBackbone(RES_CFG, C_IN).eval().to(dev)
    mine.load_state_dict(ref.state_dict(), strict=True)
    flops = res_backbone_flops(RES_CFG, C_IN, GRID, GRID, NB)
    with torch.inference_mode():
        med, lo, hi = _median_ms(torch, lambda: mine(dict(rows_map)), args.warmup, args.calls)
    rec["res_backbone"] = dict(ms_median=med, ms_min=lo, ms_max=hi, gflop=flops / 1e9, tflops=flops / (med * 1e-3) / 1e12,
                               share_of_701_tf32=flops / (med * 1e-3) / SUSTAINED_TF32)
    with torch.inference_mode():
        med, lo, hi = _median_ms(torch, lambda: mine({"spatial_features": canvas}), args.warmup, args.calls)
    rec["res_backbone_from_canvas"] = dict(ms_median=med, ms_min=lo, ms_max=hi)
    torch.backends.cudnn.allow_tf32 = True
    torch.backends.cudnn.benchmark = False
    with torch.inference_mode():
        med, lo, hi = _median_ms(torch, lambda: ref({"spatial_features": canvas}), args.warmup, args.calls)
    rec["restatement_eager_cudnn_tf32"] = dict(ms_median=med, ms_min=lo, ms_max=hi, tflops=flops / (med * 1e-3) / 1e12)
    del ref, mine, canvas, rows_map
    torch.cuda.empty_cache()

    if args.base_tree:
        ab = []  # (each entry's "tree" is the path given; the committed JSON labels them "parent commit" / "this change")
        for r in range(args.rounds):
            for tag, tree in (("before", os.path.abspath(args.base_tree)), ("after", ROOT)):
                p = subprocess.run([sys.executable, os.path.abspath(__file__), "--out", "-", "--plain-child", tree, "--warmup",
                                    str(args.warmup), "--calls", str(args.calls)], capture_output=True, text=True)
                if p.returncode != 0:
                    raise SystemExit(p.stderr[-3000:])
                ab.append(dict(json.loads(p.stdout.strip().splitlines()[-1]), side=tag, round=r))
        rec["base_bev_backbone_ab"] = ab
        for tag in ("before", "after"):
            rec[f"base_bev_backbone_{tag}_ms_median_of_rounds"] = statistics.median(x["ms_median"] for x in ab if x["side"] == tag)
        rec["base_bev_backbone_outputs_identical"] = len({x["output_sha256_16"] for x in ab}) == 1
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(rec, f, indent=1)
    print(json.dumps(rec))


if __name__ == "__main__":
    main()
