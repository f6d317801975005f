"""Golden vectors of the BEV backbone row (SURVEY 8 f-3), produced by the reference's OWN module.

Run in the build container (needs /root/reference or the oracle/_ref copy):  python tests/golden/make_golden_backbone.py
Each .npz holds the module config, its complete state dict (random weights, non-trivial BatchNorm statistics), a sparse
pillar-like canvas and the `spatial_features_2d` the unmodified `BaseBEVBackbone.forward` (base_bev_backbone.py:82-112)
returns for it on the CPU in fp32.  Weights are stored as float16-representable values to keep the files small (the module is
loaded with exactly these values on both sides, so nothing is lost).  A ``compact`` case stores instead of the state dict and
the canvas only their recipe (``pillar_oracle.golden_backbone_inputs`` on a module built after ``torch.manual_seed(seed)``), the
reference's state-dict keys in order and the SHA-256 of the inputs, so that no file exceeds 1 MB."""
import json
import os
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))
from oracle import pillar_oracle as po  # noqa: E402
from oracle import ref_loader as R  # noqa: E402

CASES = {
    "bb_2level_half_stride": dict(cfg=dict(LAYER_NUMS=[1, 1], LAYER_STRIDES=[2, 2], NUM_FILTERS=[64, 128],
                                           UPSAMPLE_STRIDES=[0.5, 1], NUM_UPSAMPLE_FILTERS=[128, 128]), h=48, w=40, nb=2, seed=1),
    "bb_3level_up124": dict(cfg=dict(LAYER_NUMS=[1, 1, 0], LAYER_STRIDES=[2, 2, 2], NUM_FILTERS=[64, 128, 256],
                                     UPSAMPLE_STRIDES=[1, 2, 4], NUM_UPSAMPLE_FILTERS=[64, 64, 64]), h=64, w=32, nb=1, seed=2, compact=True),
}


def main():
    BB = R.load_bev_backbone()
    for name, c in CASES.items():
        torch.manual_seed(c["seed"])
        m = BB(R.AttrDict(c["cfg"]), 64).eval()
        sd, canvas, sha = po.golden_backbone_inputs(m, c["seed"], c["nb"], c["h"], c["w"])
        with torch.inference_mode():
            out = m({"spatial_features": canvas.clone()})["spatial_features_2d"]
        save = {"cfg": np.frombuffer(json.dumps(c["cfg"]).encode(), dtype=np.uint8), "out": out.numpy()}
        if c.get("compact"):
            save.update({"gen.seed": np.int32(c["seed"]), "gen.shape": np.int32([c["nb"], c["h"], c["w"]]),
                         "sd_keys": np.frombuffer(json.dumps(list(sd)).encode(), np.uint8), "gen.sha256": sha})
        else:
            save["canvas"] = canvas.numpy().astype(np.float16)
            for k, v in sd.items():
                save["sd." + k] = v.numpy().astype(np.float16) if v.dtype == torch.float32 else v.numpy()
        path = os.path.join(HERE, name + ".npz")
        np.savez_compressed(path, **save)
        print(name, tuple(out.shape), os.path.getsize(path) // 1024, "KiB")


if __name__ == "__main__":
    main()
