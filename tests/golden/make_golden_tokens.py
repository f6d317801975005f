"""Generates tests/golden/tok_*.npz by running the UNMODIFIED reference ``VATLiDAR`` (imported from /root/reference,
src/encoder-decoder/training/models/vat_lidar.py) and capturing the BEV K/V tokens its own forward hands to the first
VAT block (forward pre-hook on ``blocks[0]``; vat_lidar.py:206-253,285).

Run in the build container only:   python tests/golden/make_golden_tokens.py
Every file stores the reference's geometry tables (``_grid``: vat_lidar.py:123-185) and the tokens, with either the input
canvas and the tokeniser weights under the reference's state_dict keys, or (``compact``) only the recipe they are regenerated
from (``tokens_oracle.golden_token_inputs``) and the SHA-256 of those inputs; a compact case may keep the tokens of
its first ``keep`` frames only (frames are independent), so that no file exceeds 1 MB.
"""
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)

from oracle import ref_loader  # noqa: E402
from oracle import tokens_oracle as to  # noqa: E402

OUT = os.path.dirname(os.path.abspath(__file__))


def run_case(name, *, b, c, d, h, w, seed, occupancy, compact=False, keep=None):
    vat = ref_loader.load_vat_lidar()
    torch.manual_seed(seed)
    model = vat(c_in=c, d_model=d, n_queries=12, n_layers=1, n_heads=4).eval()
    bev, sd = to.golden_token_inputs(b, c, d, h, w, seed, occupancy)
    res = model.load_state_dict({k: torch.from_numpy(v) for k, v in sd.items()}, strict=False)
    assert not res.unexpected_keys and all(not k.startswith(to.TOKEN_KEYS) for k in res.missing_keys)
    tokens = ref_loader.vat_lidar_kv_tokens(model, torch.from_numpy(bev)).numpy()
    geom, sid = model._grid(h, w, torch.device("cpu"))
    save = {"out.tokens": tokens[:keep], "geom": geom.numpy(), "sid": sid.numpy().astype(np.int32),
            "c_in": np.int32(c), "d_model": np.int32(d)}
    if compact:
        save.update({"gen.batch": np.int32(b), "gen.hw": np.int32([h, w]), "gen.seed": np.int32(seed), "gen.occupancy": np.float64(occupancy),
                     "gen.sha256": to.golden_inputs_sha256(bev[:keep], sd)})
    else:
        save["bev"] = bev[:keep]
        for k, v in sd.items():
            save["sd." + k] = v
    path = os.path.join(OUT, name + ".npz")
    np.savez_compressed(path, **save)
    print(f"{name}: bev={bev[:keep].shape} tokens={tokens[:keep].shape} nonzero cells={(np.abs(bev).max(1) > 0).mean():.2f} "
          f"-> {os.path.getsize(path) / 1024:.0f} KiB")


def main():
    run_case("tok_c64_d128_16x16_dense", b=2, c=64, d=128, h=16, w=16, seed=0, occupancy=1.0)
    run_case("tok_c64_d256_24x20_sparse", b=3, c=64, d=256, h=24, w=20, seed=1, occupancy=0.07, compact=True, keep=2)
    run_case("tok_c32_d128_13x9_odd", b=2, c=32, d=128, h=13, w=9, seed=2, occupancy=0.3)
    run_case("tok_c128_d384_8x8", b=1, c=128, d=384, h=8, w=8, seed=3, occupancy=0.5)


if __name__ == "__main__":
    main()
