"""TEST INFRASTRUCTURE ONLY -- CPU restatement (numpy, float32) of the BEV tokeniser at the head of the reference's
``VATLiDAR.forward`` (src/encoder-decoder/training/models/vat_lidar.py), the first consumer of the BEV canvas
(SURVEY.md 8f-2).  Only tests/, ``__graft_entry__.smoke()`` and bench.py's checker legs import this file.

    grid_geometry   vat_lidar.py:123-185   (x, y, r, sin, cos) per cell and the 6-way sector id
    bev_tokens      vat_lidar.py:206-253   depthwise 3x3 + GELU -> 1x1 projection -> LayerNorm -> + geo PE -> + view embed

Pinned against the live reference class (tests/test_tokens_oracle.py, build container only) and against golden vectors
made by the reference's own forward (tests/golden/make_golden_tokens.py -> tok_*.npz).

Parameter names are the reference's state_dict keys: refine.0.{weight,bias}, proj.{weight,bias},
norm_tokens.{weight,bias}, geo_mlp.{0,2}.{weight,bias}, view_embed.
"""
from __future__ import annotations

import hashlib
import math

import numpy as np

NUM_VIEWS = 6
TOKEN_KEYS = ("refine.0.weight", "refine.0.bias", "proj.weight", "proj.bias", "norm_tokens.weight", "norm_tokens.bias",
              "geo_mlp.0.weight", "geo_mlp.0.bias", "geo_mlp.2.weight", "geo_mlp.2.bias", "view_embed")
LN_EPS = 1e-5  # nn.LayerNorm default (vat_lidar.py:89)

_erf = np.vectorize(math.erf, otypes=[np.float64])


def gelu(x: np.ndarray) -> np.ndarray:
    """nn.GELU() default = exact erf form (vat_lidar.py:84,96)."""
    x64 = x.astype(np.float64)
    return (0.5 * x64 * (1.0 + _erf(x64 / math.sqrt(2.0)))).astype(np.float32)


def _linspace(n: int) -> np.ndarray:
    """torch.linspace(-1, 1, n) in float32 as ATen's CPU kernel evaluates it: step = fl32(2/(n-1)); the first half counts
    up from -1, the second half down from +1, each value with ONE rounding (fused multiply-add) -- vat_lidar.py:140-141.
    The float64 product of a float32 and a small integer is exact, so rounding the float64 sum emulates the FMA."""
    if n == 1:
        return np.asarray([-1.0], np.float32)
    step = np.float64(np.float32(2.0) / np.float32(n - 1))
    i = np.arange(n)
    up = -1.0 + step * i
    down = 1.0 - step * (n - 1 - i)
    return np.where(i < n // 2, up, down).astype(np.float32)


def grid_geometry(h: int, w: int):
    """geom [h*w, 5] float32 and sector id [h*w] int64 (vat_lidar.py:139-183)."""
    yv, xv = np.meshgrid(_linspace(h), _linspace(w), indexing="ij")
    r = np.clip(np.sqrt(xv * xv + yv * yv, dtype=np.float32), 0.0, 1.0).astype(np.float32)
    theta = np.arctan2(yv, xv, dtype=np.float32)
    geom = np.stack([xv, yv, r, np.sin(theta, dtype=np.float32), np.cos(theta, dtype=np.float32)], -1).reshape(h * w, 5)
    ft = theta.reshape(-1)
    pi = np.float32(math.pi)  # the comparisons run in the tensor's dtype
    third, two3 = np.float32(math.pi / 3), np.float32(2 * math.pi / 3)
    sid = np.full(h * w, -1, np.int64)
    sid[(ft >= third) & (ft < two3)] = 0
    sid[(ft >= 0.0) & (ft < third)] = 1
    sid[(ft >= two3) & (ft <= pi)] = 2
    sid[(ft >= -two3) & (ft < -third)] = 3
    sid[(ft >= -third) & (ft < 0.0)] = 4
    sid[(ft >= -pi) & (ft < -two3)] = 5
    return geom.astype(np.float32), sid


def positional_table(sd, h: int, w: int, geom=None, sid=None) -> np.ndarray:
    """geo_mlp(geom) + view_embed[sid]: [h*w, d] (vat_lidar.py:229-245); float64 accumulation, rounded once."""
    if geom is None:
        geom, sid = grid_geometry(h, w)
    w1, b1 = sd["geo_mlp.0.weight"].astype(np.float64), sd["geo_mlp.0.bias"].astype(np.float64)
    w2, b2 = sd["geo_mlp.2.weight"].astype(np.float64), sd["geo_mlp.2.bias"].astype(np.float64)
    hid = gelu((geom.astype(np.float64) @ w1.T + b1).astype(np.float32)).astype(np.float64)
    pe = (hid @ w2.T + b2).astype(np.float32)
    return pe + sd["view_embed"][sid].astype(np.float32)


def refine(bev: np.ndarray, sd) -> np.ndarray:
    """Depthwise 3x3, padding 1, bias, then GELU (vat_lidar.py:82-85): [B,C,H,W] -> [B,C,H,W]."""
    b, c, h, w = bev.shape
    k = sd["refine.0.weight"].reshape(c, 3, 3).astype(np.float64)
    pad = np.zeros((b, c, h + 2, w + 2), np.float64)
    pad[:, :, 1:-1, 1:-1] = bev
    acc = np.zeros((b, c, h, w), np.float64)
    for dy in range(3):
        for dx in range(3):
            acc += pad[:, :, dy:dy + h, dx:dx + w] * k[None, :, dy, dx, None, None]
    acc += sd["refine.0.bias"].astype(np.float64)[None, :, None, None]
    return gelu(acc.astype(np.float32))


def layer_norm(x: np.ndarray, gamma, beta, eps=LN_EPS) -> np.ndarray:
    x64 = x.astype(np.float64)
    mu = x64.mean(-1, keepdims=True)
    var = ((x64 - mu) ** 2).mean(-1, keepdims=True)
    return ((x64 - mu) / np.sqrt(var + eps) * gamma.astype(np.float64) + beta.astype(np.float64)).astype(np.float32)


def bev_tokens(bev: np.ndarray, sd, geom=None, sid=None) -> np.ndarray:
    """[B,C,H,W] -> [B, H*W, d] (vat_lidar.py:206-245): the K/V tokens the VAT blocks attend over."""
    b, c, h, w = bev.shape
    x = refine(np.asarray(bev, np.float32), sd)
    wp = sd["proj.weight"].reshape(-1, c).astype(np.float64)  # [d, C]
    y = (x.transpose(0, 2, 3, 1).reshape(b, h * w, c).astype(np.float64) @ wp.T + sd["proj.bias"].astype(np.float64))
    y = layer_norm(y.astype(np.float32), sd["norm_tokens.weight"], sd["norm_tokens.bias"])
    return y + positional_table(sd, h, w, geom, sid)[None]


def background_token(sd) -> np.ndarray:
    """Token (before PE) of a cell whose 3x3 window holds only zeros: LN(proj(GELU(refine.bias))) -- what the sparse-aware
    kernel writes for such cells (follows from vat_lidar.py:82-90 with a zero input window)."""
    c = sd["refine.0.bias"].shape[0]
    a = gelu(sd["refine.0.bias"].astype(np.float32)).astype(np.float64)
    y = a @ sd["proj.weight"].reshape(-1, c).astype(np.float64).T + sd["proj.bias"].astype(np.float64)
    return layer_norm(y.astype(np.float32)[None], sd["norm_tokens.weight"], sd["norm_tokens.bias"])[0]


def random_token_params(c_in: int, d_model: int, seed: int):
    """Reference-keyed parameters with every tensor randomised (view_embed is zero-initialised in the reference,
    vat_lidar.py:101, which would hide the sector lookup)."""
    rng = np.random.default_rng(seed)

    def u(shape, s):
        return rng.uniform(-s, s, shape).astype(np.float32)

    return {
        "refine.0.weight": u((c_in, 1, 3, 3), 1.0 / 3.0), "refine.0.bias": u((c_in,), 1.0 / 3.0),
        "proj.weight": u((d_model, c_in, 1, 1), 1.0 / math.sqrt(c_in)), "proj.bias": u((d_model,), 0.3),
        "norm_tokens.weight": (1.0 + u((d_model,), 0.5)), "norm_tokens.bias": u((d_model,), 0.5),
        "geo_mlp.0.weight": u((d_model, 5), 1.0 / math.sqrt(5)), "geo_mlp.0.bias": u((d_model,), 0.4),
        "geo_mlp.2.weight": u((d_model, d_model), 1.0 / math.sqrt(d_model)), "geo_mlp.2.bias": u((d_model,), 0.2),
        "view_embed": u((NUM_VIEWS, d_model), 0.5),
    }


def golden_token_inputs(b: int, c: int, d: int, h: int, w: int, seed: int, occupancy: float):
    """The seeded canvas [b, c, h, w] and weights of a tests/golden/tok_*.npz case (tests/golden/make_golden_tokens.py).
    Below full occupancy it is a pillar canvas: most cells hold exact zeros in every channel, occupied ones are post-ReLU."""
    rng = np.random.default_rng(seed)
    bev = rng.standard_normal((b, c, h, w)).astype(np.float32)
    if occupancy < 1.0:
        occ = rng.random((b, 1, h, w)) < occupancy
        bev = np.where(occ, np.maximum(bev, 0.0), 0.0).astype(np.float32)
    return bev, random_token_params(c, d, seed + 7)


def golden_inputs_sha256(bev: np.ndarray, sd: dict) -> np.ndarray:
    """SHA-256 (32 uint8) of a canvas and its weights, weights in key order: pins the regenerated inputs of a compact golden."""
    h = hashlib.sha256(np.ascontiguousarray(bev).tobytes())
    for k in sorted(sd):
        h.update(np.ascontiguousarray(sd[k]).tobytes())
    return np.frombuffer(h.digest(), np.uint8)
