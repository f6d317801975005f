"""TEST INFRASTRUCTURE ONLY -- CPU oracle for the pillar hot path.

Only ``tests/``, ``__graft_entry__.smoke()`` and ``bench.py``'s ``cpu_baseline`` / ``--impl reference`` legs may
import this module, and only as the checker / the CPU baseline.  ``lidar_vision_vqa_b200`` never imports it.

Pieces (each cites the reference lines it restates; paths relative to ``src/lidar-encoder/pcdet``):

* :func:`voxelize_hard` / :func:`voxelize_hard_py` -- hard voxelisation.  The reference delegates to spconv
  (``datasets/processor/data_processor.py:16-61,133-180``), which is NOT vendored; restated in
  ``oracle/voxelize_ref.c`` from spconv's published loop.  *Ordering semantics: parity unpinned* (see that file).
* :func:`collate_voxels` -- batch-index column + concatenation (``datasets/dataset.py:232-244``) and the
  float32 cast of ``models/__init__.py:36``.
* :func:`pillar_vfe` -- ``models/backbones_3d/vfe/pillar_vfe.py:29-49`` (PFNLayer.forward) and ``:94-123``
  (PillarVFE.forward), fp32 torch on CPU.  *Pinned*: checked against the reference module itself
  (``tests/golden/*.npz`` made by ``tests/golden/make_golden.py`` in the build container).
* :func:`scatter_bev` -- ``models/backbones_2d/map_to_bev/pointpillar_scatter.py:14-37``.  *Pinned* likewise.
* :func:`dynamic_pillar_vfe` -- ``models/backbones_3d/vfe/dynamic_pillar_vfe.py:35-46,90-142`` (DynamicPillarVFE +
  PFNLayerV2) and ``:193-240`` (DynamicPillarVFESimple2D) restated with plain torch index ops.  *Pinned* against the
  reference modules' goldens (``dyn_*.npz``).
* :func:`dynamic_pillar_sets` -- the on-device quantisation of
  ``models/backbones_3d/vfe/dynamic_pillar_vfe.py:93-103`` (set of pillars + counts), used as a second opinion
  for the voxeliser's quantisation.  *Pinned* against the reference DynamicPillarVFE golden.
"""
from __future__ import annotations

import ctypes
import hashlib
import os
import subprocess
from typing import Dict, List, Optional, Sequence, Tuple

import numpy as np
import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
_SO = os.path.join(_HERE, "_build", "liboracle_pillars.so")
_LIB = None


def build_oracle_lib(force: bool = False) -> str:
    src = os.path.join(_HERE, "voxelize_ref.c")
    if force or not os.path.isfile(_SO) or os.path.getmtime(_SO) < os.path.getmtime(src):
        subprocess.check_call(["make", "-C", _HERE, "-B" if force else "-s"], stdout=subprocess.DEVNULL)
    return _SO


def _lib():
    global _LIB
    if _LIB is None:
        lib = ctypes.CDLL(build_oracle_lib())
        fp = ctypes.POINTER(ctypes.c_float)
        ip = ctypes.POINTER(ctypes.c_int32)
        lib.oracle_voxelize_hard.restype = ctypes.c_int
        lib.oracle_voxelize_hard.argtypes = [fp, ctypes.c_int64, ctypes.c_int, fp, fp, ip, ctypes.c_int,
                                             ctypes.c_int, fp, ip, ip, ip, ip]
        lib.oracle_scatter_bev.restype = ctypes.c_int
        lib.oracle_scatter_bev.argtypes = [fp, ip, ctypes.c_int64, ctypes.c_int, ctypes.c_int, ctypes.c_int,
                                           ctypes.c_int, ctypes.c_int, fp]
        _LIB = lib
    return _LIB


def _fptr(a):
    return a.ctypes.data_as(ctypes.POINTER(ctypes.c_float)) if a is not None else None


def _iptr(a):
    return a.ctypes.data_as(ctypes.POINTER(ctypes.c_int32)) if a is not None else None


def grid_size_of(point_cloud_range: Sequence[float], voxel_size: Sequence[float]) -> np.ndarray:
    """data_processor.py:135-136 -- float64 numpy arithmetic, then round."""
    r = np.asarray(point_cloud_range, dtype=np.float64)
    g = (r[3:6] - r[0:3]) / np.asarray(voxel_size, dtype=np.float64)
    return np.round(g).astype(np.int64)


# --------------------------------------------------------------------------------------------------
# hard voxelisation
# --------------------------------------------------------------------------------------------------
def voxelize_hard(points: np.ndarray, point_cloud_range, voxel_size, max_points: int, max_voxels: int,
                  want_voxels: bool = True):
    """One frame through the C restatement.  Returns a dict with
    ``voxels [M,P,C] f32`` (or None), ``coords [M,3] i32 (z,y,x)``, ``num_points [M] i32``,
    ``point_voxel [N] i32`` and ``point_slot [N] i32`` (-1 = not stored)."""
    pts = np.ascontiguousarray(points, dtype=np.float32)
    n, c = pts.shape
    rng = np.asarray(point_cloud_range, dtype=np.float32)
    vs = np.asarray(voxel_size, dtype=np.float32)
    grid = grid_size_of(point_cloud_range, voxel_size).astype(np.int32)
    cap = int(min(max_voxels, max(n, 1)))
    voxels = np.empty((cap, max_points, c), dtype=np.float32) if want_voxels else None
    coords = np.zeros((cap, 3), dtype=np.int32)
    npts = np.zeros((cap,), dtype=np.int32)
    pv = np.empty((n,), dtype=np.int32)
    ps = np.empty((n,), dtype=np.int32)
    m = _lib().oracle_voxelize_hard(_fptr(pts), n, c, _fptr(rng), _fptr(vs), _iptr(grid), int(max_points), cap,
                                    _fptr(voxels), _iptr(coords), _iptr(npts), _iptr(pv), _iptr(ps))
    if m < 0:
        raise RuntimeError("oracle_voxelize_hard: bad arguments")
    return {
        "voxels": voxels[:m] if want_voxels else None,
        "coords": coords[:m],
        "num_points": npts[:m],
        "point_voxel": pv,
        "point_slot": ps,
    }


def voxelize_hard_py(points: np.ndarray, point_cloud_range, voxel_size, max_points: int, max_voxels: int):
    """Same algorithm as ``oracle/voxelize_ref.c`` as a pure-Python loop with numpy float32 scalars -- small inputs
    only; exists so the C restatement is itself double-checked by an independent transcription."""
    pts = np.asarray(points, dtype=np.float32)
    rng = np.asarray(point_cloud_range, dtype=np.float32)
    vs = np.asarray(voxel_size, dtype=np.float32)
    grid = grid_size_of(point_cloud_range, voxel_size)
    table: Dict[Tuple[int, int, int], int] = {}
    coords: List[Tuple[int, int, int]] = []
    members: List[List[int]] = []
    pv = np.full(len(pts), -1, np.int32)
    ps = np.full(len(pts), -1, np.int32)
    for i in range(len(pts)):
        c3 = []
        for j in range(3):
            f = np.floor(np.float32(np.float32(pts[i, j] - rng[j]) / vs[j]))
            if not (f >= 0 and f < grid[j]):
                break
            c3.append(int(f))
        if len(c3) < 3:
            continue
        key = (c3[2], c3[1], c3[0])
        vid = table.get(key, -1)
        if vid < 0:
            if len(coords) >= max_voxels:
                continue
            vid = len(coords)
            table[key] = vid
            coords.append(key)
            members.append([])
        pv[i] = vid
        if len(members[vid]) < max_points:
            ps[i] = len(members[vid])
            members[vid].append(i)
    m = len(coords)
    voxels = np.zeros((m, max_points, pts.shape[1]), np.float32)
    npts = np.zeros((m,), np.int32)
    for v, idxs in enumerate(members):
        voxels[v, :len(idxs)] = pts[idxs]
        npts[v] = len(idxs)
    return {"voxels": voxels, "coords": np.asarray(coords, np.int32).reshape(m, 3), "num_points": npts,
            "point_voxel": pv, "point_slot": ps}


def voxelize_batch(points: np.ndarray, frame_offsets: np.ndarray, point_cloud_range, voxel_size, max_points: int,
                   max_voxels: int, want_voxels: bool = True):
    """All frames of a packed batch + the collate step (dataset.py:232-244): ``coords`` becomes ``[sum M, 4]``
    ``(b,z,y,x)``; ``point_voxel`` becomes the row in the concatenated arrays (or -1)."""
    outs = []
    base = 0
    pv_all = np.full(points.shape[0], -1, np.int32)
    ps_all = np.full(points.shape[0], -1, np.int32)
    counts = []
    for b in range(len(frame_offsets) - 1):
        lo, hi = int(frame_offsets[b]), int(frame_offsets[b + 1])
        o = voxelize_hard(points[lo:hi], point_cloud_range, voxel_size, max_points, max_voxels, want_voxels)
        m = o["coords"].shape[0]
        pv = o["point_voxel"]
        pv_all[lo:hi] = np.where(pv >= 0, pv + base, -1)
        ps_all[lo:hi] = o["point_slot"]
        o["coords4"] = np.concatenate([np.full((m, 1), b, np.int32), o["coords"]], axis=1)
        outs.append(o)
        counts.append(m)
        base += m
    return {
        "voxels": np.concatenate([o["voxels"] for o in outs], 0) if want_voxels else None,
        "coords": np.concatenate([o["coords4"] for o in outs], 0),
        "num_points": np.concatenate([o["num_points"] for o in outs], 0),
        "point_voxel": pv_all,
        "point_slot": ps_all,
        "pillars_per_frame": np.asarray(counts, np.int32),
    }


def golden_backbone_inputs(module: torch.nn.Module, seed: int, nb: int, h: int, w: int):
    """The inputs of a tests/golden/bb_*.npz case (tests/golden/make_golden_backbone.py) for a BaseBEVBackbone built right
    after ``torch.manual_seed(seed)``: non-trivial BatchNorm statistics, every float parameter rounded to float16, and a
    sparse pillar-like canvas [nb, 64, h, w] of float16 values.  Updates ``module`` in place; returns its state dict, the
    canvas (float32) and the SHA-256 (32 uint8) of both, parameters in state-dict order."""
    g = torch.Generator().manual_seed(seed + 100)
    with torch.no_grad():
        for mod in module.modules():
            if isinstance(mod, torch.nn.BatchNorm2d):
                mod.weight.copy_(0.5 + torch.rand(mod.weight.shape, generator=g))
                mod.bias.copy_(0.2 * torch.randn(mod.bias.shape, generator=g))
                mod.running_mean.copy_(0.2 * torch.randn(mod.bias.shape, generator=g))
                mod.running_var.copy_(0.5 + 1.5 * torch.rand(mod.bias.shape, generator=g))
        for v in module.state_dict().values():
            if v.dtype == torch.float32:
                v.copy_(v.half().float())
    occ = torch.rand((nb, 1, h, w), generator=g) < 0.08
    canvas = (torch.rand((nb, 64, h, w), generator=g) * occ).half().float()
    sd = module.state_dict()
    digest = hashlib.sha256()
    for v in list(sd.values()) + [canvas]:
        digest.update((v.half() if v.dtype == torch.float32 else v).numpy().tobytes())
    return sd, canvas, np.frombuffer(digest.digest(), np.uint8)


# --------------------------------------------------------------------------------------------------
# pillar feature net
# --------------------------------------------------------------------------------------------------
def random_pfn_params(c_in: int, num_filters: Sequence[int], use_norm: bool = True, seed: int = 0):
    """Randomised weights AND BatchNorm running statistics -- default-initialised BN hides the padded-slot term
    (SURVEY.md section 7).  Returned as a state_dict with the reference's keys (pillar_vfe.py:21-25,74)."""
    g = torch.Generator().manual_seed(seed)
    sd = {}
    dims = [c_in] + list(num_filters)
    for i in range(len(dims) - 1):
        last = i >= len(dims) - 2
        out = dims[i + 1] if last else dims[i + 1] // 2
        fan_in = dims[i]
        sd[f"pfn_layers.{i}.linear.weight"] = (torch.rand(out, fan_in, generator=g) * 2 - 1) / fan_in ** 0.5
        if use_norm:
            sd[f"pfn_layers.{i}.norm.weight"] = torch.rand(out, generator=g) + 0.5
            sd[f"pfn_layers.{i}.norm.bias"] = torch.randn(out, generator=g) * 0.5
            sd[f"pfn_layers.{i}.norm.running_mean"] = torch.randn(out, generator=g) * 0.5
            sd[f"pfn_layers.{i}.norm.running_var"] = torch.rand(out, generator=g) * 1.5 + 0.5
            sd[f"pfn_layers.{i}.norm.num_batches_tracked"] = torch.tensor(100, dtype=torch.long)
        else:
            sd[f"pfn_layers.{i}.linear.bias"] = torch.randn(out, generator=g) * 0.3
    return sd


def _pfn_layer(x: torch.Tensor, sd: dict, i: int, use_norm: bool, last: bool) -> torch.Tensor:
    """pillar_vfe.py:29-49.  x is [M,P,Cin]."""
    w = sd[f"pfn_layers.{i}.linear.weight"].float()
    y = x @ w.t()  # Linear; the 50 000-row chunking at :30-37 is numerically neutral
    if use_norm:
        gamma = sd[f"pfn_layers.{i}.norm.weight"].float()
        beta = sd[f"pfn_layers.{i}.norm.bias"].float()
        mu = sd[f"pfn_layers.{i}.norm.running_mean"].float()
        var = sd[f"pfn_layers.{i}.norm.running_var"].float()
        y = (y - mu) / torch.sqrt(var + 1e-3) * gamma + beta  # BatchNorm1d eval, eps=1e-3 (:23)
    else:
        y = y + sd[f"pfn_layers.{i}.linear.bias"].float()
    y = torch.relu(y)
    y_max = y.max(dim=1, keepdim=True)[0]  # padded rows take part in the max (:42)
    if last:
        return y_max
    return torch.cat([y, y_max.expand(-1, x.shape[1], -1)], dim=2)  # :46-49, padded rows NOT re-masked


def pillar_vfe(voxels, num_points, coords, state_dict: dict, voxel_size, point_cloud_range,
               use_norm: bool = True, with_distance: bool = False, use_absolute_xyz: bool = True) -> torch.Tensor:
    """pillar_vfe.py:94-123 on CPU in fp32.  ``coords`` is ``[M,4] (b,z,y,x)``, any of int32/float32;
    ``num_points`` int32/float32.  Returns ``[M, F]`` (the reference additionally ``squeeze()``-es, so M == 1
    gives ``[F]`` there)."""
    v = torch.as_tensor(voxels, dtype=torch.float32)
    n = torch.as_tensor(num_points)
    c = torch.as_tensor(coords)
    vx, vy, vz = (float(s) for s in voxel_size)
    # ctor :76-81 -- python float arithmetic
    x_off = vx / 2 + float(point_cloud_range[0])
    y_off = vy / 2 + float(point_cloud_range[1])
    z_off = vz / 2 + float(point_cloud_range[2])
    xyz = v[:, :, :3]
    mean = xyz.sum(dim=1, keepdim=True) / n.to(v.dtype).view(-1, 1, 1)  # :97 (sum over ALL P slots)
    f_cluster = xyz - mean  # :98
    cf = c.to(v.dtype)
    f_center = torch.stack([
        xyz[:, :, 0] - (cf[:, 3].unsqueeze(1) * vx + x_off),  # :101
        xyz[:, :, 1] - (cf[:, 2].unsqueeze(1) * vy + y_off),  # :102
        xyz[:, :, 2] - (cf[:, 1].unsqueeze(1) * vz + z_off),  # :103
    ], dim=-1)
    parts = [v if use_absolute_xyz else v[..., 3:], f_cluster, f_center]  # :105-108
    if with_distance:
        parts.append(torch.linalg.vector_norm(xyz, ord=2, dim=2, keepdim=True))  # :110-112
    feats = torch.cat(parts, dim=-1)
    p = feats.shape[1]
    mask = (n.int().view(-1, 1) > torch.arange(p, dtype=torch.int32).view(1, -1)).to(v.dtype)  # :86-92
    feats = feats * mask.unsqueeze(-1)  # :115-118
    n_layers = len([k for k in state_dict if k.endswith("linear.weight")])
    for i in range(n_layers):
        feats = _pfn_layer(feats, state_dict, i, use_norm, last=(i == n_layers - 1))
    return feats[:, 0, :]


def collate_voxels(v: dict, as_float: bool = True):
    """What the model sees after ``load_data_to_gpu`` (models/__init__.py:36): every array float32."""
    if not as_float:
        return v["voxels"], v["num_points"], v["coords"]
    return v["voxels"], v["num_points"].astype(np.float32), v["coords"].astype(np.float32)


# --------------------------------------------------------------------------------------------------
# BEV scatter
# --------------------------------------------------------------------------------------------------
def scatter_bev(pillar_features, coords, nx: int, ny: int, batch_size: Optional[int] = None, nz: int = 1) -> np.ndarray:
    """pointpillar_scatter.py:14-37 (nz == 1) and :40-73 (PointPillarScatter3d, nz > 1 -> ``[B, F*nz, ny, nx]``).
    ``batch_size`` None reproduces the reference's ``coords[:,0].max()+1`` (:17).  Runs the C restatement."""
    f = np.ascontiguousarray(np.asarray(pillar_features, dtype=np.float32))
    c = np.ascontiguousarray(np.asarray(coords).astype(np.int32))
    nb = int(c[:, 0].max()) + 1 if batch_size is None else int(batch_size)
    bev = np.empty((nb, f.shape[1] * nz, ny, nx), dtype=np.float32)
    rc = _lib().oracle_scatter_bev(_fptr(f), _iptr(c), f.shape[0], nb, f.shape[1], nx, ny, nz, _fptr(bev))
    if rc != 0:
        raise RuntimeError(f"oracle_scatter_bev failed: {rc}")
    return bev


# --------------------------------------------------------------------------------------------------
# dynamic (on-device) quantisation, set level
# --------------------------------------------------------------------------------------------------
def dynamic_pillar_sets(points_b: np.ndarray, point_cloud_range, voxel_size):
    """dynamic_pillar_vfe.py:93-103: ``floor((xy - min) / v).int()``, x/y range mask only, merged key
    ``b*nx*ny + ix*ny + iy``, unique + counts.  ``points_b`` is ``[N, 1+C]`` with the batch index first.
    Returns ``(coords [M,4] (b,0,iy,ix) i32 sorted by key, counts [M] i64)``."""
    p = torch.as_tensor(points_b, dtype=torch.float32)
    rng = torch.tensor(np.asarray(point_cloud_range, dtype=np.float32))  # torch.tensor(list).cuda() -> fp32
    vs = torch.tensor(np.asarray(voxel_size, dtype=np.float32))
    grid = torch.tensor(grid_size_of(point_cloud_range, voxel_size))
    ij = torch.floor((p[:, [1, 2]] - rng[[0, 1]]) / vs[[0, 1]]).int()
    ok = ((ij >= 0) & (ij < grid[[0, 1]])).all(dim=1)
    p, ij = p[ok], ij[ok]
    sxy, sy = int(grid[0] * grid[1]), int(grid[1])
    key = p[:, 0].int() * sxy + ij[:, 0] * sy + ij[:, 1]
    uq, cnt = torch.unique(key, return_counts=True)
    uq = uq.int()
    coords = torch.stack([uq // sxy, torch.zeros_like(uq), uq % sy, (uq % sxy) // sy], dim=1)
    return coords.numpy().astype(np.int32), cnt.numpy()


def _pfn_layer_v2(x: torch.Tensor, inv: torch.Tensor, m: int, sd: dict, i: int, use_norm: bool, last: bool) -> torch.Tensor:
    """dynamic_pillar_vfe.py:35-46 (PFNLayerV2.forward): x is [N, Cin], inv [N] the pillar of each point."""
    y = x @ sd[f"pfn_layers.{i}.linear.weight"].float().t()
    if use_norm:
        gamma = sd[f"pfn_layers.{i}.norm.weight"].float()
        beta = sd[f"pfn_layers.{i}.norm.bias"].float()
        mu = sd[f"pfn_layers.{i}.norm.running_mean"].float()
        var = sd[f"pfn_layers.{i}.norm.running_var"].float()
        y = (y - mu) / torch.sqrt(var + 1e-3) * gamma + beta
    else:
        y = y + sd[f"pfn_layers.{i}.linear.bias"].float()
    y = torch.relu(y)
    y_max = torch.full((m, y.shape[1]), float("-inf"), dtype=y.dtype)
    y_max = y_max.scatter_reduce(0, inv.view(-1, 1).expand_as(y), y, reduce="amax", include_self=True)  # scatter_max :40
    if last:
        return y_max
    return torch.cat([y, y_max[inv]], dim=1)  # :44-45


def dynamic_pillar_vfe(points_b, state_dict: dict, voxel_size, point_cloud_range, use_norm: bool = True,
                       with_distance: bool = False, use_absolute_xyz: bool = True, simple2d: bool = False):
    """DynamicPillarVFE.forward (dynamic_pillar_vfe.py:90-142) or, with ``simple2d``, DynamicPillarVFESimple2D.forward
    (:193-240) on CPU in fp32.  Returns ``(pillar_features [M,F], coords)`` with coords ``[M,4] (b,0,iy,ix)`` or, for
    simple2d, ``[M,3] (b,iy,ix)``; rows sorted by the merged key."""
    p = torch.as_tensor(points_b, dtype=torch.float32)
    rng = torch.tensor(np.asarray(point_cloud_range, dtype=np.float32))
    vs = torch.tensor(np.asarray(voxel_size, dtype=np.float32))
    grid = torch.tensor(grid_size_of(point_cloud_range, voxel_size))
    vx, vy, vz = (float(v) for v in voxel_size)
    x_off = vx / 2 + float(point_cloud_range[0])
    y_off = vy / 2 + float(point_cloud_range[1])
    z_off = vz / 2 + float(point_cloud_range[2])
    ij = torch.floor((p[:, [1, 2]] - rng[[0, 1]]) / vs[[0, 1]]).int()  # :93
    ok = ((ij >= 0) & (ij < grid[[0, 1]])).all(dim=1)  # :94
    p, ij = p[ok], ij[ok]
    xyz = p[:, [1, 2, 3]].contiguous()
    sxy, sy = int(grid[0] * grid[1]), int(grid[1])
    key = p[:, 0].int() * sxy + ij[:, 0] * sy + ij[:, 1]  # :99-101
    uq, inv, cnt = torch.unique(key, return_inverse=True, return_counts=True)  # :103
    m = uq.shape[0]
    f_center = torch.zeros_like(xyz)
    f_center[:, 0] = xyz[:, 0] - (ij[:, 0].to(xyz.dtype) * vx + x_off)  # :109
    f_center[:, 1] = xyz[:, 1] - (ij[:, 1].to(xyz.dtype) * vy + y_off)  # :110
    f_center[:, 2] = xyz[:, 2] - z_off  # :111
    if simple2d:
        feats = [f_center, p[:, 1:] if use_absolute_xyz else p[:, 4:]]  # :209-213
    else:
        mean = torch.zeros((m, 3), dtype=xyz.dtype).index_add_(0, inv, xyz) / cnt.to(xyz.dtype).view(-1, 1)  # :105
        f_cluster = xyz - mean[inv]  # :106
        feats = [p[:, 1:] if use_absolute_xyz else p[:, 4:], f_cluster, f_center]  # :113-116
    if with_distance:
        feats.append(torch.linalg.vector_norm(p[:, 1:4], ord=2, dim=1, keepdim=True))
    x = torch.cat(feats, dim=-1)
    n_layers = len([k for k in state_dict if k.endswith("linear.weight")])
    for i in range(n_layers):
        x = _pfn_layer_v2(x, inv, m, state_dict, i, use_norm, last=(i == n_layers - 1))
    uq = uq.int()
    if simple2d:
        coords = torch.stack([uq // sxy, uq % sy, (uq % sxy) // sy], dim=1)  # :232-237 then [:, [0, 2, 1]]
    else:
        coords = torch.stack([uq // sxy, torch.zeros_like(uq), uq % sy, (uq % sxy) // sy], dim=1)  # :132-138
    return x, coords.numpy().astype(np.int32), cnt.numpy()
