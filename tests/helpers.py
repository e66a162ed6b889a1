"""Shared helpers for the parity tests (test infrastructure; may use oracle/)."""
import glob
import os

import numpy as np
import torch

import workloads
from oracle import port

GOLDEN = workloads.GOLDEN


def golden(name):
    """Arrays of tests/golden/<name>.npz merged with those of its parts <name>.<part>.npz (a fixture is split into
    parts to keep every file small)."""
    out = {}
    for path in [os.path.join(GOLDEN, name + ".npz")] + sorted(glob.glob(os.path.join(GOLDEN, name + ".*.npz"))):
        with np.load(path) as z:
            assert not set(z.files) & set(out), path
            out.update({k: z[k] for k in z.files})
    return out


def port_mesh(name):
    v, f = workloads.fixture_mesh(name)
    return port.MeshPort(vertices=v, faces=f, name=name)


def pv_factory(name, **kw):
    import pytorch_volumetric_b200 as pv
    v, f = workloads.fixture_mesh(name)
    return pv.MeshObjectFactory(name, mesh=(v, f), **kw)


# ---- host mirror of the kernel's deterministic ray jitter (pvb_device.cuh: mix32 / hash_normal) ----
def _mix32(x):
    x = x.astype(np.uint32)
    x ^= x >> np.uint32(16)
    x = (x * np.uint32(0x7feb352d)).astype(np.uint32)
    x ^= x >> np.uint32(15)
    x = (x * np.uint32(0x846ca68b)).astype(np.uint32)
    x ^= x >> np.uint32(16)
    return x


def hash_normal(seed, idx, comp):
    idx = np.asarray(idx, dtype=np.uint64)
    lo = (idx & np.uint64(0xFFFFFFFF)).astype(np.uint32)
    hi = (idx >> np.uint64(32)).astype(np.uint32)
    with np.errstate(over="ignore"):
        a = _mix32(lo * np.uint32(3) + np.uint32(comp) + np.uint32(0x9e3779b9))
        b = _mix32(hi + np.uint32(0x85ebca6b))
        h0 = _mix32(np.uint32(seed) ^ a ^ b)
        h1 = _mix32(h0 + np.uint32(0x6a09e667))
    s = ((h0 & np.uint32(0xffff)).astype(np.float32) + (h0 >> np.uint32(16)).astype(np.float32)
         + (h1 & np.uint32(0xffff)).astype(np.float32) + (h1 >> np.uint32(16)).astype(np.float32))
    return (s - np.float32(131070.0)) * np.float32(2.6428816e-05)


def ray_noise(seed, n):
    idx = np.arange(n, dtype=np.uint64)
    return np.stack([hash_normal(seed, idx, c) for c in range(3)], axis=1).astype(np.float64)


def classify_mesh_mismatch(d_gpu, g_gpu, d_ref, g_ref, tol=1e-5, coord_scale=0.1):
    """Returns (n_bad_value, n_bad_grad_unexplained, report).

    Gradient tolerance: `tol` plus the fp32 conditioning of (closest - p) / |d| -- the closest point carries a
    few ulps of the coordinate magnitude, which the division by a small |d| amplifies.  A remaining exceedance
    is 'explained' when the point sits on the |d| = 1e-3 shell (sdf.py:162) or when the two sides agree on the
    distance but pick different closest features (ties on the medial axis)."""
    dv = np.abs(d_gpu - d_ref)
    bad_v = dv > tol
    dg = np.abs(g_gpu - g_ref).max(axis=-1)
    gtol = tol + 8 * np.finfo(np.float32).eps * coord_scale / np.maximum(np.abs(d_ref), 1e-12)
    bad_g = dg > gtol
    shell = np.abs(np.abs(d_ref) - 1e-3) < 2e-6
    explained = bad_g & (shell | (dv <= tol))     # same distance, different closest feature / shell flip
    unexplained = bad_g & ~explained
    rep = dict(n=len(d_ref), bad_val=int(bad_v.sum()), bad_grad=int(bad_g.sum()), explained=int(explained.sum()),
               max_dval=float(dv.max()), max_dgrad=float(dg.max()))
    return int(bad_v.sum()), int(unexplained.sum()), rep


# ---------------------------------------------------------------------------------------------------------------
# Per-exceedance classification for composed / robot queries (SURVEY 8c): every output that differs from the
# reference by more than the tolerance must be one of
#   (i)   a voxel-boundary flip: the fp32 rigid transform (an FMA chain here, a bmm in the reference) moved the
#         link-frame point across a cell boundary it sits on (|frac - 0.5| < FLIP_BAND cells) or across the edge of
#         the cached range, and the output equals the entry of that neighbouring cell / the other side's rule;
#   (ii)  the |d| = 1e-3 shell of sdf.py:162 or a closest-feature tie (same distance, another gradient) of a mesh;
#   (iii) an argmin tie between sub-SDFs (values within the tolerance, the other one's gradient reported).
# Anything else is unexplained and fails the test.
FLIP_BAND = 1.5e-4      # cells; rounding of the S*|A| rigid transforms: ~3 ulp of |q| over the cell size


def grid_spec(cached):
    """What the classifier needs from a pytorch_volumetric_b200.CachedSDF (tables are the ones the kernel reads)."""
    shape = tuple(cached.voxels.shape)
    return {"kind": "grid", "val": cached.voxels.raw_data.detach().cpu().numpy().reshape(shape).astype(np.float64),
            "grad": cached.voxels_grad.detach().cpu().numpy().reshape(*shape, 3).astype(np.float64),
            "lo": np.array([float(min(r)) for r in cached.ranges]), "hi": np.array([float(max(r)) for r in cached.ranges]),
            "bb": cached.bb.detach().cpu().numpy().astype(np.float64)}


def sphere_spec(radius):
    return {"kind": "sphere", "radius": float(radius)}


def _aabb_rule(bb, q):
    below = np.maximum(bb[:, 0] - q, 0.0)
    above = np.maximum(q - bb[:, 1], 0.0)
    delta = np.where(below > 0, -below, above)
    dist = np.linalg.norm(delta)
    return dist, (delta / dist if dist > 0 else delta)


def flip_candidates(specs, M, p):
    """All (value, object-frame gradient) pairs the reference's rules can produce for point p (3,) under the
    object->sub-frame matrices M (S,4,4, fp64) when every link-frame coordinate within FLIP_BAND of a cell boundary
    (or 1e-6 m of the range edge) is allowed to fall on either side."""
    out = []
    for s, spec in enumerate(specs):
        R, t = M[s, :3, :3], M[s, :3, 3]
        q = R @ p + t
        if spec["kind"] == "sphere":
            r = np.linalg.norm(q)
            out.append((r - spec["radius"], (q / (r + 1e-12)) @ R, s))
            continue
        lo, hi, val, grad = spec["lo"], spec["hi"], spec["val"], spec["grad"]
        n = np.array(val.shape)
        res = (hi - lo) / (n - 1)
        edge = 1e-6
        maybe_in = np.all((q >= lo - edge) & (q <= hi + edge))
        maybe_out = np.any((q < lo + edge) | (q > hi - edge))
        if maybe_in:
            u = (q - lo) / res
            opts = []
            for a in range(3):
                k = int(np.clip(np.rint(u[a]), 0, n[a] - 1))
                o = {k}
                f = u[a] - np.floor(u[a])
                if abs(f - 0.5) < FLIP_BAND:
                    o.update({int(np.clip(np.floor(u[a]), 0, n[a] - 1)), int(np.clip(np.floor(u[a]) + 1, 0, n[a] - 1))})
                opts.append(sorted(o))
            for kx in opts[0]:
                for ky in opts[1]:
                    for kz in opts[2]:
                        out.append((val[kx, ky, kz], grad[kx, ky, kz] @ R, s))
        if maybe_out:
            d, g = _aabb_rule(spec["bb"], q)
            out.append((d, g @ R, s))
    return out


def classify_composed(v_gpu, g_gpu, v_ref, g_ref, specs, mats, pts, tol=1e-5):
    """v_*: (A, P) values, g_*: (A, P, 3); mats: (S, A, 4, 4) object->sub-frame; pts (P, 3).
    Returns (n_exceed, n_unexplained, report).  An exceedance is explained when the GPU output equals, within `tol`,
    one of the legitimate alternatives of flip_candidates AND is a possible minimum over the sub-SDFs (between the
    min over sub-SDFs of their smallest and of their largest alternative)."""
    v_gpu = np.asarray(v_gpu, dtype=np.float64); g_gpu = np.asarray(g_gpu, dtype=np.float64)
    bad = (np.abs(v_gpu - v_ref) > tol) | (np.abs(g_gpu - g_ref).max(-1) > tol)
    idx = np.argwhere(bad)
    mats = np.asarray(mats, dtype=np.float64)
    pts = np.asarray(pts, dtype=np.float64)
    unexplained = []
    for a, i in idx:
        cands = flip_candidates(specs, mats[:, a], pts[i])
        # a valid output is min over sub-SDFs of ONE alternative each: it lies between the two extreme choices
        per_s = {}
        for cv, _cg, s_ in cands:
            lo_hi = per_s.setdefault(s_, [cv, cv])
            lo_hi[0], lo_hi[1] = min(lo_hi[0], cv), max(lo_hi[1], cv)
        lower = min(v[0] for v in per_s.values())
        upper = min(v[1] for v in per_s.values())
        ok = False
        if lower - tol <= v_gpu[a, i] <= upper + tol:
            for cv, cg, _s in cands:
                if abs(cv - v_gpu[a, i]) <= tol and np.abs(cg - g_gpu[a, i]).max() <= tol:
                    ok = True
                    break
        if not ok:
            unexplained.append((int(a), int(i), float(v_gpu[a, i]), float(v_ref[a, i])))
    rep = {"n": int(bad.size), "exceed": int(len(idx)), "unexplained": len(unexplained), "first": unexplained[:5]}
    return len(idx), len(unexplained), rep
