"""GPU parity: batch_chamfer_dist (reference chamfer.py:62-94) and sample_mesh_points (sdf.py:617-670)."""
import numpy as np
import pytest
import torch

import workloads
from helpers import golden, pv_factory

pytestmark = pytest.mark.gpu


@pytest.mark.parametrize("name", ["probe", "wrench"])
def test_chamfer_vs_reference_golden(name):
    import pytorch_volumetric_b200 as pv
    z = golden(f"ref_chamfer_{name}")
    obj = pv_factory(name)
    pts = torch.from_numpy(z["pts_world"]).cuda()
    err0 = pv.batch_chamfer_dist(torch.from_numpy(z["w2o"]).cuda(), pts, obj)
    assert err0.shape == (len(z["w2o"]),)
    assert err0.max() < 1e-4                      # tests/test_chamfer.py:36-38 (mm^2 at the true pose)
    err1 = pv.batch_chamfer_dist(torch.from_numpy(z["w2o_p"]).cuda(), pts, obj, scale=1)
    np.testing.assert_allclose(err1.cpu().numpy(), z["err1"], rtol=2e-5)
    # CPU tensors in -> CPU tensor out
    e_cpu = pv.batch_chamfer_dist(torch.from_numpy(z["w2o_p"]), torch.from_numpy(z["pts_world"]), obj, scale=1)
    assert e_cpu.device.type == "cpu" and torch.allclose(e_cpu, err1.cpu())
    with pytest.raises(ValueError):
        pv.batch_chamfer_dist(torch.from_numpy(z["w2o"]).cuda(), pts)


def test_chamfer_reference_invariants(tmp_path):
    """tests/test_chamfer.py:40-66: mesh chamfer < point-cloud chamfer and within 5 % of it."""
    import pytorch_volumetric_b200 as pv
    torch.manual_seed(3)
    obj = pv_factory("probe")
    N, B = 1000, 64
    pts, normals, _ = pv.sample_mesh_points(obj, name="probe", num_points=N, device="cuda", cache={})
    R = pv.transforms.random_rotations(1, device="cuda")[0]
    gt = torch.eye(4, device="cuda"); gt[:3, :3] = R; gt[:3, 3] = torch.randn(3, device="cuda")
    gt_tf = pv.Transform3d(matrix=gt.unsqueeze(0))
    pts_world = gt_tf.transform_points(pts)
    pert = gt_tf.sample_perturbations(B, radian_sigma=0.1, translation_sigma=0.1)
    err = pv.batch_chamfer_dist(pert.inverse().get_matrix(), pts_world, obj, scale=1) * N
    perturbed_pts = pert.transform_points(pts)
    manual = torch.cdist(pts_world.unsqueeze(0), perturbed_pts).min(dim=2).values.square().sum(dim=1)
    assert torch.all(err < manual)
    assert torch.all(manual - err < 0.05 * manual)
    # obj_sdf route (chamfer.py:84-85) on a CachedSDF of the same object
    c = pv.CachedSDF("probe", 0.001, obj.bounding_box(padding=0.3), pv.MeshSDF(obj), device="cuda",
                     cache_path=str(tmp_path / "cache.pkl"), clean_cache=True)
    err_c = pv.batch_chamfer_dist(pert.inverse().get_matrix(), pts_world, obj_sdf=c, scale=1) * N
    assert torch.all((err_c - err).abs() < 0.1 * err + 1e-3)


def test_plausible_diversity_identities():
    """tests/test_chamfer.py:88-130."""
    import pytorch_volumetric_b200 as pv
    torch.manual_seed(3)
    obj = pv_factory("probe")
    B, tol = 10, 1e-4
    pts, _, _ = pv.sample_mesh_points(obj, name="probe", num_points=500, device="cuda", cache={})
    base = torch.eye(4, device="cuda"); base[:3, :3] = pv.transforms.random_rotations(1, device="cuda")[0]
    base[:3, 3] = torch.randn(3, device="cuda")
    gt_tf = pv.Transform3d(matrix=base.unsqueeze(0)).sample_perturbations(B, radian_sigma=0.05, translation_sigma=0.01)
    pd = pv.PlausibleDiversity(obj, model_points_eval=pts)
    r = pd(gt_tf.inverse().get_matrix(), gt_tf.get_matrix())
    assert r.plausibility < tol and r.coverage < tol
    part = pv.Transform3d(matrix=gt_tf.get_matrix()[:B // 2])
    r2 = pd(part.inverse().get_matrix(), gt_tf.get_matrix(), bidirectional=True)
    assert r2.plausibility < tol and r2.coverage > tol


@pytest.mark.parametrize("name", ["probe", "wrench", "drill"])
def test_sample_mesh_points(name, tmp_path):
    """tests/test_sdf.py:18-29 plus distributional checks of the area-uniform sampler."""
    import pytorch_volumetric_b200 as pv
    obj = pv_factory(name)
    db = str(tmp_path / "mp.pkl")
    pts, normals, cache = pv.sample_mesh_points(obj, name=name, num_points=1000, dbpath=db, device="cuda")
    assert pts.shape == (1000, 3) and normals.shape == (1000, 3) and pts.dtype == torch.float32
    v, g = pv.MeshSDF(obj)(pts)
    assert v.abs().max() < 1e-4
    assert (normals.norm(dim=-1) - 1).abs().max() < 1e-5
    # determinism + cache round trip (same layout as the reference: {name: {seed: {n: (pts, normals, None)}}})
    pts2, normals2, _ = pv.sample_mesh_points(None, name=name, num_points=1000, dbpath=db, device="cuda")
    assert torch.equal(pts, pts2) and torch.equal(normals, normals2)
    pts3, _, _ = pv.sample_mesh_points(obj, name=name, num_points=1000, device="cuda", cache={})
    assert torch.equal(pts, pts3)
    pts4, _, _ = pv.sample_mesh_points(obj, name=name, num_points=1000, seed=1, device="cuda", cache={})
    assert not torch.equal(pts, pts4)
    with pytest.raises(RuntimeError):
        pv.sample_mesh_points(None, name="nope", num_points=7, dbpath=str(tmp_path / "none.pkl"))
    # area uniformity: stratified allocation => every face holds round-to-nearest of (area share * n) samples
    from pytorch_volumetric_b200.sdf import _sample_surface
    n_big = 400_000
    big, face = _sample_surface(obj, n_big, 0, torch.device("cuda", 0), return_faces=True)
    vv, ff = workloads.fixture_mesh(name)
    tri = vv[ff]
    area = 0.5 * np.linalg.norm(np.cross(tri[:, 1] - tri[:, 0], tri[:, 2] - tri[:, 0]), axis=1)
    counts = np.bincount(face.cpu().numpy(), minlength=len(ff))
    assert counts.sum() == n_big and np.abs(counts - area / area.sum() * n_big).max() <= 1.0 + 1e-6
    # every sample lies on its face: barycentric reconstruction
    big = big.cpu().numpy()
    t = tri[face.cpu().numpy()]
    nrm = np.cross(t[:, 1] - t[:, 0], t[:, 2] - t[:, 0])
    nrm /= np.linalg.norm(nrm, axis=1, keepdims=True)
    assert np.abs(((big - t[:, 0]) * nrm).sum(-1)).max() < 1e-12
    # and the samples are spread inside the faces: mean barycentric weights ~ 1/3 each
    e0, e1, r = t[:, 1] - t[:, 0], t[:, 2] - t[:, 0], big - t[:, 0]
    d00, d01, d11 = (e0 * e0).sum(-1), (e0 * e1).sum(-1), (e1 * e1).sum(-1)
    d20, d21 = (r * e0).sum(-1), (r * e1).sum(-1)
    den = d00 * d11 - d01 * d01
    bv, bw = (d11 * d20 - d01 * d21) / den, (d00 * d21 - d01 * d20) / den
    assert bv.min() > -1e-9 and bw.min() > -1e-9 and (bv + bw).max() < 1 + 1e-9
    assert abs(bv.mean() - 1 / 3) < 5e-3 and abs(bw.mean() - 1 / 3) < 5e-3
