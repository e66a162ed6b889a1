"""Generate tests/golden/*.npz in the BUILD container (needs /root/reference).

TEST INFRASTRUCTURE.  Two kinds of fixtures:

1. meshes.npz -- the reference's own test meshes (tests/probe.obj,
   tests/offset_wrench_nogrip.obj, tests/YcbPowerDrill/textured_simple_reoriented.obj,
   tests/pv_sdf_debug/scene_mesh_{overlap,separated}.obj) parsed to (vertices fp64, faces int32) arrays,
   because /root/reference does not exist on the GPU box.

2. ref_*.npz -- input/output vectors produced by the UNMODIFIED reference source
   (/root/reference/src/pytorch_volumetric) imported over oracle/shims (the restated third-party
   dependencies).  They pin oracle/port.py (tests/test_oracle_pinning.py) and serve as golden vectors for
   the CUDA path (tests/test_gpu_mesh.py, test_gpu_cached.py, test_gpu_composed.py, test_gpu_chamfer_sample.py).

Run:  python -m oracle.make_golden
"""
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REF = "/root/reference"
GOLD = os.path.join(ROOT, "tests", "golden")

MESHES = {
    "probe": "tests/probe.obj",
    "wrench": "tests/offset_wrench_nogrip.obj",
    "drill": "tests/YcbPowerDrill/textured_simple_reoriented.obj",
    "scene_overlap": "tests/pv_sdf_debug/scene_mesh_overlap.obj",
    "scene_separated": "tests/pv_sdf_debug/scene_mesh_separated.obj",
}


def import_reference():
    """Import the real reference package with the third-party shims on the path."""
    sys.path.insert(0, ROOT)
    sys.path.insert(0, os.path.join(ROOT, "oracle", "shims"))
    sys.path.insert(0, os.path.join(REF, "src"))
    import pytorch_volumetric as pv
    assert pv.__file__.startswith(REF), pv.__file__
    return pv


def make_meshes():
    from oracle import tp_open3d as o3d
    out = {}
    for name, rel in MESHES.items():
        m = o3d.read_triangle_mesh(os.path.join(REF, rel))
        out[name + "_v"] = m.vertices
        out[name + "_f"] = m.triangles
    np.savez_compressed(os.path.join(GOLD, "meshes.npz"), **out)
    print("meshes.npz:", {k: v.shape for k, v in out.items()})


def save_split(name, arrays):
    """<name>.npz, with the voxel tables in <name>.tables.npz and the fp32-range variant in <name>.f32range.npz so that
    every fixture file stays below 1 MB (tests/helpers.py golden() merges the parts)."""
    parts = {"": {}, ".tables": {}, ".f32range": {}}
    for k, v in arrays.items():
        if k.startswith("table_") and k != "table_shape":
            parts[".tables"][k] = v
        elif k.endswith("_f32range"):
            parts[".f32range"][k] = v
        else:
            parts[""][k] = v
    for suffix, part in parts.items():
        if part:
            np.savez_compressed(os.path.join(GOLD, f"{name}{suffix}.npz"), **part)


def ray_noise_for(n, seed):
    """Seeds numpy's global generator so that the reference's np.random.randn(*shape) draw (sdf.py:149) is
    reproducible; returns nothing -- the port re-seeds identically."""
    np.random.seed(seed)


def make_reference_vectors():
    pv = import_reference()
    import pytorch_kinematics as pk
    tmp = "/tmp/pvb_golden_cache"
    os.makedirs(tmp, exist_ok=True)
    g = torch.Generator().manual_seed(1234)

    # ---- MeshSDF on probe / wrench / drill: random points around the mesh (sdf.py:122-172) ----
    for name in ("probe", "wrench", "drill"):
        obj = pv.MeshObjectFactory(os.path.join(REF, MESHES[name]))
        sdf = pv.MeshSDF(obj)
        bb = torch.tensor(obj.bounding_box(padding=0.02))
        n = 4000
        pts = (bb[:, 0] + (bb[:, 1] - bb[:, 0]) * torch.rand(n, 3, generator=g, dtype=torch.float64)).float()
        np.random.seed(7)
        res = obj.object_frame_closest_point(pts, compute_normal=True)
        # surface samples (tests/test_sdf.py:18-23)
        spts, snormals, _ = pv.sample_mesh_points(obj, name=name, num_points=500, seed=3,
                                                  dbpath=os.path.join(tmp, f"mp_{name}.pkl"), clean_cache=True)
        np.random.seed(8)
        sval, sgrad = sdf(spts)
        np.savez_compressed(os.path.join(GOLD, f"ref_meshsdf_{name}.npz"),
                            pts=pts.numpy(), closest=res.closest.numpy(), distance=res.distance.numpy(),
                            gradient=res.gradient.numpy(), normal=res.normal.numpy(),
                            bbox=obj.bounding_box(), bbox_pad=obj.bounding_box(padding=0.1, padding_ratio=0.05),
                            surf_pts=spts.numpy(), surf_normals=snormals.numpy(), surf_val=sval.numpy(),
                            surf_grad=sgrad.numpy())
        print(name, "meshsdf: inside fraction", float((res.distance < 0).float().mean()))

    # ---- CachedSDF on probe (both OOB strategies) and drill (sdf.py:444-602) ----
    for name, res_, pad in (("probe", 0.002, 0.01), ("drill", 0.01, 0.1)):
        obj = pv.MeshObjectFactory(os.path.join(REF, MESHES[name]))
        sdf = pv.MeshSDF(obj)
        rng = obj.bounding_box(padding=pad)
        np.random.seed(9)
        c = pv.CachedSDF(name, res_, rng, sdf, cache_path=os.path.join(tmp, f"sdf_{name}.pkl"), clean_cache=True)
        lo = torch.tensor([r[0] for r in c.ranges])
        hi = torch.tensor([r[1] for r in c.ranges])
        n = 20000
        q = (lo - 0.15 * (hi - lo) + 1.3 * (hi - lo) * torch.rand(n, 3, generator=g, dtype=torch.float64)).float()
        # add exact voxel centres and cell-boundary points (index rounding, half-to-even)
        coords, centres = pv.get_coordinates_and_points_in_grid(res_, c.ranges)
        pick = torch.randperm(len(centres), generator=g)[:2000]
        half = centres[pick] + 0.5 * torch.tensor(
            [float(c.voxels._resolution[k]) for k in range(3)], dtype=torch.float32)
        q = torch.cat([q, centres[pick], half])
        val, grad = c(q)
        keys = c.voxels.ravel_multi_index(c.voxels.ensure_index_key(q), c.voxels.shape)
        inb = c.voxels.get_valid_values(q)
        outside = c.outside_surface(q)
        out = dict(resolution=res_, range_in=rng, ranges=np.array(c.ranges), table_val=c.voxels.raw_data.numpy(),
                   table_shape=np.array(c.voxels.shape), table_grad=c.voxels_grad.numpy(), q=q.numpy(),
                   val=val.numpy(), grad=grad.numpy(), keys=keys.numpy(), inbound=inb.numpy(),
                   outside=outside.numpy(), bb=np.array(obj.bounding_box()))
        if name == "probe":
            cg = pv.CachedSDF(name, res_, rng, sdf, out_of_bounds_strategy=pv.OutOfBoundsStrategy.LOOKUP_GT_SDF,
                              cache_path=os.path.join(tmp, f"sdf_{name}.pkl"))
            np.random.seed(10)
            vg, gg = cg(q[:6000])
            out.update(val_gt=vg.numpy(), grad_gt=gg.numpy())
            # Python-float range -> fp32 index arithmetic in the third-party view
            rng32 = [(float(a), float(b)) for a, b in rng]
            c32 = pv.CachedSDF(name + "32", res_, rng32, sdf, cache_path=os.path.join(tmp, f"sdf32_{name}.pkl"),
                               clean_cache=True)
            v32, g32 = c32(q)
            k32 = c32.voxels.ravel_multi_index(c32.voxels.ensure_index_key(q), c32.voxels.shape)
            out.update(val_f32range=v32.numpy(), grad_f32range=g32.numpy(), keys_f32range=k32.numpy(),
                       inbound_f32range=c32.voxels.get_valid_values(q).numpy(),
                       table_val_f32range=c32.voxels.raw_data.numpy(), table_grad_f32range=c32.voxels_grad.numpy(),
                       ranges_f32range=np.array(c32.ranges))
        save_split(f"ref_cachedsdf_{name}", out)
        print(name, "cachedsdf: table", tuple(c.voxels.shape), "inbound fraction", float(inb.float().mean()))

    # ---- ComposedSDF: 3 cached probes + sphere, plain and config-batched (sdf.py:332-433) ----
    obj = pv.MeshObjectFactory(os.path.join(REF, MESHES["probe"]))
    msdf = pv.MeshSDF(obj)
    np.random.seed(11)
    cs = pv.CachedSDF("probe", 0.002, obj.bounding_box(padding=0.01), msdf,
                      cache_path=os.path.join(tmp, "sdf_probe.pkl"))
    S, A = 4, 3
    sdfs = [cs, cs, pv.SphereSDF(0.02), cs]
    R = pk.random_rotations(S * A, dtype=torch.float32)
    tmat = torch.eye(4).repeat(S * A, 1, 1)
    tmat[:, :3, :3] = R
    tmat[:, :3, 3] = (torch.rand(S * A, 3, generator=g) - 0.5) * 0.1
    n = 3000
    q = (torch.rand(n, 3, generator=g) - 0.5) * 0.25
    comp = pv.ComposedSDF(sdfs, pk.Transform3d(matrix=tmat[:S]))
    v1, g1 = comp(q)
    comp.set_transforms(pk.Transform3d(matrix=tmat), batch_dim=(A,))
    v2, g2 = comp(q.reshape(30, 100, 3))
    bbc = comp.surface_bounding_box(padding=0.01)
    np.savez_compressed(os.path.join(GOLD, "ref_composed.npz"), tmat=tmat.numpy(), q=q.numpy(), S=S, A=A,
                        val_plain=v1.numpy(), grad_plain=g1.numpy(), val_batched=v2.numpy(), grad_batched=g2.numpy(),
                        bbox_batched=bbc.numpy(), sphere_radius=0.02)
    print("composed:", v1.shape, v2.shape, bbc.shape)

    # ---- RobotSDF on the reference's single-link URDF (tests/test_model_to_sdf.py:263-326) ----
    urdf = open(os.path.join(REF, "tests", "offset_wrench.urdf")).read()
    chain = pk.build_serial_chain_from_urdf(urdf, "offset_wrench")
    np.random.seed(12)
    rs = pv.RobotSDF(chain, path_prefix=os.path.join(REF, "tests"),
                     link_sdf_cls=pv.cache_link_sdf_factory(resolution=0.004, padding=0.05,
                                                            cache_path=os.path.join(tmp, "sdf_wrench.pkl"),
                                                            clean_cache=True))
    B = 5
    th = torch.zeros(B, 6)
    th[1:, :3] = (torch.rand(B - 1, 3, generator=g) - 0.5) * 0.05
    th[1:, 3:] = (torch.rand(B - 1, 3, generator=g) - 0.5) * 1.0
    rs.set_joint_configuration(th)
    q = torch.cat([(torch.rand(2000, 3, generator=g) - 0.5) * torch.tensor([0.3, 0.2, 0.2]),
                   (torch.rand(1000, 3, generator=g) - 0.5) * 2.0])
    rv, rg = rs(q)
    rbb = rs.surface_bounding_box(padding=0.05)
    link0 = rs.sdf.sdfs[0]
    np.savez_compressed(os.path.join(GOLD, "ref_robot_wrench.npz"), th=th.numpy(), q=q.numpy(), val=rv.numpy(),
                        grad=rg.numpy(), bbox=rbb.numpy(), obj_to_link=rs.object_to_link_frames.get_matrix().numpy(),
                        table_val=link0.voxels.raw_data.numpy(), table_grad=link0.voxels_grad.numpy(),
                        table_shape=np.array(link0.voxels.shape), ranges=np.array(link0.ranges))
    print("robot:", rv.shape, rbb.shape)

    # ---- chamfer (tests/test_chamfer.py:16-66) ----
    for name in ("probe", "wrench"):
        obj = pv.MeshObjectFactory(os.path.join(REF, MESHES[name]))
        pts, _, _ = pv.sample_mesh_points(obj, name=name, num_points=1000, seed=0,
                                          dbpath=os.path.join(tmp, f"mpc_{name}.pkl"), clean_cache=True)
        torch.manual_seed(3)
        gt = pk.Transform3d(pos=torch.randn(3), rot=pk.random_rotation())
        pts_world = gt.transform_points(pts)
        Bc = 40
        w2o = gt.inverse().get_matrix().repeat(Bc, 1, 1)
        np.random.seed(13)
        err0 = pv.batch_chamfer_dist(w2o, pts_world, obj)
        pert = gt.sample_perturbations(Bc, radian_sigma=0.1, translation_sigma=0.1)
        w2o_p = pert.inverse().get_matrix()
        np.random.seed(14)
        err1 = pv.batch_chamfer_dist(w2o_p, pts_world, obj, scale=1)
        np.savez_compressed(os.path.join(GOLD, f"ref_chamfer_{name}.npz"), pts_world=pts_world.numpy(),
                            w2o=w2o.numpy(), err0=err0.numpy(), w2o_p=w2o_p.numpy(), err1=err1.numpy())
        print(name, "chamfer: err0 max", float(err0.max()), "err1 mean", float(err1.mean()))


def make_robot_build_vectors():
    """The single-link robot of tests/test_model_to_sdf.py:263-290 with the link table built by the reference itself
    (resolution 0.008): pins the port's table build + RobotSDF query (tests/test_oracle_pinning.py)."""
    pv = import_reference()
    import pytorch_kinematics as pk
    tmp = "/tmp/pvb_golden_cache"
    os.makedirs(tmp, exist_ok=True)
    urdf = open(os.path.join(REF, "tests", "offset_wrench.urdf")).read()
    chain = pk.build_serial_chain_from_urdf(urdf, "offset_wrench")
    np.random.seed(1)
    rs = pv.RobotSDF(chain, path_prefix=os.path.join(REF, "tests"),
                     link_sdf_cls=pv.cache_link_sdf_factory(resolution=0.008, padding=0.05,
                                                            cache_path=os.path.join(tmp, "sdf_wrench_008.pkl"),
                                                            clean_cache=True))
    th = torch.tensor([[0.01, -0.02, 0.0, 0.3, -0.2, 0.5], [0.0, 0.0, 0.0, 0.0, 0.0, 0.0]])
    rs.set_joint_configuration(th)
    q = (torch.rand(500, 3, generator=torch.Generator().manual_seed(5)) - 0.5) * 0.4
    v, g = rs(q)
    bb = rs.surface_bounding_box(padding=0.01)
    np.savez_compressed(os.path.join(GOLD, "ref_robot_wrench_built.npz"), th=th.numpy(), q=q.numpy(), val=v.numpy(),
                        grad=g.numpy(), bbox=bb.numpy())
    print("robot (reference-built table):", v.shape, bb.shape)


def make_voxel_vectors():
    """The reference's voxel containers (src/pytorch_volumetric/voxel.py:42-171) run unmodified over the shims:
    VoxelGrid set / get / list / resize, ExpandingVoxelGrid growth, voxel_down_sample on the reference's own test
    surface (tests/test_voxel_sdf.py:8-39) with numpy (fp32) and explicit ranges, 3-D and flat-z clouds, and
    ObjectFrameSDF.get_filtered_points (sdf.py:273-282) of the probe's CachedSDF voxel view."""
    pv = import_reference()
    g = torch.Generator().manual_seed(99)
    out = {}
    # ---- VoxelGrid: scatter-set, gather (incl. out-of-range -> invalid 0), list, resize_to_fit ----
    box = [(-1, 1), (-0.5, 0.5), (0, 0.6)]
    vg = pv.VoxelGrid(0.05, box)
    p = (torch.rand(3000, 3, generator=g) * torch.tensor([2.4, 1.3, 0.8]) + torch.tensor([-1.2, -0.65, -0.1])).float()
    val = torch.rand(3000, generator=g) + 0.5
    vg[p] = val
    out["vg_box"] = np.array(box, dtype=np.float64)
    out["vg_pts"], out["vg_val"] = p.numpy(), val.numpy()
    q = (torch.rand(2000, 3, generator=g) * torch.tensor([2.4, 1.3, 0.8]) + torch.tensor([-1.2, -0.65, -0.1])).float()
    out["vg_q"] = q.numpy()
    out["vg_q_out"] = vg[q].numpy()
    out["vg_data"] = vg.get_voxel_values().numpy()
    pos, kv = vg.get_known_pos_and_values()
    out["vg_known_pos"], out["vg_known_val"] = pos.numpy(), kv.numpy()
    vg.resize_to_fit()
    out["vg_fit_range"] = np.array(vg.range_per_dim, dtype=np.float64)
    out["vg_fit_shape"] = np.array(vg.get_voxel_values().shape)
    out["vg_fit_q_out"] = vg[q].numpy()
    # ---- ExpandingVoxelGrid ----
    ev = pv.ExpandingVoxelGrid(0.1, [(0, 1), (0, 1), (0, 1)])
    e1 = torch.tensor([[0.5, 0.5, 0.5], [0.93, 0.12, 0.31]])
    e2 = torch.tensor([[2.03, -0.47, 0.5], [-0.76, 1.88, 1.41]])
    ev[e1] = torch.tensor([4.0, 5.0])
    ev[e2] = torch.tensor([7.0, 8.0])
    out["ev_p1"], out["ev_p2"] = e1.numpy(), e2.numpy()
    out["ev_range"] = np.array(ev.range_per_dim, dtype=np.float64)
    out["ev_shape"] = np.array(ev.get_voxel_values().shape)
    out["ev_read"] = ev[torch.cat((e1, e2))].numpy()
    # ---- voxel_down_sample: the reference's own test surface (tests/test_voxel_sdf.py:8-29) ----
    N = 100
    x = torch.linspace(-2, 2, N)
    xx, yy = torch.meshgrid(x, x, indexing="ij")
    zz = torch.sin(xx) + 2 * torch.cos(yy)
    surf = torch.stack((xx.flatten(), yy.flatten(), zz.flatten()), dim=-1)
    out["ds_pts"] = surf.numpy()
    out["ds_02"] = pv.voxel_down_sample(surf, 0.2).numpy()
    out["ds_007"] = pv.voxel_down_sample(surf, 0.07).numpy()
    rng = np.array([[-1.0, 1.0], [-1.5, 0.5], [-3.0, 3.0]])           # does not enclose the data: honoured (voxel.py:153)
    out["ds_range"] = rng
    out["ds_ranged"] = pv.voxel_down_sample(surf, 0.1, range_per_dim=rng).numpy()
    flat = torch.cat((surf[:, :2], torch.zeros(len(surf), 1)), dim=1)
    frng = np.array([[-1.7, 1.9], [-2.5, 1.5], [0.0, 0.0]])
    out["ds_flat_range"] = frng
    out["ds_flat"] = pv.voxel_down_sample(flat, 0.15, range_per_dim=frng, ignore_flat_dim=True).numpy()
    # ---- get_filtered_points of a CachedSDF voxel view (sdf.py:273-282): the interior of the probe ----
    obj = pv.MeshObjectFactory(os.path.join(REF, MESHES["probe"]))
    sdf = pv.MeshSDF(obj)
    np.random.seed(5)
    cached = pv.CachedSDF("probe", 0.002, obj.bounding_box(padding=0.01), sdf, cache_path="/tmp/pvb_golden_voxel.pkl",
                          clean_cache=True)
    inner = cached.get_filtered_points(lambda v: v < -0.001)
    out["fp_interior"] = inner.numpy()
    out["fp_table"] = cached.voxels.raw_data.numpy()
    out["fp_shape"] = np.array(cached.voxels.shape)
    out["fp_ranges"] = np.array(cached.ranges, dtype=np.float64)
    np.savez_compressed(os.path.join(GOLD, "ref_voxel.npz"), **out)
    print("ref_voxel.npz:", {k: getattr(v, "shape", v) for k, v in out.items()})


if __name__ == "__main__":
    os.makedirs(GOLD, exist_ok=True)
    if len(sys.argv) > 1 and sys.argv[1] == "voxel":
        make_voxel_vectors()
    elif len(sys.argv) > 1 and sys.argv[1] == "robot_build":
        make_robot_build_vectors()
    else:
        make_meshes()
        make_reference_vectors()
        make_robot_build_vectors()
        make_voxel_vectors()
