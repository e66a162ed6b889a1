"""CPU: pins oracle/port.py (the restatement of the reference's own code) against the golden vectors written by the
UNMODIFIED reference source over oracle/shims (oracle/make_golden.py).  The third-party layer under both is the same
restatement, so agreement here is bit-exact."""
import numpy as np
import pytest
import torch

from helpers import golden, port_mesh
from oracle import port, tp_pytorch_kinematics as opk


@pytest.mark.parametrize("name", ["probe", "wrench", "drill"])
def test_port_mesh_query_equals_reference_golden(name, oracle_lib):
    z = golden(f"ref_meshsdf_{name}")
    mesh = port_mesh(name)
    n = 4000 if name != "drill" else 1500          # brute force on the drill: keep the CPU suite short
    np.random.seed(7)
    noise = np.random.randn(4000, 3)[:n]
    c, d, g, nrm = mesh.closest_point(torch.from_numpy(z["pts"][:n]), compute_normal=True, ray_noise=noise)
    assert np.array_equal(c.numpy(), z["closest"][:n])
    assert np.array_equal(d.numpy(), z["distance"][:n])
    assert np.array_equal(g.numpy(), z["gradient"][:n])
    assert np.array_equal(nrm.numpy(), z["normal"][:n])
    np.testing.assert_array_equal(mesh.bounding_box(), z["bbox"])
    np.testing.assert_array_equal(mesh.bounding_box(padding=0.1, padding_ratio=0.05), z["bbox_pad"])


@pytest.mark.parametrize("name", ["probe", "wrench"])
def test_port_sample_mesh_points_equals_reference_golden(name, oracle_lib):
    z = golden(f"ref_meshsdf_{name}")
    mesh = port_mesh(name)
    pts, normals = port.sample_mesh_points_port(mesh, num_points=500, seed=3)
    assert np.array_equal(pts.numpy(), z["surf_pts"])
    assert np.array_equal(normals.numpy(), z["surf_normals"])
    # the reference's invariant (tests/test_sdf.py:23)
    assert np.abs(z["surf_val"]).max() < 1e-4


@pytest.mark.parametrize("name", ["probe", "drill"])
def test_port_cached_lookup_equals_reference_golden(name, oracle_lib):
    z = golden(f"ref_cachedsdf_{name}")
    mesh = port_mesh(name)
    shape = tuple(int(s) for s in z["table_shape"])
    c = port.CachedSDFPort(name, float(z["resolution"]), z["range_in"], port.MeshSDFPort(mesh),
                           tables=(torch.from_numpy(z["table_val"]).reshape(shape), torch.from_numpy(z["table_grad"])))
    np.testing.assert_array_equal(np.array(c.ranges), z["ranges"])
    q = torch.from_numpy(z["q"])
    keys, flat, inb = c.index_and_mask(q)
    assert np.array_equal(inb.numpy(), z["inbound"])
    assert np.array_equal(flat.numpy()[z["inbound"]], z["keys"][z["inbound"]])
    v, g = c(q)
    assert np.array_equal(v.numpy(), z["val"]) and np.array_equal(g.numpy(), z["grad"], equal_nan=True)
    assert np.array_equal(c.outside_surface(q).numpy(), z["outside"])
    # fp64 index arithmetic: numpy ranges make the third-party view hold float64 min/max/resolution
    assert c.voxels._min.dtype == torch.float64


def test_port_cached_table_build_equals_reference_golden(oracle_lib):
    z = golden("ref_cachedsdf_probe")
    mesh = port_mesh("probe")
    np.random.seed(9)
    c = port.CachedSDFPort("probe", float(z["resolution"]), z["range_in"], port.MeshSDFPort(mesh))
    assert np.array_equal(c.voxels.raw_data.numpy(), z["table_val"])
    assert np.array_equal(c.voxels_grad.numpy(), z["table_grad"])
    # fp32-range variant (Python floats)
    rng32 = [(float(a), float(b)) for a, b in z["range_in"]]
    shape = tuple(int(s) for s in z["table_shape"])
    c32 = port.CachedSDFPort("probe32", float(z["resolution"]), rng32, port.MeshSDFPort(mesh),
                             tables=(torch.from_numpy(z["table_val_f32range"]).reshape(shape),
                                     torch.from_numpy(z["table_grad_f32range"])))
    assert c32.voxels._min.dtype == torch.float32
    q = torch.from_numpy(z["q"])
    _, flat, inb = c32.index_and_mask(q)
    assert np.array_equal(inb.numpy(), z["inbound_f32range"])
    assert np.array_equal(flat.numpy()[z["inbound_f32range"]], z["keys_f32range"][z["inbound_f32range"]])
    v, g = c32(q)
    assert np.array_equal(v.numpy(), z["val_f32range"])


def test_port_composed_equals_reference_golden(oracle_lib):
    zc = golden("ref_cachedsdf_probe")
    z = golden("ref_composed")
    mesh = port_mesh("probe")
    shape = tuple(int(s) for s in zc["table_shape"])
    cs = port.CachedSDFPort("probe", float(zc["resolution"]), zc["range_in"], port.MeshSDFPort(mesh),
                            tables=(torch.from_numpy(zc["table_val"]).reshape(shape),
                                    torch.from_numpy(zc["table_grad"])))
    S, A = int(z["S"]), int(z["A"])
    sdfs = [cs, cs, port.SphereSDFPort(float(z["sphere_radius"])), cs]
    tmat = torch.from_numpy(z["tmat"])
    q = torch.from_numpy(z["q"])
    comp = port.ComposedSDFPort(sdfs, opk.Transform3d(matrix=tmat[:S]))
    v, g = comp(q)
    assert np.array_equal(v.numpy(), z["val_plain"]) and np.array_equal(g.numpy(), z["grad_plain"])
    comp.set_transforms(opk.Transform3d(matrix=tmat), batch_dim=(A,))
    vb, gb = comp(q.reshape(30, 100, 3))
    assert np.array_equal(vb.numpy(), z["val_batched"]) and np.array_equal(gb.numpy(), z["grad_batched"])
    assert np.array_equal(comp.surface_bounding_box(padding=0.01).numpy(), z["bbox_batched"])


def test_port_chamfer_equals_reference_golden(oracle_lib):
    z = golden("ref_chamfer_probe")
    mesh = port_mesh("probe")
    np.random.seed(14)
    err1 = port.batch_chamfer_dist_port(torch.from_numpy(z["w2o_p"]), torch.from_numpy(z["pts_world"]), mesh, scale=1)
    assert np.array_equal(err1.numpy(), z["err1"])
    with pytest.raises(ValueError):
        port.batch_chamfer_dist_port(torch.from_numpy(z["w2o_p"]), torch.from_numpy(z["pts_world"]))


def test_port_equals_live_reference_source(tmp_path, oracle_lib):
    """The single link robot of tests/test_model_to_sdf.py:263-290 with the link table built by the port itself:
    values, gradients and bounding box equal what the unmodified reference source computed for the same inputs
    with its own table build (oracle/make_golden.py: ref_robot_wrench_built)."""
    from test_gpu_composed import write_wrench_urdf
    z = golden("ref_robot_wrench_built")
    urdf = write_wrench_urdf(str(tmp_path))
    chain = opk.build_serial_chain_from_urdf(open(urdf).read(), "offset_wrench")
    np.random.seed(1)
    rp = port.RobotSDFPort(chain, path_prefix=str(tmp_path),
                           link_sdf_factory=port.cache_link_sdf_factory_port(resolution=0.008, padding=0.05))
    rp.set_joint_configuration(torch.from_numpy(z["th"]))
    v, g = rp(torch.from_numpy(z["q"]))
    assert np.array_equal(v.numpy(), z["val"]) and np.array_equal(g.numpy(), z["grad"])
    assert np.array_equal(rp.surface_bounding_box(padding=0.01).numpy(), z["bbox"])


def test_port_robot_equals_reference_golden(tmp_path, oracle_lib):
    """RobotSDFPort on the procedural twin of the reference's tests/offset_wrench.urdf reproduces the vectors the
    unmodified reference produced (oracle/make_golden.py: ref_robot_wrench) -- FK + offset composition bit-exact,
    values / gradients bit-exact on the reference-built link table."""
    from oracle import tp_pytorch_kinematics as opk
    from test_gpu_composed import write_wrench_urdf
    z = golden("ref_robot_wrench")
    urdf = write_wrench_urdf(str(tmp_path))
    chain = opk.build_serial_chain_from_urdf(open(urdf).read(), "offset_wrench")
    shape = tuple(int(s) for s in z["table_shape"])
    tables = (torch.from_numpy(z["table_val"]).reshape(shape), torch.from_numpy(z["table_grad"]))
    rp = port.RobotSDFPort(chain, path_prefix=str(tmp_path),
                           link_sdf_factory=port.cache_link_sdf_factory_port(resolution=0.004, padding=0.05,
                                                                             tables=tables))
    np.testing.assert_allclose(np.array(rp.sdf.sdfs[0].ranges), z["ranges"], atol=1e-12)
    rp.set_joint_configuration(torch.from_numpy(z["th"]))
    assert np.array_equal(rp.object_to_link.get_matrix().numpy(), z["obj_to_link"])
    v, g = rp(torch.from_numpy(z["q"]))
    assert np.array_equal(v.numpy(), z["val"]) and np.array_equal(g.numpy(), z["grad"], equal_nan=True)
    np.testing.assert_array_equal(rp.surface_bounding_box(padding=0.05).numpy(), z["bbox"])
