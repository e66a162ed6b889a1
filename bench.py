#!/usr/bin/env python
"""bench.py -- SDF+grad queries/s of the batched signed-distance query path on B200.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--workload default|c4|c2|mesh10k|mesh50k|c3|c3cached|c5|c4readme]
                    [--impl reference] [--dump-outputs DIR]

One "step" = one pass of the hot path over one batch of synthetic input.  Every timed loop of a run times exactly K
steps.

`--dump-outputs DIR` writes what the last timed step of the headline (or of the one --workload) returned, as
DIR/value.npy and DIR/gradient.npy (rank 0).  Inputs are seeded, so two builds run with the same arguments can be
compared output for output; see dump_outputs for the sampling of large results.

DEFAULT (no --workload): the headline line.
  * headline = BASELINE.json configs[3] (C4), the workload north_star's multi-GPU target names: RobotSDF of a
    7-DOF arm (8 link SDFs), 200 joint configurations x 100 000 query points, value + gradient.  With N > 1
    (torchrun, one rank per GPU) the CONFIGURATION batch is split over the ranks (strong scaling: total work fixed)
    and the timed step ends with the FULL (200, 100 000) result on EVERY rank -- re-assembly inside the timed
    region.  `value` = 2*10^7 (configuration, point) pairs / max-over-ranks device time.  The `reassembly` object
    carries the sub-values next to it: no_reassembly (every rank keeps its slab), nccl_all_gather, peer_stores
    (kernel epilogue stores into all ranks' buffers over NVLink), multicast_stores (one multimem.st per chunk through
    an NVLS multicast mapping), each timed the same way.
  * `workloads`: every other BASELINE config on the same GPUs in the same run -- mesh10k (the north-star
    single-GPU target: MeshSDF on a 10 000-triangle mesh, 10^7 queries), c2, c3, c3cached, c5 -- each with value,
    ms_per_step, roofline{achieved, frac, traffic, kernel_ms}, e2e and (N=1) cpu_baseline.

`roofline.kernel_ms` is an independent measurement: the library brackets the dominant kernel launch of one call with
its own pair of CUDA events on the launch stream (pvb_timing_enable / pvb_timing_last_ms); median of 7 launches.
`roofline.traffic` is the ncu dram__bytes_read+write of that kernel from the committed capture (profiles/ncu_traffic.json).

`--impl reference` times the CPU restatement of the reference (oracle/port.py, torch-cpu + OpenMP BVH, all host
threads that help) on a bounded sample of the same workloads; the reference itself is pure Python over third-party
wheels that are not installable in this image (SURVEY.md section 0), so the oracle port is the reference arm.

Prints ONE JSON line (rank 0).
"""
import argparse
import atexit
import json
import os
import shutil
import statistics
import sys
import tempfile
import threading
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
import workloads  # noqa: E402

METRIC = "sdf_grad_queries_per_s"
UNIT = "queries/s"
HEADLINE = "c4"
OTHER_WORKLOADS = ("mesh10k", "c2", "c3", "c3cached", "c5")


# ------------------------------------------------------------------------------------------------ helpers
_scratch = None


def scratch_dir():
    """Directory for the files a run writes (link meshes, URDFs, SDF table caches): created fresh for this process,
    so that no table cached by an earlier run or another build is read back, and removed when the process exits."""
    global _scratch
    if _scratch is None:
        _scratch = tempfile.mkdtemp(prefix="pvb_bench_")
        atexit.register(shutil.rmtree, _scratch, ignore_errors=True)
    return _scratch


DUMP_MAX_BYTES = 48 << 20


def dump_outputs(out, dirname):
    """Writes the tensors one step returned as <dirname>/value.npy [and gradient.npy], float32 (float64 kept).
    Value is [..., P] and gradient [..., P, 3] over P query points; when they hold more than DUMP_MAX_BYTES, the
    same seeded, sorted sample of the P points is kept in every run."""
    tensors = [t for t in (out if isinstance(out, (tuple, list)) else (out,)) if torch.is_tensor(t)]
    n = tensors[0].shape[-1]
    per_point = sum(t.numel() // n * 4 * (2 if t.dtype == torch.float64 else 1) for t in tensors)
    k = min(n, DUMP_MAX_BYTES // per_point)
    idx = None if k == n else torch.randperm(n, generator=torch.Generator().manual_seed(0))[:k].sort().values
    os.makedirs(dirname, exist_ok=True)
    for name, t, axis in zip(("value", "gradient"), tensors, (-1, -2)):
        if idx is not None:
            t = t.index_select(t.dim() + axis, idx.to(t.device))
        if t.dtype != torch.float64:
            t = t.float()
        np.save(os.path.join(dirname, name + ".npy"), t.cpu().numpy())


def measured_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as fh:
            return float(json.load(fh)["hbm_gbs"]), "measured"
    return 6650.0, "fallback"


def ncu_traffic(workload):
    """DRAM bytes per launch of the dominant kernel from the committed ncu --set full capture (profiles/)."""
    path = os.path.join(ROOT, "profiles", "ncu_traffic.json")
    if os.path.exists(path):
        with open(path) as fh:
            return json.load(fh).get(workload)
    return None


def ncu_limits(workload):
    """Issue-slot / L1 data pipe / DRAM utilisation of the dominant kernel from the same committed capture: says what
    bounds a kernel whose HBM fraction is small by nature (tree walks, the RobotSDF kernel)."""
    path = os.path.join(ROOT, "profiles", "ncu_limits.json")
    if os.path.exists(path):
        with open(path) as fh:
            return json.load(fh).get(workload)
    return None


class ClockSampler:
    """SM clock + throttle reasons sampled DURING the timed region through NVML (nvidia_ml_py).

    Measured on this pool (gpurun_out/bisect.log, round 1): NVML queries and `nvidia-smi -lms` contend with kernel
    launches for a driver lock -- a 2 ms sampling period doubled the host issue time per step (25 -> 55 us) and
    made a 58 us/step kernel loop host-bound.  So: NVML is initialised before the warm-up, a background thread
    samples every 100 ms (long runs), and one sample is always taken right after the last timed launch has been
    ENQUEUED, i.e. while the timed kernels are still executing on the GPU, where it cannot delay any launch."""
    REASONS = (("hw_slowdown", 0x8), ("hw_thermal_slowdown", 0x40), ("sw_thermal_slowdown", 0x20),
               ("sw_power_cap", 0x4), ("hw_power_brake", 0x80))

    def __init__(self, index, period_s=0.1):
        self.period = period_s
        self.sm, self.reasons_seen, self.max = [], set(), None
        self._run = False
        self.h = None
        try:
            import pynvml
            self.nv = pynvml
            pynvml.nvmlInit()
            vis = os.environ.get("CUDA_VISIBLE_DEVICES")
            phys = int(vis.split(",")[index]) if vis and vis.split(",")[index].isdigit() else index
            self.h = pynvml.nvmlDeviceGetHandleByIndex(phys)
            self.max = float(pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM))
            self._sample()          # touch every entry point once, outside the timed region
            self.sm.clear(); self.reasons_seen.clear()
        except Exception as e:      # no NVML: report it, never fail the benchmark
            self.err = repr(e)
            self.h = None

    def _sample(self):
        nv = self.nv
        self.sm.append(float(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM)))
        mask = int(nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)) if hasattr(
            nv, "nvmlDeviceGetCurrentClocksEventReasons") else int(nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h))
        for name, bit in self.REASONS:
            if mask & bit:
                self.reasons_seen.add(name)

    def sample_now(self):
        if self.h is not None:
            try:
                self._sample()
            except Exception:
                pass

    def _loop(self):
        while self._run:
            time.sleep(self.period)
            if not self._run:
                break
            try:
                self._sample()
            except Exception:
                break

    def start(self):
        if self.h is None or os.environ.get("PVB_BENCH_NO_SAMPLER"):
            return
        self._run = True
        self.t = threading.Thread(target=self._loop, daemon=True)
        self.t.start()

    def stop(self):
        if self.h is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [f"nvml unavailable: {getattr(self, 'err', '')}"]}
        self._run = False
        if hasattr(self, "t"):
            self.t.join(timeout=1)
        if not self.sm:
            try:
                self._sample()
            except Exception:
                pass
        return {"sm_mhz": statistics.median(self.sm) if self.sm else None, "sm_max_mhz": self.max,
                "reasons": sorted(self.reasons_seen), "samples": len(self.sm)}


def dist_setup(n_gpus):
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world > 1:
        import torch.distributed as dist
        torch.cuda.set_device(local)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    else:
        torch.cuda.set_device(0)
    return rank, world, local


def barrier(world):
    if world > 1:
        import torch.distributed as dist
        dist.barrier()
    torch.cuda.synchronize()


def max_over_ranks(x, world):
    if world > 1:
        import torch.distributed as dist
        t = torch.tensor([x], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())
    return x


# ---------------------------------------------------------------------------------------------- workloads
class Workload:
    """name, units per step (per GPU), algorithmic bytes per step, step(i) on resident inputs,
    step_host(i) through the public API with host buffers."""
    kernel = ""


class C2(Workload):
    """BASELINE C2: CachedSDF(res=0.005) on the drill, 10^7 uniform points over the cache range inflated 10 % per
    side (~42 % out of range -> AABB rule), 3 rotating input buffers (120 MB each, > L2)."""
    name = "c2"
    kernel = "grid_lookup_tma_kernel"
    n_points = 10_000_000

    def __init__(self, rank, n_buffers=3, cache_dir=None):
        import pytorch_volumetric_b200 as pv
        v, f = workloads.fixture_mesh("drill")
        self.obj = pv.MeshObjectFactory("drill", mesh=(v, f))
        gt = pv.MeshSDF(self.obj)
        cache = os.path.join(cache_dir or scratch_dir(), f"pvb_bench_c2_{rank}.pkl")
        self.sdf = pv.CachedSDF("drill", 0.005, self.obj.bounding_box(padding=0.1), gt, device="cuda",
                                cache_path=cache, clean_cache=True)
        # same object for host callers: results come back as host tensors (tables still live on the GPU)
        self.sdf_host = pv.CachedSDF("drill", 0.005, self.obj.bounding_box(padding=0.1), gt, device="cpu",
                                     cache_path=cache)
        lo = np.array([r[0] for r in self.sdf.ranges]); hi = np.array([r[1] for r in self.sdf.ranges])
        self.lo, self.hi = lo - 0.1 * (hi - lo), hi + 0.1 * (hi - lo)
        self.host = [workloads.uniform_points(self.n_points, self.lo, self.hi, seed=1000 * rank + b).pin_memory()
                     for b in range(n_buffers)]
        self.dev = [h.cuda() for h in self.host]
        self.units = self.n_points
        n_vox = int(np.prod(self.sdf.voxels.shape))
        # 12 B point in + 4 B value + 12 B gradient out per query, + the 16 B/voxel table once per launch
        self.alg_bytes = 28 * self.n_points + 16 * n_vox
        self.h2d_bytes = 12 * self.n_points
        self.d2h_bytes = 16 * self.n_points
        self.launches_per_step = 1
        self.desc = {"workload": "C2 CachedSDF(drill, res=0.005, 74x66x78 voxels) x 1e7 uniform points "
                                 "(range +10%/side, ~42% out-of-range -> AABB rule), value+gradient",
                     "points_per_step_per_gpu": self.n_points, "l2_policy": "inputs > L2 (120 MB in + 160 MB out "
                     "per step), 3 rotating input buffers", "oob_strategy": "BOUNDING_BOX"}

    def step(self, i):
        return self.sdf(self.dev[i % len(self.dev)])

    def step_host(self, i):
        # public API, host tensor in -> host tensors out (the reference's own default is device="cpu")
        return self.sdf_host(self.host[i % len(self.host)])

    # CPU arm: the oracle port on the same tables
    def cpu_setup(self):
        from oracle import port
        v, f = workloads.fixture_mesh("drill")
        mesh = port.MeshPort(vertices=v, faces=f, name="drill")
        shape = tuple(self.sdf.voxels.shape)
        self.cpu_sdf = port.CachedSDFPort("drill", 0.005, mesh.bounding_box(padding=0.1), port.MeshSDFPort(mesh),
                                          tables=(self.sdf.voxels.raw_data.cpu().reshape(shape),
                                                  self.sdf.voxels_grad.cpu()))
        self.cpu_sample = 2_000_000
        self.cpu_pts = self.host[0][:self.cpu_sample].clone()
        return f"{self.cpu_sample} of the {self.n_points} points of one step (oracle/port.py CachedSDFPort, torch-cpu)"

    def cpu_step(self):
        self.cpu_sdf(self.cpu_pts)
        return self.cpu_sample


class Mesh10k(Workload):
    """North-star target: MeshSDF (BVH closest point + ray parity) on the 10 000-triangle bumpy sphere, 10^7
    uniform points in AABB + 0.05."""
    name = "mesh10k"
    kernel = "mesh_query_kernel"
    n_points = 10_000_000

    def __init__(self, rank, n_buffers=3, cache_dir=None, n_lon=100, n_lat=51):
        import pytorch_volumetric_b200 as pv
        v, f = workloads.bumpy_sphere(n_lon, n_lat)
        self.v, self.f = v, f
        self.obj = pv.MeshObjectFactory(f"bumpy{len(f)}", mesh=(v, f))
        self.sdf = pv.MeshSDF(self.obj)
        self.host = [workloads.uniform_points(self.n_points, v.min(0) - 0.05, v.max(0) + 0.05,
                                              seed=2 + 1000 * rank + b).pin_memory() for b in range(n_buffers)]
        self.dev = [h.cuda() for h in self.host]
        self.units = self.n_points
        self.alg_bytes = 28 * self.n_points + 48 * len(f) + 128 * self.obj._bvh_host[0].shape[0]
        self.h2d_bytes = 12 * self.n_points
        self.d2h_bytes = 16 * self.n_points
        self.launches_per_step = 1
        self.desc = {"workload": f"MeshSDF on a closed {len(f)}-triangle bumpy sphere x 1e7 uniform points in "
                                 f"AABB+0.05 (BVH4 closest point + ray-parity sign + gradient)",
                     "points_per_step_per_gpu": self.n_points, "l2_policy": "inputs > L2, 3 rotating input buffers",
                     "note": "tree walk: latency/L1-bound, not HBM-bound; roofline.frac on compulsory bytes"}

    def step(self, i):
        return self.sdf(self.dev[i % len(self.dev)])

    def step_host(self, i):
        return self.sdf(self.host[i % len(self.host)])

    def cpu_setup(self):
        from oracle import port, tp_open3d
        tp_open3d.QUERY_METHOD = "bvh"        # OpenMP BVH evaluator of the oracle (not the brute-force checker)
        self.cpu_mesh = port.MeshPort(vertices=self.v, faces=self.f)
        self.cpu_sample = 400_000
        self.cpu_pts = self.host[0][:self.cpu_sample].clone()
        return f"{self.cpu_sample} of the {self.n_points} points of one step (oracle MeshPort over the OpenMP BVH)"

    def cpu_step(self):
        self.cpu_mesh.closest_point(self.cpu_pts)
        return self.cpu_sample


def c4_config(n_cfg=200, n_pts=100_000):
    """The `config` object of the headline, IDENTICAL in the GPU arm and the reference arm."""
    return {"workload": f"C4 RobotSDF synthetic 7-DOF arm (8 links, per-link CachedSDF res=0.02 pad=1.0) x {n_cfg} joint "
                        f"configurations x {n_pts} uniform points, value+gradient; configurations sharded over the "
                        f"ranks, full ({n_cfg}, {n_pts}) result on every rank inside the timed region",
            "n_cfg": n_cfg, "n_pts": n_pts, "units_per_step": n_cfg * n_pts,
            "l2_policy": "output 320 MB/step > L2 (126 MB); 3 rotating point buffers",
            "result_reassembly": "full result on every rank; method = the fastest of NCCL all-gather / peer stores / "
                                 "multicast stores measured in this run (reassembly.chosen); no collective at N=1"}


class C4(Workload):
    """BASELINE C4: RobotSDF, synthetic iiwa-like 7-DOF arm (8 link meshes), per-link CachedSDF(res 0.02, padding
    1.0), 200 joint configurations x 100 000 points.  With N GPUs the configuration batch is split into contiguous
    slabs (strong scaling); `mode` selects what a step leaves behind: "none" (every rank keeps its slab), "nccl"
    (all-gather of the slabs), "peer" (the kernel epilogue stores each slab into all ranks' buffers)."""
    name = "c4"
    kernel = "robot_query_kernel<8,unrolled> | composed_query_kernel<false,2,16> (by configuration-tile fill)"

    def __init__(self, rank, world=1, n_cfg=200, n_pts=100_000, cache_dir=None, mode="none"):
        import pytorch_volumetric_b200 as pv
        from pytorch_volumetric_b200 import distributed as pd
        self.pv, self.pd = pv, pd
        self.rank, self.world = rank, world
        self.mode = mode if world > 1 else "none"
        self.peer = None
        self.peer_error = None
        d = os.path.join(cache_dir or scratch_dir(), f"pvb_bench_arm_{rank}")
        urdf, end = workloads.write_arm(d)
        chain = pv.build_serial_chain_from_urdf(open(urdf).read(), end).to(device="cuda")
        self.robot = pv.RobotSDF(chain, path_prefix=d,
                                 link_sdf_cls=pv.cache_link_sdf_factory(resolution=0.02, padding=1.0, device="cuda",
                                                                        cache_path=os.path.join(d, "cache.pkl")))
        self.th_host = workloads.arm_configurations(n_cfg).pin_memory()
        self.th = self.th_host.cuda()
        self.robot.set_joint_configuration(self.th)
        lo = [r[0] for r in workloads.ARM_QUERY_RANGE]; hi = [r[1] for r in workloads.ARM_QUERY_RANGE]
        self.host = [workloads.uniform_points(n_pts, lo, hi, seed=4 + b).pin_memory() for b in range(3)]
        self.dev = [h.cuda() for h in self.host]
        self.begin, self.end = pd.shard_range(n_cfg, rank, world)
        self.n_pts, self.n_cfg = n_pts, n_cfg
        self.units = (self.end - self.begin) * n_pts           # pairs this rank evaluates per step
        n_vox = sum(int(np.prod(s.voxels.shape)) for s in self.robot.sdf.sdfs)
        self.n_vox = n_vox
        # SURVEY 8(d): 16 B per (configuration, point) pair out + points + transforms + tables once per launch
        self.alg_bytes = 16 * self.units + 12 * n_pts + 48 * 8 * (self.end - self.begin) + 16 * n_vox
        self.h2d_bytes = 12 * n_pts + 4 * 7 * (self.end - self.begin)
        self.d2h_bytes = 16 * self.units
        self.launches_per_step = 1
        self.desc = c4_config(n_cfg, n_pts) if (n_cfg, n_pts) == (200, 100_000) else \
            {"workload": f"RobotSDF synthetic 7-DOF arm x {n_cfg} configurations x {n_pts} points"}

    def enable_peer(self):
        """Allocate + map the peer result buffers (collective).  Returns None or the reason it is unavailable."""
        if self.world == 1 or self.peer is not None:
            return None
        try:
            self.peer = self.pd.PeerResult(self.n_cfg, self.n_pts)
        except Exception as e:        # no peer access between these GPUs, IPC refused, ...
            self.peer_error = repr(e)[:300]
        # all ranks must agree
        ok = torch.tensor([0.0 if self.peer is None else 1.0], device="cuda")
        torch.distributed.all_reduce(ok, op=torch.distributed.ReduceOp.MIN)
        if ok.item() == 0.0 and self.peer is not None:
            self.peer.close()
            self.peer = None
            self.peer_error = self.peer_error or "another rank could not map the peer buffers"
        elif ok.item() == 0.0:
            torch.distributed.barrier()
        return self.peer_error

    def set_mode(self, mode):
        self.mode = mode if self.world > 1 else "none"

    def step(self, i):
        pts = self.dev[i % 3]
        if self.world == 1:
            return self.robot(pts)                                 # the public RobotSDF.__call__
        if self.mode == "peer":   # full result on every rank, written by the kernels themselves
            return self.pd.sharded_robot_query(self.robot, pts, gather="peer", result=self.peer)
        if self.mode == "dma":    # slab evaluated locally, pushed to the peers by the copy engines (chunks overlap)
            return self.pd.sharded_robot_query(self.robot, pts, gather="dma", result=self.peer)
        if self.mode == "mc":     # ... through the NVLS multicast mapping: one multimem.st reaches every rank
            return self.pd.sharded_robot_query(self.robot, pts, gather="multicast", result=self.peer)
        if self.mode == "nccl":   # full result on every rank: one NCCL all-gather per tensor
            return self.pd.sharded_robot_query(self.robot, pts, gather=True)
        return self.pd.sharded_robot_query(self.robot, pts, gather=False)

    def step_reconfigure(self, i):
        """set_joint_configuration (FK + link-frame composition) + the query, through the public RobotSDF API."""
        self.robot.set_joint_configuration(self.th)
        return self.step(i)

    def step_host(self, i):
        """Public API end to end: host joint values + host points in, this rank's slab of the result in pinned host
        memory out (the union over ranks is the full result)."""
        self.robot.set_joint_configuration(self.th_host[self.begin:self.end].to("cuda", non_blocking=True))
        out = self.robot(self.host[i % 3])
        return out

    def restore(self):
        self.robot.set_joint_configuration(self.th)

    def close(self):
        if self.peer is not None:
            self.peer.close()
            self.peer = None


class C5(Workload):
    """BASELINE C5: chamfer of a 5*10^6-point cloud against a 50 000-triangle mesh, B=1 transform; the cloud is
    sharded over ranks."""
    name = "c5"
    kernel = "chamfer_partial_kernel"

    def __init__(self, rank, world=1, n_pts=5_000_000, n_tf=1, cache_dir=None):
        import pytorch_volumetric_b200 as pv
        from pytorch_volumetric_b200 import distributed as pd
        from pytorch_volumetric_b200.sdf import _sample_surface
        v, f = workloads.bumpy_sphere(250, 101)
        self.obj = pv.MeshObjectFactory("bumpy50k", mesh=(v, f))
        surf = _sample_surface(self.obj, n_pts, 5, torch.device("cuda", torch.cuda.current_device())).float()
        g = torch.Generator(device="cuda").manual_seed(5)
        tf = workloads.random_rigid(1, seed=5, t_range=0.1).cuda()[0]
        world_pts = surf @ tf[:3, :3].T + tf[:3, 3] + 0.002 * torch.randn(n_pts, 3, device="cuda", generator=g)
        begin, end = pd.shard_range(n_pts, rank, world)
        self.pts = world_pts[begin:end].contiguous()
        self.host_pts = self.pts.cpu().pin_memory()
        # 60 MB cloud < L2: rotate 3 device copies (180 MB) so that no step finds its input in L2, instead of a flush
        # memset inside the timed step
        self.copies = [self.pts] + [self.pts.clone() for _ in range(2 if (end - begin) * 36 < 400e6 else 0)]
        pert = workloads.random_rigid(n_tf, seed=6, t_range=0.01).cuda()
        self.w2o = torch.linalg.inv(tf.unsqueeze(0)) @ pert
        self.units = (end - begin) * n_tf
        self.alg_bytes = 12 * (end - begin) + 48 * len(f) + 128 * self.obj._bvh_host[0].shape[0] + 4 * n_tf
        self.h2d_bytes = 12 * (end - begin) + 64 * n_tf
        self.d2h_bytes = 4 * n_tf
        self.launches_per_step = 2
        self.pv = pv
        self.desc = {"workload": f"C5 chamfer: {n_pts}-point cloud -> 50 000-triangle bumpy sphere, B={n_tf} "
                                 f"transform(s), cloud sharded over ranks", "points_this_rank": end - begin,
                     "l2_policy": "60 MB cloud fits L2: 3 rotating device copies of the cloud (180 MB > L2)"}

    def step(self, i):
        return self.pv.batch_chamfer_dist(self.w2o, self.copies[i % len(self.copies)], self.obj)

    def step_host(self, i):
        return self.pv.batch_chamfer_dist(self.w2o.cpu(), self.host_pts, self.obj)


class C3(Workload):
    """BASELINE C3: ComposedSDF of 16 drills (MeshSDF sharing one BVH) under random SE(3), 126^3 grid points."""
    name = "c3"
    kernel = "composed_query_kernel<true>"

    def __init__(self, rank, world=1, cache_dir=None, cached=False):
        import pytorch_volumetric_b200 as pv
        v, f = workloads.fixture_mesh("drill")
        obj = pv.MeshObjectFactory("drill", mesh=(v, f))
        gt = pv.MeshSDF(obj)
        if cached:
            sub = pv.CachedSDF("drill", 0.005, obj.bounding_box(padding=0.1), gt, device="cuda",
                               cache_path=os.path.join(cache_dir or scratch_dir(), f"pvb_c3_{rank}.pkl"))
        else:
            sub = gt
        tm = workloads.random_rigid(16, seed=1, t_range=0.5).cuda()
        self.comp = pv.ComposedSDF([sub] * 16, pv.Transform3d(matrix=tm))
        axis = torch.arange(126, dtype=torch.float32) * (1.4 / 125) - 0.7
        pts = torch.cartesian_prod(axis, axis, axis)
        from pytorch_volumetric_b200 import distributed as pd
        b, e = pd.shard_range(len(pts), rank, world)
        self.host_pts = pts[b:e].contiguous().pin_memory()
        self.pts = self.host_pts.cuda()
        # 24 MB of points + 32 MB of results per step fit L2: rotate 6 device copies of the point set (144 MB > L2)
        # instead of a flush memset inside the timed step
        self.copies = [self.pts] + [self.pts.clone() for _ in range(5)]
        self.units = e - b
        self.alg_bytes = 28 * self.units
        self.h2d_bytes = 12 * self.units
        self.d2h_bytes = 16 * self.units
        self.launches_per_step = 1
        self.desc = {"workload": f"C3 ComposedSDF of 16 drills ({'CachedSDF res=0.005' if cached else 'MeshSDF, one shared BVH'}) "
                                 f"random SE(3), 126^3 grid points + gradient", "points_this_rank": self.units,
                     "l2_policy": "6 rotating device copies of the point set (144 MB > L2); results are fresh buffers"}
        if cached:
            self.kernel = "composed_query_kernel<false>"
            self.name = "c3cached"          # its own entry in profiles/ncu_traffic.json

    def step(self, i):
        return self.comp(self.copies[i % len(self.copies)])

    def step_host(self, i):
        return self.comp(self.host_pts)


def make_workload(name, rank, world):
    if name == "c2":
        return C2(rank)
    if name == "mesh10k":
        return Mesh10k(rank)
    if name == "mesh50k":
        return Mesh10k(rank, n_lon=250, n_lat=101)
    if name == "c4":
        return C4(rank, world)
    if name == "c4readme":
        return C4(rank, world, n_cfg=200, n_pts=15251)
    if name == "c5":
        return C5(rank, world)
    if name == "c3":
        return C3(rank, world)
    if name == "c3cached":
        return C3(rank, world, cached=True)
    raise SystemExit(f"unknown workload {name}")


WEAK_SCALED = ("c2", "mesh10k", "mesh50k")       # every rank runs the full batch on its own points


# ------------------------------------------------------------------------------------------- reference arm
class CpuArm:
    """One workload on the host through the oracle port.  `run(n)` evaluates the first n sample points (n <= max_n);
    one point is `units_per_point` units of the metric (the number of configurations for RobotSDF)."""

    def __init__(self, run, max_n, what, label, units_per_point=1):
        self.run, self.max_n, self.what, self.label, self.units_per_point = run, max_n, what, label, units_per_point


def cpu_arm(name):
    """CPU implementation of one workload from the oracle port (never touches the GPU).  Tables the GPU arm builds
    on the device are rebuilt on the host with the oracle's OpenMP BVH evaluator, untimed."""
    from oracle import port, tp_open3d
    from oracle import tp_pytorch_kinematics as opk
    tp_open3d.QUERY_METHOD = "bvh"
    np.random.seed(0)
    if name == "c2":
        v, f = workloads.fixture_mesh("drill")
        mesh = port.MeshPort(vertices=v, faces=f, name="drill")
        sdf = port.CachedSDFPort("drill", 0.005, mesh.bounding_box(padding=0.1), port.MeshSDFPort(mesh))
        lo = np.array([r[0] for r in sdf.ranges]); hi = np.array([r[1] for r in sdf.ranges])
        max_n = 2_000_000
        pts = workloads.uniform_points(max_n, lo - 0.1 * (hi - lo), hi + 0.1 * (hi - lo), seed=0)
        return CpuArm(lambda n: sdf(pts[:n]), max_n,
                      "oracle/port.py CachedSDFPort (op-for-op torch-cpu restatement of sdf.py:535-571)",
                      "C2 CachedSDF(drill, res=0.005) value+gradient")
    if name in ("mesh10k", "mesh50k"):
        v, f = workloads.bumpy_sphere(*((100, 51) if name == "mesh10k" else (250, 101)))
        mesh = port.MeshPort(vertices=v, faces=f)
        max_n = 400_000
        pts = workloads.uniform_points(max_n, v.min(0) - 0.05, v.max(0) + 0.05, seed=2)
        return CpuArm(lambda n: mesh.closest_point(pts[:n]), max_n,
                      "oracle MeshPort.closest_point over the OpenMP BVH evaluator (sdf.py:122-172 restated)",
                      f"MeshSDF on {len(f)}-triangle bumpy sphere")
    if name in ("c3", "c3cached"):
        v, f = workloads.fixture_mesh("drill")
        mesh = port.MeshPort(vertices=v, faces=f, name="drill")
        sub = port.MeshSDFPort(mesh)
        if name == "c3cached":
            sub = port.CachedSDFPort("drill", 0.005, mesh.bounding_box(padding=0.1), sub)
        comp = port.ComposedSDFPort([sub] * 16, opk.Transform3d(matrix=workloads.random_rigid(16, seed=1, t_range=0.5)))
        max_n = 200_000 if name == "c3cached" else 50_000
        pts = workloads.uniform_points(max_n, [-0.7] * 3, [0.7] * 3, seed=3)
        return CpuArm(lambda n: comp(pts[:n]), max_n,
                      "uniform points of the [-0.7, 0.7]^3 query box x 16 sub-SDFs; oracle/port.py ComposedSDFPort "
                      "(sdf.py:392-433 restated: per-SDF loop + argmin)",
                      f"C3 ComposedSDF of 16 drills ({'CachedSDF res=0.005' if name == 'c3cached' else 'MeshSDF'})")
    if name in ("c4", "c4readme"):
        d = os.path.join(scratch_dir(), "pvb_bench_arm_cpu")
        urdf, end = workloads.write_arm(d)
        chain = opk.build_serial_chain_from_urdf(open(urdf).read(), end)
        robot = port.RobotSDFPort(chain, path_prefix=d, link_sdf_factory=port.cache_link_sdf_factory_port(0.02, 1.0))
        n_cfg, max_n = 20, 50_000
        robot.set_joint_configuration(workloads.arm_configurations(n_cfg))
        lo = [r[0] for r in workloads.ARM_QUERY_RANGE]; hi = [r[1] for r in workloads.ARM_QUERY_RANGE]
        pts = workloads.uniform_points(max_n, lo, hi, seed=4)
        return CpuArm(lambda n: robot(pts[:n]), max_n,
                      f"{n_cfg} of the 200 configurations per point (8 links each); oracle/port.py RobotSDFPort "
                      f"(model_to_sdf.py:82-125 + sdf.py:392-433 restated)",
                      "C4 RobotSDF synthetic 7-DOF arm (8 links, CachedSDF res=0.02 pad=1.0)", units_per_point=n_cfg)
    if name == "c5":
        v, f = workloads.bumpy_sphere(250, 101)
        mesh = port.MeshPort(vertices=v, faces=f)
        max_n = 1_000_000
        g = torch.Generator().manual_seed(5)
        idx = torch.randint(0, len(v), (max_n,), generator=g)
        tf = workloads.random_rigid(1, seed=5, t_range=0.1)[0]
        surf = torch.from_numpy(np.asarray(v, dtype=np.float32))[idx]
        cloud = surf @ tf[:3, :3].T + tf[:3, 3] + 0.002 * torch.randn(max_n, 3, generator=g)
        w2o = torch.linalg.inv(tf.unsqueeze(0))
        return CpuArm(lambda n: port.batch_chamfer_dist_port(w2o, cloud[:n], mesh=mesh), max_n,
                      "cloud points, B=1; oracle/port.py batch_chamfer_dist_port (chamfer.py:79-94 restated, OpenMP "
                      "BVH closest point)", "C5 chamfer: point cloud -> 50 000-triangle bumpy sphere")
    raise SystemExit(f"unknown workload {name}")


def usable_cpus():
    """CPUs this process may actually run on: affinity mask, capped by the cgroup CPU quota when there is one."""
    n = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    try:                                            # cgroup v2
        quota, period = open("/sys/fs/cgroup/cpu.max").read().split()[:2]
        if quota != "max":
            n = min(n, max(1, int(quota) // int(period)))
    except (OSError, ValueError):
        pass
    try:                                            # cgroup v1
        quota = int(open("/sys/fs/cgroup/cpu/cpu.cfs_quota_us").read())
        period = int(open("/sys/fs/cgroup/cpu/cpu.cfs_period_us").read())
        if quota > 0:
            n = min(n, max(1, quota // period))
    except (OSError, ValueError):
        pass
    return n


def pick_cpu_threads(probe):
    """Run the CPU arm with the thread count that is FASTEST on this host.  `probe()` is a small slice of the
    workload.  Asking torch-cpu / OpenMP for every core the OS reports is not always that: the masked-index ops of
    the reference path are memory bound and a 128-thread launch of each of them read 35x slower than 8 threads on a
    2 M-point sample (first bench lines of this round), which would flatter the GPU arm.  Returns (threads, tried)."""
    from oracle import _geom
    top = usable_cpus()
    tried = {}
    probe()                                         # first-touch / lazy-initialisation cost stays out of the comparison
    for c in sorted({top, max(1, top // 2), 32, 16, 8, 4}, reverse=True):
        if c > top:
            continue
        torch.set_num_threads(c)
        _geom.set_num_threads(c)
        t0 = time.perf_counter()
        probe()
        tried[c] = time.perf_counter() - t0
    best = min(tried, key=tried.get)
    torch.set_num_threads(best)
    _geom.set_num_threads(best)
    return best, tried


# headline of the --impl reference run (warm-up + timed steps) is sized to about this many seconds, each entry of its
# `workloads` object to about the second figure (PVB_BENCH_REF_BUDGET_S: the CPU test tier shortens both)
REFERENCE_ARM_BUDGET_S = float(os.environ.get("PVB_BENCH_REF_BUDGET_S", 120.0))
REFERENCE_OTHER_BUDGET_S = min(6.0, REFERENCE_ARM_BUDGET_S)


def _time_cpu_arm(arm, steps, warmup, budget_s):
    """Bounded sample of one CPU arm: thread count = the fastest on this host, step size from a throughput probe so
    that warm-up + `steps` steps take about `budget_s`.  Returns the cpu_baseline-style dict + ms per step."""
    probe = max(1000, arm.max_n // 20)
    cores, tried = pick_cpu_threads(lambda: arm.run(probe))
    t0 = time.perf_counter()
    arm.run(probe)
    per_point = (time.perf_counter() - t0) / probe
    n = int(budget_s / (steps + max(warmup, 1)) / per_point)
    n = max(1000, min(arm.max_n, n))
    sample = n * arm.units_per_point
    for _ in range(max(warmup, 1)):
        arm.run(n)
    t0 = time.perf_counter()
    for _ in range(steps):
        arm.run(n)
    dt = time.perf_counter() - t0
    what = (f"{n} points per step ({sample} units); {arm.what}; {cores} host threads = the fastest of "
            f"{sorted(tried)} tried on {usable_cpus()} usable CPUs")
    return {"value": sample * steps / dt, "unit": UNIT, "cores": cores, "kind": "port", "sample": what}, 1e3 * dt / steps


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    name = HEADLINE if args.workload == "default" else args.workload
    arm = cpu_arm(name)
    cpu, ms = _time_cpu_arm(arm, args.steps, args.warmup, REFERENCE_ARM_BUDGET_S)
    config = c4_config() if name == "c4" else {"workload": arm.label}
    line = {"impl": "reference", "metric": METRIC, "value": cpu["value"], "unit": UNIT, "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms,
            "higher_is_better": True, "scaling": "strong" if name not in WEAK_SCALED else "weak",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": config,
            "cpu_baseline": cpu,
            "e2e": {"value": cpu["value"], "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    if args.workload == "default":
        others = {}
        for w in OTHER_WORKLOADS:
            try:
                c, ms_w = _time_cpu_arm(cpu_arm(w), args.steps, args.warmup, REFERENCE_OTHER_BUDGET_S)
                others[w] = {"value": c["value"], "unit": UNIT, "ms_per_step": ms_w, "cpu_baseline": c}
            except Exception as e:      # never lose the headline to a secondary arm
                others[w] = {"error": repr(e)[:200]}
        line["workloads"] = others
    print(json.dumps(line))
    return 0


# ------------------------------------------------------------------------------------------------ GPU arms
def sum_over_ranks(x, world):
    if world > 1:
        import torch.distributed as dist
        t = torch.tensor([x], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.SUM)
        return float(t.item())
    return x


def timed_steps(step, steps, warmup, world, sampler=None, last=None):
    """`warmup` untimed steps, then exactly `steps` steps bracketed by barrier + synchronize on both sides, timed with
    CUDA events on the launch stream; returns (max-over-ranks ms for all steps, this rank's ms, host issue us/step).
    `last`, if given, receives the result of the last timed step once the timing has ended."""
    out = None
    for i in range(warmup):             # same ownership pattern as the timed loop (the previous result stays alive
        out = step(i)                   # while the next one is allocated), so the allocator is in steady state
    stream = torch.cuda.current_stream()
    t_begin, t_end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier(world)
    if sampler is not None:
        sampler.start()
    t_cpu0 = time.perf_counter()
    t_begin.record(stream)
    for i in range(steps):              # nothing but the public API call in the timed loop
        out = step(i)
    t_end.record(stream)
    issue_us = (time.perf_counter() - t_cpu0) / steps * 1e6
    if sampler is not None:
        sampler.sample_now()            # the GPU is still executing the queued timed steps here
    barrier(world)
    mine = t_begin.elapsed_time(t_end)
    if last is not None:
        last(out)
    del out
    return max_over_ranks(mine, world), mine, issue_us


def kernel_time_ms(step, n=7):
    """Device time of ONE launch of the workload's dominant kernel, measured by the library's own event pair around
    that launch (median of n calls, each followed by a synchronize): independent of ms_per_step."""
    from pytorch_volumetric_b200 import _native
    _native.timing_enable(True)
    ts = []
    try:
        for i in range(n):
            out = step(i)
            ts.append(_native.timing_last_ms())
            torch.cuda.synchronize()
            del out
    finally:
        _native.timing_enable(False)
    return statistics.median(ts)


def e2e_arm(wl, units_all, world, steps):
    """Host buffers through the public API, H2D + D2H inside the timed region (wall clock around a synchronize,
    max over ranks)."""
    r = None
    for i in range(3):                  # steady state of the pinned host allocator
        r = wl.step_host(i)
    torch.cuda.synchronize()
    barrier(world)
    t0 = time.perf_counter()
    for i in range(steps):
        r = wl.step_host(i)
    torch.cuda.synchronize()
    dt_mine = time.perf_counter() - t0
    barrier(world)
    dt = max_over_ranks(dt_mine, world)
    del r
    return {"value": units_all * steps / dt, "unit": UNIT, "h2d_bytes_per_step": wl.h2d_bytes,
            "d2h_bytes_per_step": wl.d2h_bytes, "ms_per_step": 1e3 * dt / steps, "steps": steps}


def roofline_of(wl, kernel_ms):
    peak, peak_kind = measured_peaks()
    achieved = wl.alg_bytes / (kernel_ms * 1e-3) / 1e9
    return {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
            "traffic": ncu_traffic(wl.name), "ncu": ncu_limits(wl.name), "kernel": wl.kernel, "kernel_ms": kernel_ms,
            "algorithmic_bytes_per_launch": wl.alg_bytes, "peak_source": f"of {peak_kind}"}


class all_host_cpus:
    """The CPU arm may use every core the process was started with, not only the GPU's NUMA node; the NUMA binding
    is put back afterwards so that later pinned buffers stay local."""

    def __init__(self, full_affinity):
        self.full = full_affinity

    def __enter__(self):
        self.bound = os.sched_getaffinity(0) if self.full is not None else None
        if self.full is not None:
            os.sched_setaffinity(0, self.full)

    def __exit__(self, *exc):
        if self.bound is not None:
            os.sched_setaffinity(0, self.bound)
        return False


def cpu_baseline_of(name, wl=None, seconds=6.0):
    """Oracle port of one workload on the host cores, bounded sample (rank 0, N=1 only)."""
    if wl is not None and hasattr(wl, "cpu_setup"):          # same tables / points as the GPU arm
        sample = wl.cpu_setup()
        cpu_step = wl.cpu_step
    else:
        arm = cpu_arm(name)
        n = max(1000, arm.max_n // 4)
        sample = f"{n} points per step; {arm.what}"
        cpu_step = lambda: (arm.run(n), n * arm.units_per_point)[1]      # noqa: E731
    cpu_threads, tried = pick_cpu_threads(cpu_step)
    sample += f"; {cpu_threads} host threads = the fastest of {sorted(tried)} tried"
    t0 = time.perf_counter()
    done = 0
    while time.perf_counter() - t0 < seconds:
        done += cpu_step()
    dt = time.perf_counter() - t0
    return {"value": done / dt, "unit": UNIT, "cores": cpu_threads, "kind": "port", "sample": sample}


def run_workload(name, rank, world, steps, warmup, with_e2e, with_cpu, sampler=None, full_affinity=None, last=None):
    """One non-headline workload: device-resident value, independent kernel time + roofline, e2e, CPU baseline."""
    wl = make_workload(name, rank, world)
    torch.cuda.synchronize()
    total_ms, _, issue_us = timed_steps(wl.step, steps, warmup, world, sampler, last)
    units_all = max_over_ranks(float(wl.units), world) * world if name in WEAK_SCALED \
        else sum_over_ranks(float(wl.units), world)
    res = {"value": units_all * steps / (total_ms * 1e-3), "unit": UNIT, "ms_per_step": total_ms / steps,
           "steps": steps, "scaling": "weak" if name in WEAK_SCALED else "strong", "config": wl.desc,
           "gpu_launches": wl.launches_per_step * steps, "host_issue_us_per_step": issue_us}
    res["roofline"] = roofline_of(wl, kernel_time_ms(wl.step))
    if with_e2e:
        res["e2e"] = e2e_arm(wl, units_all, world, steps)
    if with_cpu:
        with all_host_cpus(full_affinity):
            res["cpu_baseline"] = cpu_baseline_of(name, wl)
    return wl, res


# -------------------------------------------------------------------------------------------------- main
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--workload", default="default")
    ap.add_argument("--impl", default="native", choices=["native", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-workloads", action="store_true", help="default run: headline only")
    ap.add_argument("--mode", default=None, choices=[None, "none", "nccl", "peer", "mc", "dma"],
                    help="C4 at N>1: force the re-assembly method of the headline instead of picking the faster one")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the result of the last timed step as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "native":
        ap.error("--dump-outputs writes the results of the native path")
    args.warmup = max(args.warmup, 3) if args.impl == "native" else args.warmup
    if args.impl == "reference":
        return run_reference(args)

    rank, world, local = dist_setup(args.gpus)
    from pytorch_volumetric_b200 import _native
    from pytorch_volumetric_b200 import distributed as pd
    if _native.lib_missing() and rank == 0:      # normally prebuilt by __graft_entry__.build(); the product never builds itself
        _native.build()
    # pin the rank next to its GPU before any pinned host buffer exists (e2e across the box, VERDICT r01 item 6)
    bound = pd.bind_to_gpu_numa_node(local)
    full_affinity = bound[2] if bound else None
    barrier(world)
    sampler = ClockSampler(local)
    with_cpu = rank == 0 and world == 1 and not args.no_cpu_baseline
    dump = (lambda out: dump_outputs(out, args.dump_outputs)) if args.dump_outputs and rank == 0 else None

    if args.workload != "default" and args.workload not in ("c4", "c4readme"):
        # ---- single-workload mode (tuning / profiling scripts) ----
        wl, res = run_workload(args.workload, rank, world, args.steps, args.warmup, not args.no_e2e, with_cpu,
                               sampler, full_affinity, dump)
        clocks = sampler.stop()
        if rank == 0:
            line = {"metric": METRIC, "value": res["value"], "unit": UNIT, "n_gpus": world, "steps": args.steps,
                    "warmup": args.warmup, "ms_per_step": res["ms_per_step"], "higher_is_better": True,
                    "scaling": res["scaling"], "vs_baseline": None, "dtype": "f32", "data": "synthetic",
                    "config": wl.desc, "clocks": clocks, "e2e": res.get("e2e"), "gpu_launches": res["gpu_launches"],
                    "roofline": res["roofline"], "host_issue_us_per_step": res["host_issue_us_per_step"],
                    "cpu_baseline": res.get("cpu_baseline")}
            print(json.dumps(line))
        return finish(world)

    # ---- headline: C4 RobotSDF, configurations split over the ranks, full result on every rank ----
    wl = make_workload("c4" if args.workload == "default" else args.workload, rank, world)
    torch.cuda.synchronize()
    units_all = sum_over_ranks(float(wl.units), world)
    reassembly = None
    if world > 1:
        reassembly = {}
        wl.set_mode("none")
        ms, _, _ = timed_steps(wl.step, args.steps, args.warmup, world)
        reassembly["no_reassembly"] = {"ms_per_step": ms / args.steps, "value": units_all * args.steps / (ms * 1e-3)}
        wl.set_mode("nccl")
        ms, _, _ = timed_steps(wl.step, args.steps, args.warmup, world)
        reassembly["nccl_all_gather"] = {"ms_per_step": ms / args.steps, "value": units_all * args.steps / (ms * 1e-3)}
        err = wl.enable_peer()
        if err is None:
            wl.set_mode("peer")
            ms, _, _ = timed_steps(wl.step, args.steps, args.warmup, world)
            remote = 16.0 * wl.units * (world - 1)          # bytes this rank pushes to its peers per step
            reassembly["peer_stores"] = {"ms_per_step": ms / args.steps, "value": units_all * args.steps / (ms * 1e-3),
                                         "nvlink_out_GBps_per_rank": remote / (ms / args.steps * 1e-3) / 1e9,
                                         "nvlink_in_bytes_per_rank": remote, "buffers": wl.peer.backend}
            slab = wl.end - wl.begin
            for pieces in (1, 2, 4):         # copy-engine pushes: the slab at once, or in pieces that overlap the kernel
                wl.peer.dma_chunk_cfgs = 0 if pieces == 1 else max(1, -(-slab // pieces))
                wl.set_mode("dma")
                ms, _, _ = timed_steps(wl.step, args.steps, args.warmup, world)
                reassembly[f"dma_push_{pieces}"] = {
                    "ms_per_step": ms / args.steps, "value": units_all * args.steps / (ms * 1e-3),
                    "chunk_cfgs": wl.peer.dma_chunk_cfgs or slab,
                    "nvlink_ingest_GBps_per_rank": 16.0 * (units_all - wl.units) / (ms / args.steps * 1e-3) / 1e9}
            if wl.peer.multicast:
                wl.set_mode("mc")
                ms, _, _ = timed_steps(wl.step, args.steps, args.warmup, world)
                reassembly["multicast_stores"] = {"ms_per_step": ms / args.steps,
                                                  "value": units_all * args.steps / (ms * 1e-3),
                                                  "nvlink_out_GBps_per_rank": 16.0 * wl.units / (ms / args.steps * 1e-3) / 1e9}
            else:
                reassembly["multicast_stores"] = {"unavailable": wl.peer.backend_note or
                                                  f"no multicast mapping (buffers: {wl.peer.backend})"}
        else:
            reassembly["peer_stores"] = {"unavailable": err}
            reassembly["multicast_stores"] = {"unavailable": err}
        for k in ("nccl_all_gather", "peer_stores", "multicast_stores"):
            if "ms_per_step" in reassembly.get(k, {}):
                reassembly[k]["nvlink_ingest_GBps_per_rank"] = \
                    16.0 * (units_all - wl.units) / (reassembly[k]["ms_per_step"] * 1e-3) / 1e9
        reassembly["nvlink_peak_GBps_per_direction"] = 770.0      # B200_PROFILING.md
        if args.mode:
            chosen = args.mode
        else:
            cands = {"nccl": reassembly["nccl_all_gather"]["ms_per_step"]}
            if "ms_per_step" in reassembly["peer_stores"]:
                cands["peer"] = reassembly["peer_stores"]["ms_per_step"]
            if "ms_per_step" in reassembly["multicast_stores"]:
                cands["mc"] = reassembly["multicast_stores"]["ms_per_step"]
            dma = {k: v for k, v in reassembly.items() if k.startswith("dma_push") and "ms_per_step" in v}
            if dma:
                best_dma = min(dma, key=lambda k: dma[k]["ms_per_step"])
                cands["dma"] = dma[best_dma]["ms_per_step"]
            chosen = min(cands, key=cands.get)
        flag = torch.tensor([{"none": 0, "nccl": 1, "peer": 2, "mc": 3, "dma": 4}[chosen]], device="cuda")     # rank 0 decides
        chunk_flag = torch.tensor([0], device="cuda")
        if chosen == "dma" and rank == 0:
            chunk_flag[0] = int(dma[best_dma]["chunk_cfgs"]) if dma[best_dma]["chunk_cfgs"] < (wl.end - wl.begin) else 0
        torch.distributed.broadcast(flag, src=0)
        torch.distributed.broadcast(chunk_flag, src=0)
        chosen = ("none", "nccl", "peer", "mc", "dma")[int(flag.item())]
        if chosen == "dma":
            wl.peer.dma_chunk_cfgs = int(chunk_flag.item())
        reassembly["chosen"] = chosen
        wl.set_mode(chosen)

    total_ms, _, issue_us = timed_steps(wl.step, args.steps, args.warmup, world, sampler, dump)
    clocks = sampler.stop()
    value = units_all * args.steps / (total_ms * 1e-3)
    kernel_ms = kernel_time_ms(wl.step)
    roofline = roofline_of(wl, kernel_ms)
    # FK + query through the public API (set_joint_configuration is part of every control-loop iteration)
    rq_ms, _, _ = timed_steps(wl.step_reconfigure, args.steps, 3, world)
    reconfigure = {"ms_per_step": rq_ms / args.steps, "value": units_all * args.steps / (rq_ms * 1e-3),
                   "what": "RobotSDF.set_joint_configuration(q[200,7]) + the headline step, device-resident inputs"}
    e2e = None
    if not args.no_e2e:
        e2e = e2e_arm(wl, units_all, world, args.steps)
        wl.restore()
    cpu = None
    if with_cpu:
        with all_host_cpus(full_affinity):
            cpu = cpu_baseline_of("c4")
    launches = wl.launches_per_step * args.steps
    wl.close()
    desc = wl.desc
    del wl
    torch.cuda.empty_cache()

    # ---- every other BASELINE config, same run ----
    others = None
    if args.workload == "default" and not args.no_workloads:
        others = {}
        for name in OTHER_WORKLOADS:
            try:
                w, res = run_workload(name, rank, world, args.steps, args.warmup, not args.no_e2e,
                                      with_cpu, None, full_affinity)
                others[name] = res
                del w
            except Exception as e:      # a secondary workload never takes the headline down with it
                others[name] = {"error": repr(e)[:300]}
                if world > 1:
                    raise               # ... but ranks must not diverge inside collectives
            torch.cuda.empty_cache()

    if rank == 0:
        # The one number the reference publishes for this path is the README shape (200 configurations x 15 251 points,
        # 8 links, per-link CachedSDF res 0.02 / padding 1.0): 2.37e7 queries/s on an RTX 2080 Ti (README.md:200;
        # BASELINE.md section 1).  The headline config (200 x 100 000) has no published number.
        vs_baseline = value / 2.37e7 if (args.workload == "c4readme" and world == 1) else None
        line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
                "warmup": args.warmup, "ms_per_step": total_ms / args.steps, "higher_is_better": True,
                "scaling": "strong", "vs_baseline": vs_baseline, "dtype": "f32", "data": "synthetic", "config": desc,
                "clocks": clocks, "e2e": e2e, "gpu_launches": launches, "roofline": roofline,
                "host_issue_us_per_step": issue_us, "cpu_baseline": cpu, "reassembly": reassembly,
                "reconfigure_and_query": reconfigure,
                "numa_binding": {"node": bound[0], "cpus": bound[1]} if bound else None,
                "workloads": others}
        print(json.dumps(line))
    return finish(world)


def finish(world):
    if world > 1:
        import torch.distributed as dist
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
