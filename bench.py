#!/usr/bin/env python
"""bench.py -- depth-frames/s of the depth-integration hot path (TSDF + ESDF every frame).

One step = one pass of the hot path over one batch of synthetic input: the 80-frame
"Replica-shape" sequence C2 of SURVEY.md 8(d) (sphere-in-box room, circular trajectory,
640x480 depth, 5 cm voxels) integrated into an empty map: per frame
    Mapper::integrateDepth  (view raycast -> block compaction/allocation -> TSDF update)
    Mapper::updateEsdf      (allocate/mark -> clear -> wavefront)
`value`  : frames/s with the depth frames already resident in HBM, device-timed (CUDA events
           on the mapper's stream), max over ranks.
`e2e`    : the same sequence through the synchronous reference-facing calls with HOST depth
           buffers (H2D of every frame and D2H of every frame's updated_blocks inside the
           timed region).
Weak scaling: every rank owns one camera stream and one map replica; the only exchange is
the NCCL merge of the ranks' updated-block lists (isaac_ros_nvblox_b200/multi_gpu.py).
`--impl reference` times the CPU restatement of the reference (oracle/, all host threads).
"""
import argparse
import json
import os
import re
import statistics
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

VOXEL = 0.05
ROWS, COLS = 480, 640
METRIC = "depth-frames/sec (TSDF+ESDF integrate, 640x480 @ 5 cm voxels)"
WORKLOAD = ("C2 Replica-shape synthetic sequence: sphere-in-box room, 80-pose circle r=4 m h=2 m, "
            "640x480 depth, 5 cm voxels, TSDF+ESDF every frame, empty map at step start")


def make_frames(num_frames, rank, world):
    from isaac_ros_nvblox_b200 import synthetic as syn
    cam = syn.PinholeCamera()
    # every rank is its own camera stream: same circle, phase-shifted start
    poses = syn.circle_trajectory(80, yaw_offset=0.0)
    shift = (rank * 80) // max(world, 1)
    poses = (poses[shift:] + poses[:shift])[:num_frames]
    return cam, syn.make_sequence(syn.sphere_in_box(), cam, poses)


BATCH = 8  # frames per rank between two merges of the ranks' block lists (BASELINE.json configs[4]: "8-frame batch")


class Workload:
    """One rank's share of a benchmark workload: the frames it integrates per step, how a frame is integrated, and the same
    on the oracle (CPU baseline + parity check). `frames`: list of (depth (H,W) f32, T_L_C 4x4 f32, mask (H,W) u8 or None)."""
    name = "c2"
    occupancy = False
    decay_every = 0

    def __init__(self, args, rank, world):
        self.args, self.rank, self.world = args, rank, world
        self.cam_s, seq = make_frames(args.frames, rank, world)
        self.frames = [(d, T, None) for d, T in seq]
        self.description = WORKLOAD
        self.parallelism = "%d independent camera streams (one map replica per GPU)" % world

    def new_mapper(self, nvb, device, voxel, esdf_mode):
        return nvb.Mapper(voxel, device=device, esdf_persistent=esdf_mode)

    def after_frame_device(self, m, i):
        pass

    def oracle_map(self, orc, frames, voxel):
        ocam = orc.Camera(self.cam_s.fu, self.cam_s.fv, self.cam_s.cu, self.cam_s.cv, self.cam_s.width, self.cam_s.height)
        o = orc.OracleMap(voxel)
        for depth, T, _ in frames:
            o.integrate_esdf(o.integrate_depth(depth, T, ocam))
        return o


class RigWorkload(Workload):
    """BASELINE.json configs[3]: a 4-camera rig (cameras at 90 degree yaw steps on one rig pose), 640x480 per camera, 5 cm voxels,
    per-camera frame shard: rank r integrates the cameras r, r + world, ... of the rig into its own map replica; the ranks merge
    their updated-block lists every 8 frames. With more than 4 ranks the rig has one camera per rank (360 / world degrees apart).
    Every rank integrates `--frames` frames per step (weak scaling): rig poses x its cameras."""
    name = "c4"

    def __init__(self, args, rank, world):
        from isaac_ros_nvblox_b200 import synthetic as syn
        import math
        self.args, self.rank, self.world = args, rank, world
        self.cam_s = syn.PinholeCamera()
        n_cams = max(4, world)
        mine = list(range(rank, n_cams, world))
        rig_poses = max(1, args.frames // len(mine))
        scene = syn.sphere_in_box()
        self.frames = []
        for j in range(rig_poses):
            theta = 2.0 * math.pi * j / 80.0
            for c in mine:
                T = syn.circle_pose(theta, yaw_offset=2.0 * math.pi * c / n_cams)
                self.frames.append((syn.render_depth(scene, self.cam_s, T), np.asarray(T, np.float32), None))
        self.description = ("C4 %d-camera synthetic rig: cameras %d degrees apart in yaw on one rig pose moving on the r=4 m circle in the "
                            "sphere-in-box room, 640x480 per camera, 5 cm voxels, TSDF+ESDF every frame, empty map at step start"
                            % (n_cams, 360 // n_cams))
        self.parallelism = ("per-camera frame shard: %d camera(s) per rank, one map replica per GPU, block-list merge every %d frames"
                            % (len(mine), BATCH))


class DynamicWorkload(Workload):
    """BASELINE.json configs[4]: dynamic scene (a sphere moving through the room) with its image-space mask, 5 cm voxels,
    ProjectiveOccupancyIntegrator on the masked pixels + ESDF from occupancy every frame + OccupancyDecayIntegrator (exclude
    last view, deallocating fully decayed blocks) every 8 frames; ranks merge their block lists every 8-frame batch."""
    name = "c5"
    occupancy = True
    decay_every = BATCH

    def __init__(self, args, rank, world):
        from isaac_ros_nvblox_b200 import synthetic as syn
        self.args, self.rank, self.world = args, rank, world
        self.cam_s = syn.PinholeCamera()
        poses = syn.circle_trajectory(80)
        shift = (rank * 80) // max(world, 1)
        poses = (poses[shift:] + poses[:shift])[:args.frames]
        self.frames = [(d, T, k) for d, T, k in syn.moving_sphere_sequence(self.cam_s, poses, step_m=0.05)]
        self.description = ("C5 dynamic-scene synthetic: sphere-in-box room + a sphere moving 5 cm per frame with its image mask, 640x480, "
                            "5 cm voxels, occupancy integrator on the masked pixels + ESDF every frame, occupancy decay (exclude last view) "
                            "every %d frames, empty map at step start" % BATCH)
        self.parallelism = "%d independent camera streams (one map replica per GPU), block-list merge every %d-frame batch" % (world, BATCH)

    def new_mapper(self, nvb, device, voxel, esdf_mode):
        return nvb.Mapper(voxel, device=device, esdf_persistent=esdf_mode, projective_layer_type=nvb.ProjectiveLayerType.kOccupancy,
                          keep_last_view=True)

    def after_frame_device(self, m, i):
        if (i + 1) % self.decay_every == 0:
            m.decay_exclude_last_view()

    def oracle_map(self, orc, frames, voxel):
        ocam = orc.Camera(self.cam_s.fu, self.cam_s.fv, self.cam_s.cu, self.cam_s.cv, self.cam_s.width, self.cam_s.height)
        o = orc.OracleMap(voxel)
        tp, dp = orc.default_tsdf_params(), orc.default_occupancy_decay_params()
        all_next = False  # Mapper::decay* hands every block to the tracker again (mapper_impl.h:208-211)
        for i, (d, T, k) in enumerate(frames):
            b = o.integrate_occupancy(d, T, ocam, tp, mask=k, mask_mode=0)
            o.integrate_esdf_occupancy(o.occupancy_block_indices() if all_next else b)
            all_next = False
            if (i + 1) % self.decay_every == 0:
                o.decay_occupancy(dp, depth=d, T_L_C=T, cam=ocam, max_view_distance_m=tp.max_integration_distance_m,
                                  truncation_distance_m=tp.truncation_distance_vox * voxel)
                all_next = True
        return o


WORKLOADS = {"c2": Workload, "c4": RigWorkload, "c5": DynamicWorkload}


class ClockSampler:
    """SM clock and throttle reasons DURING the timed region, sampled in-process through NVML every 5 ms
    (the timed region is a fraction of a second, too short for `nvidia-smi -lms`); falls back to one
    nvidia-smi query if NVML is not importable."""

    REASONS = {"hw_slowdown": 0x8, "hw_thermal_slowdown": 0x40, "sw_thermal_slowdown": 0x20, "sw_power_cap": 0x4}

    def __init__(self, index):
        self.index, self.sm, self.reasons, self.max_mhz = index, [], set(), None
        self._stop = threading.Event()
        self._thread = None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = float(pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM))
        except Exception:
            self.nv = None

    def _loop(self):
        nv = self.nv
        while not self._stop.is_set():
            try:
                self.sm.append(float(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM)))
                r = int(nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)) if hasattr(
                    nv, "nvmlDeviceGetCurrentClocksEventReasons") else int(nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h))
                for name, bit in self.REASONS.items():
                    if r & bit:
                        self.reasons.add(name)
            except Exception:
                pass
            time.sleep(0.005)

    def start(self):
        if self.nv is not None:
            self._thread = threading.Thread(target=self._loop, daemon=True)
            self._thread.start()

    def stop(self):
        if self._thread is not None:
            self._stop.set()
            self._thread.join(timeout=1)
        if not self.sm:
            try:
                out = subprocess.run(["nvidia-smi", "-i", str(self.index), "--query-gpu=clocks.sm,clocks.max.sm",
                                      "--format=csv,noheader,nounits"], capture_output=True, text=True, timeout=10).stdout
                a, b = [float(x) for x in out.strip().split(",")]
                return {"sm_mhz": a, "sm_max_mhz": b, "samples": 1, "reasons": [], "source": "nvidia-smi after the run"}
            except Exception:
                return {"sm_mhz": None, "sm_max_mhz": None, "samples": 0, "reasons": ["no clock source"]}
        return {"sm_mhz": statistics.median(self.sm), "sm_max_mhz": self.max_mhz, "samples": len(self.sm),
                "reasons": sorted(self.reasons), "source": "NVML, 5 ms period, timed region only"}


def ncu_traffic_by_kernel():
    """{kernel name fragment: dram__bytes_read.sum + dram__bytes_write.sum per launch} from the newest committed
    `ncu --set full` raw page of the bench's launch sequence (profiles/ncu_full_raw_r*.csv); {} if absent."""
    import csv
    import glob
    out = {}
    paths = sorted(glob.glob(os.path.join(ROOT, "profiles", "ncu_full_raw_r2*.csv"))) or sorted(glob.glob(os.path.join(ROOT, "profiles", "ncu_full_raw_r1_final.csv")))
    names = ("esdfWaveXKernel", "esdfWaveKernel", "esdfWaveGesKernel", "esdfMarkTmaKernel", "esdfMarkOccupancyKernel", "esdfClearKernel",
             "tsdfIntegrateKernel", "occupancyIntegrateKernel", "compactAllocateKernel", "viewRaycastKernel")
    for path in paths:
        try:
            rows = list(csv.reader(open(path)))
            hdr, units = rows[0], rows[1]
            ik, ir, iw = hdr.index("Kernel Name"), hdr.index("dram__bytes_read.sum"), hdr.index("dram__bytes_write.sum")
            scale = {"byte": 1.0, "Kbyte": 1e3, "Mbyte": 1e6, "Gbyte": 1e9}
            for n in names:
                pat = re.compile(re.escape(n) + r"T?(<[^>]*>)?(\(|$)")  # plain, templated (<0>) and ...KernelT<mode> instantiations
                vals = [float(r[ir]) * scale[units[ir]] + float(r[iw]) * scale[units[iw]] for r in rows[2:] if pat.search(r[ik])]
                if vals:
                    out[n] = sum(vals) / len(vals)
        except Exception:
            pass
    return out


def measured_peak_gbs():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    try:
        return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md)"


def cpu_threads():
    """OpenMP threads for the CPU port: its parallel regions are short (one per ESDF phase), so beyond ~16
    threads the fork/join cost outweighs the work on a many-core host."""
    return max(1, min(os.cpu_count() or 1, 16))


def cpu_baseline(wl, sample_frames, voxel=VOXEL):
    """The reference's algorithm on the host cores (oracle port, OpenMP where the reference's kernels are race-free) on the first
    `sample_frames` frames of this rank's workload (default: all of them, i.e. the same work as one GPU step). Returns the
    baseline record and the oracle map (the checker of the post-timing parity check)."""
    from oracle import oracle as orc
    orc.set_num_threads(cpu_threads())
    t0 = time.perf_counter()
    o = wl.oracle_map(orc, wl.frames[:sample_frames], voxel)
    dt = time.perf_counter() - t0
    whole = sample_frames == len(wl.frames)
    return {"value": sample_frames / dt, "unit": "frames/s", "cores": orc.num_threads(), "kind": "port",
            "sample": ("the whole %d-frame step" if whole else "first %d frames of the same sequence") % sample_frames
                      + " of workload %s, %.1f s" % (wl.name, dt)}, o


def layer_checksum(layer, fields):
    """Order-independent checksum of a {block index: voxels} layer (sum of per-block CRC32s); the same function as
    tests/helpers.py::layer_checksum."""
    import zlib
    total = 0
    for k in sorted(layer):
        h = zlib.crc32(np.asarray(k, dtype=np.int32).tobytes())
        for f in fields:
            h = zlib.crc32(np.ascontiguousarray(layer[k][f]).tobytes(), h)
        total = (total + h) & 0xFFFFFFFFFFFF
    return total


ESDF_FIELDS = ("squared_distance_vox", "parent_direction", "is_inside", "observed", "is_site")


def log_odds_layer(layer):
    """{index: {"log_odds": (8,8,8) float32}} of an occupancy layer, whatever the container."""
    return {k: {"log_odds": np.ascontiguousarray(v["log_odds"] if getattr(v, "dtype", None) is not None and v.dtype.names else v,
                                                 dtype=np.float32)} for k, v in layer.items()}


DUMP_MAX_BLOCKS = 2048  # per layer: 2048 ESDF blocks are 29 MB of float32, 2048 TSDF blocks 8 MB


def dump_outputs(out_dir, projective, esdf, occupancy):
    """Writes the map a step built as out_dir/<layer>_<field>.npy, so that two builds can be compared output for output.
    <layer>_block_indices: every allocated block, sorted, (n, 3) float64. <layer>_sample: the positions in that list of the
    blocks whose voxels are written (all of them, or DUMP_MAX_BLOCKS drawn with a fixed seed), float64.
    <layer>_<field>: those blocks' voxel field, float32."""
    os.makedirs(out_dir, exist_ok=True)
    if occupancy:
        layers = (("occupancy", log_odds_layer(projective), ("log_odds",)), ("esdf", esdf, ESDF_FIELDS))
    else:
        layers = (("tsdf", projective, ("distance", "weight")), ("esdf", esdf, ESDF_FIELDS))
    for name, layer, fields in layers:
        keys = sorted(layer)
        pick = np.arange(len(keys))
        if len(keys) > DUMP_MAX_BLOCKS:
            pick = np.sort(np.random.default_rng(0).choice(len(keys), DUMP_MAX_BLOCKS, replace=False))
        np.save(os.path.join(out_dir, name + "_block_indices.npy"), np.array(keys, np.float64).reshape(-1, 3))
        np.save(os.path.join(out_dir, name + "_sample.npy"), pick.astype(np.float64))
        for f in fields:
            np.save(os.path.join(out_dir, "%s_%s.npy" % (name, f)), np.array([layer[keys[i]][f] for i in pick], np.float32))


def parity_check(m, o, occupancy=False):
    """Post-timing check, outside every timed region: the map the benchmarked pipeline just built (device-resident
    frames, asynchronous calls, ESDF wavefront overlapping the next frame's TSDF chain) against the oracle's map of
    the same sequence: allocated block sets, projective-layer bits, all five EsdfVoxel fields."""
    if occupancy:
        p_gpu, p_cpu, pf = log_odds_layer(m.occupancy_layer().as_dict()), log_odds_layer(o.occupancy_layer()), ("log_odds",)
    else:
        p_gpu, p_cpu, pf = m.tsdf_layer().as_dict(), o.tsdf_layer(), ("distance", "weight")
    e_gpu, e_cpu = m.esdf_layer().as_dict(), o.esdf_layer()
    ok = set(p_gpu) == set(p_cpu) and set(e_gpu) == set(e_cpu)
    cs = {"projective_gpu": layer_checksum(p_gpu, pf), "projective_oracle": layer_checksum(p_cpu, pf),
          "esdf_gpu": layer_checksum(e_gpu, ESDF_FIELDS), "esdf_oracle": layer_checksum(e_cpu, ESDF_FIELDS)}
    ok = ok and cs["projective_gpu"] == cs["projective_oracle"] and cs["esdf_gpu"] == cs["esdf_oracle"]
    return bool(ok), {"projective_blocks": len(p_gpu), "esdf_blocks": len(e_gpu), "checksums": cs,
                      "what": "final %s + ESDF layers of the device-resident asynchronous pipeline (the timed one) vs the oracle on the "
                              "same frames: block sets equal, CRC32 of the voxel bytes equal" % ("occupancy" if occupancy else "TSDF")}


def run_reference(args, rank, world):
    if rank != 0:
        return
    args.frames = min(args.cpu_sample_frames, args.frames)
    wl = WORKLOADS[args.workload](args, 0, 1)
    from oracle import oracle as orc
    orc.set_num_threads(cpu_threads())

    def step():
        return wl.oracle_map(orc, wl.frames, VOXEL)

    for _ in range(args.warmup):
        step()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        o = step()
    dt = time.perf_counter() - t0
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, o.occupancy_layer() if wl.occupancy else o.tsdf_layer(), o.esdf_layer(), wl.occupancy)
    value = args.steps * len(wl.frames) / dt
    sample = "each step = the %d-frame step of workload %s on the host cores (same work as one GPU step of one rank)" % (len(wl.frames), wl.name)
    print(json.dumps({
        "impl": "reference", "metric": METRIC, "value": value, "unit": "frames/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * dt / args.steps,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": wl.description, "workload_id": wl.name, "frames_per_step": len(wl.frames), "voxel_size_m": VOXEL,
                   "parallelism": "the reference's algorithm on the host cores of rank 0 (OpenMP), the same frames as one GPU rank"},
        "cpu_baseline": {"value": value, "unit": "frames/s", "cores": orc.num_threads(), "kind": "port",
                         "sample": sample},
        "e2e": {"value": value, "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0}))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--frames", type=int, default=80)
    ap.add_argument("--cpu-sample-frames", type=int, default=80,
                    help="frames per step of the CPU arm (default: the whole sequence = the same work as a GPU step)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--esdf-host-loop", action="store_true", help="reference-like per-ring launches")
    ap.add_argument("--esdf-mode", type=int, default=3, choices=[1, 2, 3],
                    help="ESDF wavefront: 3 exchange-slab (default), 1 four-phase, 2 gather-replay")
    ap.add_argument("--workload", default="c2", choices=sorted(WORKLOADS),
                    help="c2 (default, the configuration the metric is quoted on), c4 = 4-camera rig, c5 = dynamic scene + occupancy + decay")
    ap.add_argument("--no-merge", action="store_true", help="A/B only: ranks do not merge their block lists")
    ap.add_argument("--voxel-size", type=float, default=VOXEL,
                    help="side study only (e.g. 0.02 = the Redwood-shape config): the headline metric is quoted at 0.05")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write the map the last timed step built (rank 0) as DIR/<layer>_<field>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))

    if args.impl == "reference":
        run_reference(args, rank, world)
        return

    import torch
    import torch.distributed as dist
    import __graft_entry__ as g
    g.build()
    import isaac_ros_nvblox_b200 as nvb
    from isaac_ros_nvblox_b200 import multi_gpu

    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the depth-integration path has no CPU fallback")
    torch.cuda.set_device(local_rank)
    if world > 1:
        # rank 0 must print exactly one line on stdout: NCCL's version banner (NCCL_DEBUG=VERSION) goes there too
        if os.environ.get("NCCL_DEBUG", "VERSION").upper() == "VERSION":
            os.environ["NCCL_DEBUG"] = "WARN"
        # The only collective is the all-gather of a few hundred KB of block indices per batch: two NCCL channels are plenty,
        # and their CTAs then fit the SMs the cooperative ESDF wavefront leaves free (BatchMerger reserves 4), so neither
        # kernel has to wait for the other to drain (8 GPUs, profiles/r2_scale8_ab.sh: 3 007 -> 3 194 frames/s per GPU).
        os.environ.setdefault("NCCL_MAX_NCHANNELS", "2")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))

    wl = WORKLOADS[args.workload](args, rank, world)
    cam_s, frames = wl.cam_s, wl.frames
    cam = nvb.Camera(cam_s.fu, cam_s.fv, cam_s.cu, cam_s.cv, cam_s.width, cam_s.height)
    F = len(frames)
    has_mask = frames[0][2] is not None
    depth_host = torch.from_numpy(np.stack([d for d, _, _ in frames])).pin_memory()
    depth_dev = depth_host.cuda(non_blocking=False)
    depth_host_np = [depth_host[i].numpy() for i in range(F)]  # views of the pinned buffer
    mask_host = torch.from_numpy(np.stack([k for _, _, k in frames])).pin_memory() if has_mask else None
    mask_dev = mask_host.cuda() if has_mask else None
    mask_host_np = [mask_host[i].numpy() for i in range(F)] if has_mask else [None] * F
    poses = [T for _, T, _ in frames]

    voxel = args.voxel_size
    m = wl.new_mapper(nvb, local_rank, voxel, 0 if args.esdf_host_loop else args.esdf_mode)
    stream = torch.cuda.ExternalStream(m.cuda_stream(), device=torch.device("cuda", local_rank))
    frame_bytes = ROWS * COLS * 4 + (ROWS * COLS if has_mask else 0)
    # the ranks' updated-block lists are merged every BATCH frames, device-resident and overlapped with the next batch
    merger = multi_gpu.BatchMerger(m, cap_entries=BATCH * 8192) if (world > 1 and not args.no_merge) else None

    def step_device(merge=True, timed=False):
        m.clear()
        for i in range(F):
            m.integrate_depth_device(depth_dev[i].data_ptr(), ROWS, COLS, poses[i], cam,
                                     mask_ptr=mask_dev[i].data_ptr() if has_mask else 0, mask_mode=0)
            m.update_esdf(sync=False)
            if merger is not None and merge:
                merger.append_last_frame()
                if (i + 1) % BATCH == 0 or i == F - 1:
                    merger.merge(timed=timed)
            wl.after_frame_device(m, i)

    def step_e2e():
        m.clear()
        d2h = 0
        for i in range(F):
            b = m.integrate_depth(depth_host_np[i], poses[i], cam, mask=mask_host_np[i], mask_mode=0)  # pinned host in, updated_blocks out, synchronous
            m.update_esdf()
            wl.after_frame_device(m, i)
            d2h += b.nbytes
        return d2h

    def step_e2e_async():
        # same inputs and outputs, enqueued without per-frame host synchronisation: the H2D copy of frame k+1 runs on the
        # mapper's copy stream while frame k is integrated; the step's result is read back at the end
        m.clear()
        for i in range(F):
            m.integrate_depth_host_ptr_async(depth_host[i].data_ptr(), ROWS, COLS, poses[i], cam)
            m.update_esdf(sync=False)
        m.synchronize()
        return m.tsdf_layer().get_all_block_indices().nbytes

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- device-resident throughput ----
    for _ in range(max(args.warmup, 3)):
        step_device()
    m.synchronize()
    launches0 = m.kernel_launches()
    sampler = ClockSampler(local_rank)
    barrier()
    sampler.start()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev0.record(stream)
    for _ in range(args.steps):
        step_device()
    m.join_streams()  # the last ESDF wavefront runs on the mapper's side stream
    if merger is not None:
        stream.wait_stream(merger.comm)  # ... and the last merge on the merge stream
    ev1.record(stream)
    m.synchronize()
    barrier()
    clocks = sampler.stop()
    ms = ev0.elapsed_time(ev1)
    launches = m.kernel_launches() - launches0
    t = torch.tensor([ms], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_max = float(t.item())
    value = world * F * args.steps / (ms_max * 1e-3)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, (m.occupancy_layer() if wl.occupancy else m.tsdf_layer()).as_dict(),
                     m.esdf_layer().as_dict(), wl.occupancy)

    # ---- the merge on its own: device time of all-gather + union per batch (one extra, untimed step) ----
    merge_info = None
    if merger is not None:
        step_device(timed=True)
        mm = merger.merge_ms()
        union = merger.result()
        tm = torch.tensor([statistics.median(mm)], dtype=torch.float64, device="cuda")
        dist.all_reduce(tm, op=dist.ReduceOp.MAX)
        merge_info = {"batches_per_step": len(mm), "frames_per_batch": BATCH, "ms_per_merge_median_max_over_ranks": float(tm.item()),
                      "last_union_blocks": int(union.shape[0]),
                      "protocol": "frame lists appended on the device to a fixed-capacity segment, ONE ncclAllGather of the segments per "
                                  "batch (no count exchange, no host round trip), AABB + bitset + ordered compaction on the device; on "
                                  "a side stream, overlapped with the next batch's frames"}

    # ---- end to end through the synchronous reference-facing calls, host buffers ----
    for _ in range(2):
        step_e2e()
    barrier()
    t0 = time.perf_counter()
    d2h = 0
    for _ in range(args.steps):
        d2h = step_e2e()
    barrier()
    e2e_s = time.perf_counter() - t0
    te = torch.tensor([e2e_s], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(te, op=dist.ReduceOp.MAX)
    e2e_value = world * F * args.steps / float(te.item())

    e2e_async_value, d2h_async = None, 0
    if wl.name == "c2":
        for _ in range(2):
            step_e2e_async()
        barrier()
        t0 = time.perf_counter()
        for _ in range(args.steps):
            d2h_async = step_e2e_async()
        barrier()
        ta = torch.tensor([time.perf_counter() - t0], dtype=torch.float64, device="cuda")
        if world > 1:
            dist.all_reduce(ta, op=dist.ReduceOp.MAX)
        e2e_async_value = world * F * args.steps / float(ta.item())

    # ---- BASELINE.json configs[1] shape: a colour frame with every depth frame (TSDF + colour + ESDF), device-resident ----
    with_color = None
    if world == 1 and wl.name == "c2":
        yy, xx = np.mgrid[0:ROWS, 0:COLS]
        base = np.stack([xx * 255 // (COLS - 1), yy * 255 // (ROWS - 1), ((xx // 16 + yy // 16) % 2) * 200 + 20], axis=-1)
        color_dev = torch.from_numpy(np.stack([np.roll(base, 7 * i, axis=1) for i in range(F)]).astype(np.uint8)).cuda()

        def step_color():
            m.clear()
            for i in range(F):
                m.integrate_depth_device(depth_dev[i].data_ptr(), ROWS, COLS, poses[i], cam)
                m.integrate_color_device(color_dev[i].data_ptr(), ROWS, COLS, poses[i], cam)
                m.update_esdf(sync=False)

        for _ in range(max(args.warmup, 3)):
            step_color()
        m.synchronize()
        barrier()
        l0 = m.kernel_launches()
        c0, c1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        c0.record(stream)
        for _ in range(args.steps):
            step_color()
        m.join_streams()
        c1.record(stream)
        m.synchronize()
        barrier()
        cms = c0.elapsed_time(c1)
        with_color = {"value": F * args.steps / (cms * 1e-3), "unit": "frames/s", "ms_per_step": cms / args.steps,
                      "gpu_launches": int(m.kernel_launches() - l0), "color_blocks": m.color_layer().num_blocks(),
                      "workload": "the same sequence with a 640x480 RGB frame integrated after every depth frame "
                                  "(TSDF + colour + ESDF, BASELINE.json configs[1] shape), frames resident in HBM"}
        del color_dev

    # ---- BASELINE.json configs[2] flavour ("Meshing", mesh/integrate): the mesh of the touched blocks after every frame ----
    with_mesh = None
    if world == 1 and wl.name == "c2" and not wl.occupancy:
        def step_mesh():
            m.clear()
            for i in range(F):
                m.integrate_depth_device(depth_dev[i].data_ptr(), ROWS, COLS, poses[i], cam)
                m.update_esdf(sync=False)
                m.update_mesh()  # marching cubes + weld + vertex colours of the blocks touched since the last call

        for _ in range(2):
            step_mesh()
        m.synchronize()
        l0 = m.kernel_launches()
        c0, c1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        c0.record(stream)
        for _ in range(args.steps):
            step_mesh()
        m.join_streams()
        c1.record(stream)
        m.synchronize()
        mms = c0.elapsed_time(c1)
        st = m.mesh_layer().arena_stats()
        sizes = m.mesh_layer().block_sizes(m.mesh_layer().get_all_block_indices())
        with_mesh = {"value": F * args.steps / (mms * 1e-3), "unit": "frames/s", "ms_per_step": mms / args.steps,
                     "mesh_ms_per_frame": (mms / args.steps - ms_max / args.steps) / F,
                     "gpu_launches": int(m.kernel_launches() - l0), "mesh_blocks": int(len(sizes)),
                     "vertices": int(np.maximum(sizes[:, 0], 0).sum()), "triangles": int(np.maximum(sizes[:, 1], 0).sum() // 3),
                     "arena_vertices": int(st["capacity"]),
                     "workload": "the same sequence with Mapper::updateColorMesh after every depth frame (TSDF + ESDF + incremental "
                                 "mesh, welded); mesh_ms_per_frame = extra wall time per frame over the TSDF+ESDF step, including "
                                 "the one host read-back each mesh update makes"}

    # ---- per-stage device time + algorithmic bytes for the roofline (rank 0, one extra step) ----
    roofline, stages_out, map_stats = None, None, None
    if rank == 0:
        m.clear()
        m.enable_profiling(True)
        tot = {"N": 0, "marked": 0, "swept": 0, "face_passes": 0, "clear_candidates": 0, "rings": 0, "clear_read": 0}
        for i in range(F):
            m.integrate_depth_device(depth_dev[i].data_ptr(), ROWS, COLS, poses[i], cam,
                                     mask_ptr=mask_dev[i].data_ptr() if has_mask else 0, mask_mode=0)
            m.update_esdf(sync=False)
            m.synchronize()
            tot["N"] += m.last_frame_block_count()
            s = m.esdf_integrator().last_stats()
            for k in ("marked", "swept", "face_passes", "clear_candidates", "rings"):
                tot[k] += s[k]
            tot["clear_read"] += m.esdf_integrator().clear_blocks_read()
            wl.after_frame_device(m, i)
        st = m.stage_times(reset=True)
        m.enable_profiling(False)
        # algorithmic bytes per stage over the sequence (SURVEY.md 8(d), DESIGN.md "Roofline")
        proj_block = 2048 if wl.occupancy else 4096
        raycast_b = F * (4 * 121 * 161) + tot["N"] * 12
        bytes_by_stage = {
            "view_calculator/raycast": raycast_b,
            "tsdf/integrate/allocate_blocks": tot["N"] * 16,
            "tsdf/integrate/update_blocks": 2 * proj_block * tot["N"] + F * frame_bytes,
            "esdf/integrate/mark_sites": (2 * 10240 + proj_block) * tot["marked"],
            "esdf/integrate/clear": 10240 * tot["clear_read"] + 8 * tot["clear_candidates"],  # blocks read + the skipped candidates' parent boxes
            "esdf/integrate/compute": 20480 * tot["swept"] + 3840 * tot["face_passes"],
        }
        stages_out = {}
        for name, (sms, calls) in st.items():
            gbs = (bytes_by_stage[name] / (sms * 1e-3)) / 1e9 if sms > 0 else 0.0
            stages_out[name] = {"ms_per_frame": sms / max(calls, 1), "algorithmic_GBps": gbs,
                                "algorithmic_bytes_per_frame": bytes_by_stage[name] / F}
        dom = max(st, key=lambda k: st[k][0])
        peak, peak_src = measured_peak_gbs()
        dom_ms, dom_calls = st[dom]
        achieved = (bytes_by_stage[dom] / (dom_ms * 1e-3)) / 1e9
        wave = {0: "esdf host loop", 1: "esdfWaveKernel", 2: "esdfWaveGesKernel", 3: "esdfWaveXKernel"}[0 if args.esdf_host_loop else args.esdf_mode]
        kernel_of_stage = {"esdf/integrate/compute": wave,
                           "esdf/integrate/mark_sites": "esdfMarkOccupancyKernel" if wl.occupancy else "esdfMarkTmaKernel",
                           "esdf/integrate/clear": "esdfClearKernel",
                           "tsdf/integrate/update_blocks": "occupancyIntegrateKernel" if wl.occupancy else "tsdfIntegrateKernel",
                           "tsdf/integrate/allocate_blocks": "compactAllocateKernel",
                           "view_calculator/raycast": "viewRaycastKernel"}
        traffic = ncu_traffic_by_kernel()
        for name in stages_out:
            stages_out[name]["kernel"] = kernel_of_stage.get(name)
            stages_out[name]["ncu_dram_bytes_per_launch"] = traffic.get(kernel_of_stage.get(name))
        roofline = {"bound": "hbm", "kernel": "%s (%s)" % (kernel_of_stage.get(dom, dom), dom), "achieved": achieved,
                    "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                    "traffic": traffic.get(kernel_of_stage.get(dom, dom)), "peak_source": peak_src,
                    "note": "latency/dependency-bound at 5 cm voxels (see DESIGN.md section 6); traffic = DRAM bytes per launch "
                            "from the committed ncu capture (cold cache), below the algorithmic bytes because the map is L2-resident",
                    "bytes_per_launch": bytes_by_stage[dom] / max(dom_calls, 1),
                    "avg_launch_ms": dom_ms / max(dom_calls, 1)}
        proj_layer = m.occupancy_layer() if wl.occupancy else m.tsdf_layer()
        map_stats = {"projective_blocks": proj_layer.num_blocks(), "esdf_blocks": m.esdf_layer().num_blocks(),
                     "blocks_per_frame": tot["N"] / F, "esdf_rings_per_frame": tot["rings"] / F,
                     "esdf_swept_per_frame": tot["swept"] / F, "esdf_face_passes_per_frame": tot["face_passes"] / F,
                     "esdf_clear_candidates_per_frame": tot["clear_candidates"] / F,
                     "esdf_clear_blocks_read_per_frame": tot["clear_read"] / F}

    cpu, parity_ok, parity = None, None, None
    if rank == 0 and not args.no_cpu_baseline:
        cpu, omap = cpu_baseline(wl, min(args.cpu_sample_frames, F), voxel)
        if min(args.cpu_sample_frames, F) == F:
            # the oracle has just built the map of the whole step: check the benchmarked pipeline against it
            step_device(merge=False)  # rank 0 only: no collective here
            m.synchronize()
            parity_ok, parity = parity_check(m, omap, wl.occupancy)
            if with_mesh is not None:
                # the mesh of the final map, GPU vs oracle: same blocks, same vertex / normal / index arrays
                m.update_mesh(update_full_layer=True)
                omap.integrate_mesh()
                gm, om = m.mesh_layer().as_dict(), omap.mesh_layer()
                with_mesh["parity_checked"] = bool(set(gm) == set(om) and all(
                    np.array_equal(gm[k][f], om[k][f]) for k in om for f in ("vertices", "normals", "triangles")))
        del omap

    if rank == 0:
        working_set_mb = (F * frame_bytes + (map_stats["projective_blocks"] * (2048 if wl.occupancy else 4096) + map_stats["esdf_blocks"] * 10240)) / 1e6
        e2e = {"value": e2e_value, "unit": "frames/s", "h2d_bytes_per_step": F * frame_bytes,
               "d2h_bytes_per_step": int(d2h),
               "api": "nvb_mapper_integrate_depth (pinned host depth in, updated_blocks out) + nvb_mapper_update_esdf, "
                      "both synchronous, per frame (the reference's calling convention)"}
        if e2e_async_value is not None:
            e2e["async_api"] = {"value": e2e_async_value, "unit": "frames/s", "h2d_bytes_per_step": F * frame_bytes,
                                "d2h_bytes_per_step": int(d2h_async),
                                "api": "nvb_mapper_integrate_depth_async (pinned host depth) + nvb_mapper_update_esdf_async per "
                                       "frame, one nvb_mapper_synchronize + block-index read-back per step"}
        out = {
            "metric": METRIC, "value": value, "unit": "frames/s", "n_gpus": world, "steps": args.steps,
            "warmup": max(args.warmup, 3), "ms_per_step": ms_max / args.steps, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": wl.description if voxel == VOXEL else wl.description.replace("5 cm", "%g cm" % (voxel * 100)),
                       "workload_id": wl.name, "frames_per_step": F, "voxel_size_m": voxel,
                       "parallelism": wl.parallelism,
                       "l2": "no explicit flush: one step touches %.0f MB (depth frames + map), larger than the 126 MB L2"
                             % working_set_mb,
                       "esdf_driver": "host loop" if args.esdf_host_loop else {1: "four-phase wavefront", 2: "gather-replay wavefront", 3: "exchange-slab wavefront"}[args.esdf_mode] + " (one cooperative launch)",
                       "map": map_stats},
            "e2e": e2e,
            "gpu_launches": int(launches), "clocks": clocks, "roofline": roofline, "stages": stages_out,
            "cpu_baseline": cpu, "with_color": with_color, "with_mesh": with_mesh, "merge": merge_info,
            "parity_checked": parity_ok, "parity": parity,
        }
        print(json.dumps(out))
    m.close()
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
