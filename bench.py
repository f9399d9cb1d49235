#!/usr/bin/env python3
"""bench.py -- RGB-D frames/s of the ORB-SLAM2 hot path (extract + SearchByProjection match + octomap insert) at
640x480 on N x B200, with the per-kernel HBM roofline and the reference's CPU path timed beside it.

Workload (BASELINE.json configs[2] shape, scene per SURVEY §8(d)): a synthetic RGB-D stream of a 6 x 3 x 6 m textured
room (RoomStream: camera on a 0.5 m Lissajous, panning <= 1.5 deg/frame, exact depth, GT floor mask), processed in the
batched many-frame mode: 297-frame batches, ORBextractor(2000,1.2,8,20,7), per frame ComputeStereoFromRGBD + grid +
SearchByProjection(cur, last, th=15); every 12th frame is a keyframe inserted into the 0.05 m occupancy map with the
floor as ground label (mode B: ground points cast free-space rays, perfect/src/MapDrawer.cc:961-969).

A STEP = one pass over SUB x 297 = 4752 frames (16 batches; the same 297 images resident in HBM are walked 16 times --
820 MB of inputs per pass, far beyond the 126 MB L2 -- with the world turned by 22.5 degrees per batch so that every batch's
keyframes fall on a differently oriented copy of the room).  With the driver's --steps 20 the timed region is > 1 s.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference] [--nfeatures 2000] [--no-cpu]
                  [--dump-outputs DIR]

N > 1 (torchrun, one rank per GPU): STRONG scaling -- the 4752 frames of a step are sharded in contiguous ranges
(+1 halo frame each, re-extracted locally), every rank maps its own keyframes, and ocm_merge_nccl (the only collective
of the path: an exchange of per-voxel clamp-add summaries over NVLink) runs INSIDE the timed region at the end of every
step; `merge` in the line says what it cost.

value   : whole-job frames/s, inputs resident in HBM, CUDA events on the pipeline's streams, max over ranks.
e2e     : the same through the reference-facing C-ABI calls with pinned HOST buffers, copies inside the timed region.
roofline: dominant kernel, algorithmic bytes (SURVEY §8(d), DESIGN.md §4) / its CUDA-event time measured live.
cpu_baseline / --impl reference: the reference's own tracking sources (oracle/_ref: src/ORBextractor.cc, Frame.cc,
          ORBmatcher.cc compiled unmodified; OpenCV primitives are bit-exact models, not OpenCV's SIMD code) frame-parallel
          on the host cores + the occupancy port (MapDrawer needs PCL/octomap: unbuildable), timed beside each other.
"""
from __future__ import annotations

import argparse
import json
import os
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

from orb_slam2_ssd_semantic_b200 import synth  # noqa: E402
from orb_slam2_ssd_semantic_b200.distributed import shard_range  # noqa: E402

ROWS, COLS = 480, 640
SCALE, NLEVELS, INI_TH, MIN_TH = 1.2, 8, 20, 7                  # perfect/Examples/RGB-D/TUM3.yaml:45-54
TH, NNRATIO = 15.0, 0.9                                        # src/Tracking.cc:1327,1346
KF_EVERY = 12   # tool/KeyFrameTrajectory_f3_walk_src.txt holds 69 keyframes for 827 frames -> 1 in 12
# frames per batched launch set (configs[2]).  297 = 2 * 148 + 1: the matcher runs one 190 KB CTA per (frame, previous
# frame) pair, one per SM, so the 296 pairs of a batch fill the 148 SMs exactly twice (256 frames = 255 pairs left the
# second wave 28 % empty).  Every other kernel has thousands of CTAs per launch and does not care.
BATCH = int(os.environ.get("BENCH_BATCH", 297))
SUB = 16        # batches per step
REF_PASSES = 2  # passes over the batch per step of the CPU arm (bounded sample)
ROOMS = 16      # distinct world orientations the batches cycle through (the map saturates after 16 passes)
S_IN = ROWS * COLS
LEVEL_PX = [640 * 480, 533 * 400, 444 * 333, 370 * 278, 309 * 231, 257 * 193, 214 * 161, 179 * 134]
S_PYR = sum(LEVEL_PX)
METRIC = "RGB-D frames/sec (extract+match+octomap) @640x480"


def algorithmic_bytes(n_kp: float, n_cand: float) -> dict:
    """Per-frame algorithmic bytes of each tracking stage (SURVEY §8(d) / DESIGN.md §4)."""
    return {
        "resize": (S_PYR - LEVEL_PX[-1]) + (S_PYR - LEVEL_PX[0]),
        "fast": S_PYR + 4 * n_cand,
        "quadtree": 4 * n_cand + 4 * n_kp,
        "blur": 2 * S_PYR,
        "orient_desc": (4 + 60) * n_kp,   # selection in, KeyPoint + descriptor out; patch gathers not counted (§8(d))
        "glue": 69 * n_kp,
        "match": 52 * n_kp + 52 * n_kp + 4 * (64 * 48 + 1) + 8 * n_kp,
    }


def pipeline_bytes(n_kp: float) -> float:
    """B_ext + B_match of SURVEY §8(d)."""
    return S_IN + 5 * S_PYR + 60 * n_kp + (52 * n_kp + 52 * n_kp + 4 * (64 * 48 + 1) + 8 * n_kp)


def map_bytes(points: float, touched: float) -> float:
    """B_map of SURVEY §8(d) per keyframe: W*H*(4+3) + 16 P + 32 U."""
    return S_IN * 7 + 16 * points + 32 * touched


def measured_peak():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md)"


def make_batch(lo: int, hi: int, seed: int = 1234):
    """Frames [lo, hi) of the BATCH-frame room stream: gray, depth f32, rgb, floor label, Tcw."""
    rs = synth.RoomStream(seed=seed, n=BATCH)
    n = hi - lo
    gray = np.empty((n, ROWS, COLS), np.uint8)
    depth = np.empty((n, ROWS, COLS), np.float32)
    rgb = np.empty((n, ROWS, COLS, 3), np.uint8)
    label = np.empty((n, ROWS, COLS), np.uint8)
    T = np.empty((n, 4, 4), np.float32)
    for i, t in enumerate(range(lo, hi)):
        gray[i], depth[i], rgb[i], T[i], label[i] = rs.frame(t, with_label=True)
    return gray, depth, rgb, label, T


def shifted_poses(T: np.ndarray, room: int) -> np.ndarray:
    """Poses of the same camera path in a world turned by room * 360/ROOMS degrees about the vertical axis through the
    world origin: Xw' = Ry Xw  =>  Rcw' = Rcw Ry^T, tcw' = tcw.  Every batch's keyframes then fall on a differently
    oriented copy of the room (the voxel grid is not rotation invariant: new cells), while the translation of Tcw --
    which the reference uses as the sensor origin of the free-space rays (perfect/src/MapDrawer.cc:619,631-632) -- stays
    where it is, so ray lengths stay those of the room."""
    a = 2.0 * np.pi * room / ROOMS
    Ry = np.array([[np.cos(a), 0, np.sin(a)], [0, 1, 0], [-np.sin(a), 0, np.cos(a)]])
    out = T.copy()
    out[:, :3, :3] = (T[:, :3, :3].astype(np.float64) @ Ry.T).astype(np.float32)
    return out


def rank_pieces(world: int, rank: int):
    """Strong scaling: the contiguous range of the SUB * BATCH frames of a step that `rank` owns, cut at batch boundaries
    -> [(batch, lo, hi)] with lo / hi relative to the batch (tests/test_distributed_cpu.py checks the partition)."""
    g_lo, g_hi = shard_range(SUB * BATCH, world, rank)
    pieces = []
    for b in range(SUB):
        lo, hi = max(g_lo, b * BATCH), min(g_hi, (b + 1) * BATCH)
        if lo < hi:
            pieces.append((b, lo - b * BATCH, hi - b * BATCH))
    return pieces


class ClockSampler(threading.Thread):
    """Samples SM clock + throttle reasons of one GPU through NVML while the timed region runs."""
    REASONS = {0x4: "sw_power_cap", 0x8: "hw_slowdown", 0x20: "sw_thermal_slowdown", 0x40: "hw_thermal_slowdown",
               0x80: "hw_power_brake_slowdown", 0x2: "applications_clocks_setting"}

    def __init__(self, index: int):
        super().__init__(daemon=True)
        self.index, self.samples, self.reasons, self.stop_flag, self.max_mhz = index, [], set(), False, None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception:
            self.nv = None

    def run(self):
        if self.nv is None:
            return
        while not self.stop_flag:
            try:
                self.samples.append(self.nv.nvmlDeviceGetClockInfo(self.h, self.nv.NVML_CLOCK_SM))
                r = self.nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for bit, name in self.REASONS.items():
                    if r & bit:
                        self.reasons.add(name)
            except Exception:
                pass
            time.sleep(0.004)

    def result(self):
        self.stop_flag = True
        if self.nv is None or not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": self.max_mhz, "reasons": ["nvml unavailable"]}
        return {"sm_mhz": float(np.median(self.samples)), "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons),
                "samples": len(self.samples)}


def _kernel_selection():
    """Which formulations / launch shapes the library runs (b200orb_get_tuning)."""
    try:
        import ctypes as C
        from orb_slam2_ssd_semantic_b200 import _lib
        m, w, q = C.c_int(), C.c_int(), C.c_int()
        _lib.lib().b200orb_get_tuning(C.byref(m), C.byref(w), C.byref(q))
        return {"experimental_mask": m.value, "fast_warps_per_cta": w.value, "quadtree_min_ctas_per_sm": q.value}
    except Exception:
        return None


def workload_config(args, world, frames_step):
    return {"workload": "synthetic 640x480 RGB-D room stream (SURVEY 8(d)), batched many-frame mode: %d-frame batches, "
                        "ORBextractor(%d,1.2,8,20,7) + stereo-from-depth + SearchByProjection(cur,last,th=15) per frame, "
                        "every %dth frame a keyframe into the 0.05 m occupancy map with the GT floor as ground label "
                        "(free-space rays); BASELINE.json configs[2] shape + keyframe path of configs[3]"
                        % (BATCH, args.nfeatures, KF_EVERY),
            "frames_per_step": frames_step, "batches_per_step": SUB, "batch_frames": BATCH,
            "keyframes_per_step": SUB * len(range(0, BATCH, KF_EVERY)), "nfeatures": args.nfeatures,
            "parallelism": ("single GPU" if world == 1 else
                            "strong scaling: contiguous frame shards x%d (+1 halo frame), ocm_merge_nccl per step" % world),
            "l2": "inputs of one pass over the resident batch (%.0f MB gray+depth+rgb+label) exceed the 126 MB L2; no "
                  "explicit flush" % (BATCH * S_IN * 9 / 1e6),
            "kernels": _kernel_selection()}


# --------------------------------------------------------------------------------------------------------------
# CPU arm
# --------------------------------------------------------------------------------------------------------------
def cpu_step(gray, depth, rgb, label, T, nthreads, nfeat, passes):
    """`passes` walks over the BATCH-frame batch on the host cores: tracking through the reference's own sources
    (frame-parallel on nthreads) while a mapping thread inserts the keyframes (GeneratePointCloud of the keyframes on
    all threads, InsertScan sequential) -- the reference maps on its own std::thread (src/pointcloudmapping.cc:43).
    -> (wall s, tracking s, mapping s, kind)"""
    from oracle import ref
    kfs = list(range(0, len(gray), KF_EVERY))
    res = {}
    use_src = ref.refsrc_available()

    def track():
        t = 0.0
        for _ in range(passes):
            if use_src:
                t += ref.src_pipeline_run(gray, depth, T, nthreads, nfeat, SCALE, NLEVELS, INI_TH, MIN_TH, synth.FX,
                                          synth.FY, synth.CX, synth.CY, synth.BF, TH, NNRATIO, True)[0]
            else:
                t += ref.pipeline_run(gray, depth, T, nthreads, nfeat, SCALE, NLEVELS, INI_TH, MIN_TH, synth.FX, synth.FY,
                                      synth.CX, synth.CY, synth.BF, TH, NNRATIO, True, 1)[0]
        res["track"] = t

    def mapper():
        occ = ref.RefOccupancy()
        t0 = time.perf_counter()
        for p in range(passes):
            occ.insert_keyframes_mt(depth, rgb, label, kfs, shifted_poses(T[kfs], p % ROOMS), synth.FX, synth.FY, synth.CX,
                                    synth.CY, nthreads)
        res["map"] = time.perf_counter() - t0

    t0 = time.perf_counter()
    th = [threading.Thread(target=track), threading.Thread(target=mapper)]
    for t in th:
        t.start()
    for t in th:
        t.join()
    wall = time.perf_counter() - t0
    return wall, res["track"], res["map"], ("reference" if use_src else "port")


def run_reference(args):
    """--impl reference: the reference's CPU implementation of the path on this box's host cores, same config."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    world = int(os.environ.get("WORLD_SIZE", "1"))
    cores = os.cpu_count() or 1
    nthreads = min(cores, 64)
    # a step of the GPU arm is SUB passes over the batch; the CPU arm times a bounded sample of it (REF_PASSES passes):
    # the reference's mapper is one thread at ~20 keyframes/s, so a full 352-keyframe step would take ~20 s
    passes = REF_PASSES
    gray, depth, rgb, label, T = make_batch(0, BATCH)
    for _ in range(min(args.warmup, 1)):
        cpu_step(gray[:max(2 * nthreads, 16)], depth, rgb, label, T[:max(2 * nthreads, 16)], nthreads, args.nfeatures, 1)
    tot = trk = mp_ = 0.0
    kind = "port"
    for _ in range(args.steps):
        w, a, b, kind = cpu_step(gray, depth, rgb, label, T, nthreads, args.nfeatures, passes)
        tot += w; trk += a; mp_ += b
    frames = BATCH * passes
    nkf = passes * len(range(0, BATCH, KF_EVERY))
    value = frames * args.steps / tot
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": "frames/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": tot / args.steps * 1e3,
        "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "u8", "data": "synthetic",
        "config": workload_config(args, world, BATCH * SUB),
        "cpu_baseline": {"value": value, "unit": "frames/s", "cores": nthreads, "kind": kind,
                         "sample": "%d frames/step (%d of the %d passes of a step over the %d-frame batch) x %d steps; tracking "
                                   "frame-parallel on %d threads beside one mapping thread" % (frames, passes, SUB, BATCH, args.steps, nthreads),
                         "tracking_fps": frames * args.steps / trk, "mapping_kf_per_s": nkf * args.steps / mp_,
                         "bottleneck": "tracking" if trk > mp_ else "mapping",
                         "tracking": "reference sources (oracle/_ref: ORBextractor.cc, Frame.cc, ORBmatcher.cc unmodified)"
                         if kind == "reference" else "oracle port", "mapping": "oracle port (MapDrawer needs PCL/octomap)"},
        "e2e": {"value": value, "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line))
    return 0


# DRAM traffic of the single-launch stages, bytes per frame, from the ncu capture named in traffic_source
NCU_DRAM_BYTES_PER_FRAME = {}
NCU_WARP_INST_PER_FRAME = {}   # smsp__inst_executed.sum per frame of the same capture (kernels with experimental mask 0)
NCU_SOURCE = None
try:
    with open(os.path.join(ROOT, "profiles", "ncu_traffic.json")) as _f:
        _j = json.load(_f)
        NCU_DRAM_BYTES_PER_FRAME, NCU_SOURCE = _j["bytes_per_frame"], _j["source"]
        NCU_WARP_INST_PER_FRAME = _j.get("warp_inst_per_frame", {})
except Exception:
    pass
# stages whose kernel changes with a bit of b200orb_experimental(): the captured instruction count no longer applies
# (bit 1, the second FAST tile staging, changes k_fast_cells' count by ~2 %: kept, see profiles/r02_notes.md)
EXPERIMENTAL_STAGE_BITS = {"orient_desc": 1}


DUMP_FRAMES = 48       # frames of the last batch whose keypoints / descriptors / matches --dump-outputs writes
DUMP_MAX_LEAVES = 1 << 20


def _device_array(torch, ptr: int, nbytes: int):
    """Host copy of nbytes of device memory at ptr, as uint8."""
    class _View:
        __cuda_array_interface__ = {"shape": (nbytes,), "typestr": "|u1", "data": (ptr, False), "version": 3}
    return torch.as_tensor(_View(), device="cuda").cpu().numpy()


def dump_outputs(out_dir, torch, trk, nframes, pcm):
    """What a caller of the timed path receives after its last step, as float32 .npy files (< 64 MB in all): per frame
    of the last batch its keypoint and match counts; for a fixed, seeded sample of DUMP_FRAMES of those frames its
    keypoints (x, y, size, angle, response, octave, class_id), descriptors (one value per byte) and cur->last match
    vector, zero / -1 past the frame's keypoint count; and the occupancy map's leaves sorted by key (key x, y, z,
    log-odds, r, g, b), a seeded sample of DUMP_MAX_LEAVES of them if there are more."""
    from orb_slam2_ssd_semantic_b200.extractor import KP_DTYPE
    os.makedirs(out_dir, exist_ok=True)
    (p_kps, p_desc, p_nkp, p_c2l, p_nm), cap = trk.device_results()
    nkp = _device_array(torch, p_nkp, 4 * nframes).view(np.int32)
    nm = _device_array(torch, p_nm, 4 * nframes).view(np.int32)
    frames = np.sort(np.random.default_rng(0).choice(nframes, min(DUMP_FRAMES, nframes), replace=False))
    kps = _device_array(torch, p_kps, KP_DTYPE.itemsize * cap * nframes).view(KP_DTYPE).reshape(nframes, cap)[frames]
    desc = _device_array(torch, p_desc, 32 * cap * nframes).reshape(nframes, cap, 32)[frames]
    c2l = _device_array(torch, p_c2l, 4 * cap * nframes).view(np.int32).reshape(nframes, cap)[frames]
    valid = np.arange(cap)[None, :] < nkp[frames][:, None]
    kp = np.stack([kps[f].astype(np.float32) for f in KP_DTYPE.names], -1)
    keys, logodds, rgb = pcm.export_leaves()
    order = np.argsort(keys[:, 0].astype(np.uint64) | (keys[:, 1].astype(np.uint64) << np.uint64(16)) |
                       (keys[:, 2].astype(np.uint64) << np.uint64(32)), kind="stable")
    if len(order) > DUMP_MAX_LEAVES:
        order = order[np.sort(np.random.default_rng(0).choice(len(order), DUMP_MAX_LEAVES, replace=False))]
    arrays = {"nkp": nkp, "nmatch": nm, "sample_frames": frames,
              "keypoints": np.where(valid[..., None], kp, 0), "descriptors": np.where(valid[..., None], desc, 0),
              "cur2last": np.where(valid, c2l, -1),
              "map_leaves": np.concatenate([keys[order], logodds[order, None], rgb[order]], 1)}
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), np.ascontiguousarray(a, np.float32))


def run_b200(args):
    import torch
    import torch.distributed as dist
    from orb_slam2_ssd_semantic_b200 import PointCloudMapping, StreamTracker
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    nfeat = args.nfeatures
    # ---- shard of this rank: contiguous range of the SUB*BATCH frames of a step, as (batch, lo, hi) pieces; the frame
    # before `lo` is the halo (re-extracted locally for the match of frame lo), batch-initial frames have none
    pieces = rank_pieces(world, rank)
    f_lo = min(max(p[1] - 1, 0) for p in pieces)
    f_hi = max(p[2] for p in pieces)
    gray, depth, rgb, label, T = make_batch(f_lo, f_hi)          # only the frames this rank touches
    nloc = f_hi - f_lo
    st = StreamTracker(nfeat, SCALE, NLEVELS, INI_TH, MIN_TH, synth.FX, synth.FY, synth.CX, synth.CY, synth.BF, TH,
                       NNRATIO, True, BATCH, device=local)
    # second tracker handle: consecutive batches alternate between the two, each on its own stream, so that the
    # latency-bound kernels of one batch (quad-tree, matcher) leave issue slots to the other's -- two batches in flight
    st_b = StreamTracker(nfeat, SCALE, NLEVELS, INI_TH, MIN_TH, synth.FX, synth.FY, synth.CX, synth.CY, synth.BF, TH,
                         NNRATIO, True, BATCH, device=local)
    d_gray, d_depth = torch.from_numpy(gray).to(dev), torch.from_numpy(depth).to(dev)
    d_rgb, d_label, d_T = torch.from_numpy(rgb).to(dev), torch.from_numpy(label).to(dev), torch.from_numpy(T).to(dev)
    pcm = PointCloudMapping(0.05, device=local)
    pcm.nccl_init(rank, world, local) if world > 1 else None
    ext = torch.cuda.ExternalStream(st.stream(), device=dev)
    ext_map = torch.cuda.ExternalStream(pcm.stream(), device=dev)
    # per piece: frames [h, hi) are tracked (h = halo or lo), keyframes = global multiples of KF_EVERY inside [lo, hi)
    plan = []
    for (b, lo, hi) in pieces:
        h = max(lo - 1, 0)
        kf = [t for t in range(lo, hi) if t % KF_EVERY == 0]
        plan.append({"room": b, "off": h - f_lo, "n": hi - h, "own": hi - lo, "kf": np.array([t - f_lo for t in kf], np.int32),
                     "Tkf": [shifted_poses(T[[t - f_lo for t in kf]], r) if kf else None for r in range(ROOMS)]})
    frames_step_total = SUB * BATCH
    own_frames = sum(p["own"] for p in plan)
    tracked_frames = sum(p["n"] for p in plan)
    npx = ROWS * COLS
    step_no = [0]

    def step_device(serial=False, with_map=True):
        k = step_no[0]
        step_no[0] += 1
        for i, p in enumerate(plan):
            o = p["off"]
            trk_h = st if (serial or (i & 1) == 0) else st_b
            trk_h.track_batch_device(d_gray.data_ptr() + o * npx, d_depth.data_ptr() + o * npx * 4, d_T.data_ptr() + o * 64,
                                     p["n"], ROWS, COLS)
            if with_map and len(p["kf"]):
                room = (k * SUB + p["room"]) % ROOMS
                pcm.insert_keyframes_device(d_depth.data_ptr(), d_rgb.data_ptr(), ROWS, COLS, p["kf"], p["Tkf"][room],
                                            synth.FX, synth.FY, synth.CX, synth.CY, d_label=d_label.data_ptr())
        if world > 1 and with_map:
            return pcm.merge()     # ocm_merge_nccl: inside the timed region
        return None

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    ext_b = torch.cuda.ExternalStream(st_b.stream(), device=dev)
    for _ in range(args.warmup):
        step_device()
    st.sync(); st_b.sync(); pcm.sync()
    launches0 = st.launch_count() + st_b.launch_count() + pcm.launch_count()
    sampler = ClockSampler(local)
    sampler.start()
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    em0, em1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(ext); em0.record(ext_map)
    ev0 = torch.cuda.Event(); ev0.record(ext); ext_b.wait_event(ev0)   # the second handle starts inside the timed region
    merge_stats, t_merge_host = [], 0.0
    for _ in range(args.steps):
        ms = step_device()
        if ms is not None:
            merge_stats.append((ms.records_sent, ms.records_total, ms.bytes_sent, ms.bytes_received))
    em1.record(ext_map)
    ev = torch.cuda.Event(); ev.record(ext_map); ext.wait_event(ev)
    evb = torch.cuda.Event(); evb.record(ext_b); ext.wait_event(evb)
    e1.record(ext)
    st.sync(); st_b.sync(); pcm.sync()
    barrier()
    clocks = sampler.result()
    if args.dump_outputs and rank == 0:
        # every batch of a step tracks the same frames; the last one ran on the handle its index selects in step_device
        dump_outputs(args.dump_outputs, torch, st if (len(plan) - 1) % 2 == 0 else st_b, plan[-1]["n"], pcm)
    ms_total, map_ms = e0.elapsed_time(e1), em0.elapsed_time(em1)
    launches = st.launch_count() + st_b.launch_count() + pcm.launch_count() - launches0
    # per-stage durations for the roofline: ONE more step, serial on one handle with the stage events on (inside the
    # timed region the stages of two batches overlap, which would smear a kernel's duration over its neighbour's)
    st.profile_enable(True)
    st.profile_read()
    step_device(serial=True, with_map=False)
    st.sync(); pcm.sync()
    stage_ms, prof_frames, prof_runs = st.profile_read()
    st.profile_enable(False)
    stage_steps = 1
    tms = torch.tensor([ms_total], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(tms, op=dist.ReduceOp.MAX)
    ms_total = float(tms.item())
    value = frames_step_total * args.steps / (ms_total * 1e-3)

    # ---- mapping alone (own stream idle otherwise): event time of one step's keyframe inserts, for the roofline ----
    pts_sum = touched_sum = 0
    upd0 = pcm.last_batch_stats()[1]
    mm0, mm1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    mm0.record(ext_map)
    nkf_alone = 0
    for p in plan:
        if len(p["kf"]):
            pcm.insert_keyframes_device(d_depth.data_ptr(), d_rgb.data_ptr(), ROWS, COLS, p["kf"], p["Tkf"][(step_no[0] * SUB + p["room"]) % ROOMS],
                                        synth.FX, synth.FY, synth.CX, synth.CY, d_label=d_label.data_ptr())
            nkf_alone += len(p["kf"])
    mm1.record(ext_map)
    pcm.sync()
    map_alone_ms = mm0.elapsed_time(mm1)
    if nkf_alone:   # P and U of the last round (<= 32 keyframes) of the last piece
        pts_sum, upd1 = pcm.last_batch_stats()
        last_round = len(plan[-1]["kf"]) % 32 or min(len(plan[-1]["kf"]), 32)
        upd_per_kf = (upd1 - upd0) / nkf_alone
    merge_alone = None
    if world > 1:
        mg0, mg1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        mg0.record(ext_map)
        msx = pcm.merge()
        mg1.record(ext_map)
        pcm.sync()
        merge_alone = {"ms": mg0.elapsed_time(mg1), "records_sent": int(msx.records_sent), "records_total": int(msx.records_total),
                       "bytes_sent": int(msx.bytes_sent), "bytes_received": int(msx.bytes_received)}

    # ---- e2e: pinned host buffers through the reference-facing calls, copies inside the timed region ----
    depth_u16 = np.rint(depth.astype(np.float64) * synth.DEPTH_FACTOR).astype(np.uint16)
    assert (depth_u16.astype(np.float32) * np.float32(1.0 / synth.DEPTH_FACTOR) == depth).all()
    pin = lambda a: torch.from_numpy(np.ascontiguousarray(a)).pin_memory()
    p_gray, p_d16, p_T = pin(gray), pin(depth_u16), pin(T)
    h_gray, h_d16, h_T = p_gray.numpy(), p_d16.numpy(), p_T.numpy()
    kf_pins = []
    for p in plan:
        if len(p["kf"]):
            kf_pins.append((pin(depth_u16[p["kf"]]), pin(rgb[p["kf"]]), pin(label[p["kf"]])))
        else:
            kf_pins.append(None)
    factor = np.float32(1.0 / synth.DEPTH_FACTOR)
    st2 = st_b
    trk = [st, st2]
    for t in trk:
        t.set_chunk_frames(int(os.environ.get("BENCH_CHUNK", BATCH)))
    outs2 = [st.alloc_outputs(BATCH, pinned=True), st2.alloc_outputs(BATCH, pinned=True)]
    e2e_k = [0]

    def submit(j, p, kp):
        # mapper first, asynchronously on its own stream: H2D depth (CV_16U) + colour + label of the keyframes only
        if kp is not None:
            room = (e2e_k[0] * SUB + p["room"]) % ROOMS
            pcm.insert_keyframes_u16(kp[0].numpy(), kp[1].numpy(), factor, p["Tkf"][room], synth.FX, synth.FY, synth.CX,
                                     synth.CY, label=kp[2].numpy())
        o, n = p["off"], p["n"]
        if not os.environ.get("BENCH_NO_CHAIN"):
            trk[j & 1].chain_after(trk[(j + 1) & 1])
        trk[j & 1].submit_batch_u16(h_gray[o:o + n], h_d16[o:o + n], factor, h_T[o:o + n], tuple(a[:n] for a in outs2[j & 1]))

    def run_host(nsteps):
        j = 0
        last = None
        for _ in range(nsteps):
            for p, kp in zip(plan, kf_pins):
                submit(j, p, kp)
                if j > 0:
                    trk[(j - 1) & 1].sync()
                last = (j & 1, p["n"])
                j += 1
            if world > 1:
                pcm.merge()
            e2e_k[0] += 1
        trk[(j - 1) & 1].sync()
        pcm.sync()
        return last

    run_host(1)
    barrier()
    t0 = time.perf_counter()
    e2e_steps = args.steps
    which, nlast = run_host(e2e_steps)
    torch.cuda.synchronize()
    t_e2e = time.perf_counter() - t0
    te = torch.tensor([t_e2e], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(te, op=dist.ReduceOp.MAX)
    e2e_value = frames_step_total * e2e_steps / float(te.item())
    # what the host link itself gives: one pinned gray batch copied alone, each direction (context for the e2e number)
    link = {}
    dgray = torch.empty_like(p_gray[:BATCH], device=dev)
    hback = torch.empty_like(p_gray[:BATCH]).pin_memory()
    for name, dst, src in (("h2d", dgray, p_gray[:BATCH]), ("d2h", hback, dgray)):
        dst.copy_(src, non_blocking=True)
        torch.cuda.synchronize()
        l0, l1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        l0.record()
        for _ in range(8):
            dst.copy_(src, non_blocking=True)
        l1.record()
        torch.cuda.synchronize()
        link[name] = 8 * src.numel() * src.element_size() / (l0.elapsed_time(l1) * 1e-3) / 1e9
    del dgray, hback
    kps, desc, nkp, c2l, nm = [a[:nlast] for a in outs2[which]]
    n_kp = float(nkp.mean())
    n_match = float(nm[1:].mean()) if nlast > 1 else 0.0
    nkf_rank = sum(len(p["kf"]) for p in plan)
    # per step and rank: gray + poses + one 32-byte sector per keypoint of the in-place depth gather, and per keyframe
    # depth u16 + colour + label
    h2d = tracked_frames * (S_IN + 64) + int(n_kp * 32) * tracked_frames + nkf_rank * S_IN * (2 + 3 + 1)
    d2h = tracked_frames * (st.cap * (28 + 32 + 4) + 8)
    th2d = torch.tensor([float(h2d), float(d2h)], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(th2d, op=dist.ReduceOp.SUM)
    h2d, d2h = int(th2d[0].item()), int(th2d[1].item())

    if rank == 0:
        from orb_slam2_ssd_semantic_b200 import _lib
        import ctypes as C
        cand = np.zeros(NLEVELS, np.int32)
        _lib.lib().orbx_candidates_per_level(_lib.lib().orbs_extractor(st._h), 0, cand.ctypes.data_as(C.c_void_p))
        n_cand = float(cand.sum())
        ab = algorithmic_bytes(n_kp, n_cand)
        peak, peak_src = measured_peak()
        stages = {}
        prof_frames = max(prof_frames, 1)
        exp_mask = int(_lib.lib().b200orb_experimental())
        n_sm = torch.cuda.get_device_properties(dev).multi_processor_count
        sm_hz = (clocks.get("sm_mhz") or clocks.get("sm_max_mhz") or 1965) * 1e6
        issue_peak = n_sm * 4 * sm_hz                # warp instructions / s: 4 schedulers per SM, one issue per clock each
        inst_tot = t_tot = 0.0
        for k, v in stage_ms.items():
            gbs = ab[k] * prof_frames / (v * 1e-3) / 1e9 if v > 0 else 0.0
            stages[k] = {"ms_per_step": v / stage_steps, "algorithmic_bytes_per_frame": ab[k], "gbs": gbs, "frac": gbs / peak}
            # the bound these kernels actually run against: the SM's instruction-issue rate (ncu: issue-active 40-80 %)
            if k in NCU_WARP_INST_PER_FRAME and not (exp_mask & EXPERIMENTAL_STAGE_BITS.get(k, 0)) and v > 0:
                wi = NCU_WARP_INST_PER_FRAME[k]
                stages[k]["warp_inst_per_frame"] = wi
                stages[k]["issue_frac"] = wi * prof_frames / (v * 1e-3) / issue_peak
                inst_tot += wi * prof_frames
                t_tot += v * 1e-3
        if nkf_alone:
            bmap = map_bytes(pts_sum / max(last_round, 1), upd_per_kf)
            gbs = bmap * nkf_alone / (map_alone_ms * 1e-3) / 1e9
            stages["mapping"] = {"ms_per_step": map_alone_ms, "algorithmic_bytes_per_keyframe": bmap, "gbs": gbs, "frac": gbs / peak,
                                 "keyframes": nkf_alone, "points_per_keyframe": pts_sum / max(last_round, 1),
                                 "voxels_updated_per_keyframe": upd_per_kf,
                                 "note": "timed alone on the map's stream after the run; in the step it overlaps tracking"}
        # dominant KERNEL: the tracking stages are one kernel each (blur, resize: one kernel family); `mapping` is the sum
        # of six kernels whose largest, k_ocm_scan_keys, is ~40 % of it (profiles/r02_launches_v4_summary.csv) -- it is
        # reported as a stage but does not compete for the dominant-kernel slot
        dom = max((k for k in stages if k != "mapping"), key=lambda k: stages[k]["ms_per_step"])
        pipe_gbs = pipeline_bytes(n_kp) * tracked_frames * args.steps / (ms_total * 1e-3) / 1e9
        line = {
            "metric": METRIC, "value": value, "unit": "frames/s",
            "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_total / args.steps,
            "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "u8", "data": "synthetic",
            "config": workload_config(args, world, frames_step_total),
            "e2e": {"value": e2e_value, "unit": "frames/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                    "batches_in_flight": 2, "steps": e2e_steps,
                    "h2d_gbs": h2d / world / (float(te.item()) / e2e_steps) / 1e9,
                    "link_gbs_measured": link,
                    "note": "h2d_gbs = bytes one rank uploads per step / its e2e step time; link_gbs_measured = a pinned "
                            "78.6 MB gray batch copied alone over the same link"},
            "gpu_launches": int(launches),
            "clocks": clocks,
            "roofline": {"kernel": dom, "bound": "hbm", "achieved": stages[dom]["gbs"], "peak": peak, "unit": "GB/s",
                         "frac": stages[dom]["frac"],
                         "traffic": (NCU_DRAM_BYTES_PER_FRAME[dom] * prof_frames / max(prof_runs, 1)
                                     if dom in NCU_DRAM_BYTES_PER_FRAME else None),
                         "traffic_source": NCU_SOURCE, "peak_source": peak_src,
                         "stages_measured": "tracking stages: one serial step on one tracker handle, nothing else on the GPU, right "
                                            "after the timed region (inside it two batches and the mapper are in flight on three "
                                            "streams and their kernels overlap); mapping: one step's keyframes alone",
                         "issue": {"bound": "instruction issue (integer / bitwise path: no kernel is HBM-bound)",
                                   "peak_warp_inst_per_s": issue_peak, "sms": n_sm,
                                   "achieved_frac_counted_stages": (inst_tot / t_tot / issue_peak) if t_tot > 0 else None,
                                   "source": "warp_inst_per_frame: smsp__inst_executed.sum of " + str(NCU_SOURCE) +
                                             "; stages whose kernel was switched by b200orb_experimental() are left out"},
                         "pipeline": {"achieved": pipe_gbs, "frac": pipe_gbs / peak,
                                      "algorithmic_bytes_per_frame": pipeline_bytes(n_kp),
                                      "note": "B_ext + B_match per tracked frame / whole timed region (mapping overlapped)"},
                         "stages": stages},
            "stats": {"batches_in_flight": 2, "keypoints_per_frame": n_kp, "fast_candidates_frame0": n_cand, "matches_per_frame": n_match,
                      "map_leaves": pcm.num_leaves(), "mapping_stream_ms_per_step": map_ms / args.steps,
                      "frames_tracked_per_step_rank0": tracked_frames, "frames_owned_per_step_rank0": own_frames,
                      "keyframes_per_step_rank0": nkf_rank, "launches_per_step": launches / args.steps},
        }
        if world > 1:
            m = np.array(merge_stats, np.float64).mean(0) if merge_stats else np.zeros(4)
            line["merge"] = {"collective": "ocm_merge_nccl: AllGather(counts) + grouped Broadcast of 24-byte voxel records, "
                                           "replayed in rank order", "in_timed_region": True, "per_step": True,
                             "records_sent_per_step_rank0": m[0], "records_total_per_step": m[1],
                             "bytes_sent_per_step_rank0": m[2], "bytes_received_per_step_rank0": m[3], "alone": merge_alone}
        if world == 1 and not args.no_cpu:
            cores = os.cpu_count() or 1
            nthreads = min(cores, 64)
            w, a, b, kind = cpu_step(gray, depth, rgb, label, T, nthreads, nfeat, 1)
            nkf = len(range(0, BATCH, KF_EVERY))
            line["cpu_baseline"] = {"value": BATCH / w, "unit": "frames/s", "cores": nthreads, "kind": kind,
                                    "sample": "one pass over the %d-frame batch (1/%d of a step), tracking frame-parallel on %d "
                                              "host threads beside one mapping thread" % (BATCH, SUB, nthreads),
                                    "tracking_fps": BATCH / a, "mapping_kf_per_s": nkf / b,
                                    "bottleneck": "tracking" if a > b else "mapping"}
        print(json.dumps(line))
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    return 0


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--nfeatures", type=int, default=2000, help="ORBextractor nfeatures (configs[2]: 2000; TUM yaml: 1000)")
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write what the last timed step computed to DIR/<name>.npy")
    args = ap.parse_args()
    args.warmup = max(args.warmup, 3) if args.impl == "b200" else args.warmup
    if args.impl == "reference":
        return run_reference(args)
    return run_b200(args)


if __name__ == "__main__":
    sys.exit(main())
