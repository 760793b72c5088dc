#!/usr/bin/env python
"""bench.py -- headline benchmark of the B200-native Structure-PLP-SLAM hot path.

Metric (BASELINE.json): frames/s through extract + match + pose-opt on synthetic 640x480 sequences
(8-level ORB pyramid, ~1000 kp/frame).  A "step" = one pass of the front-end
    orb_extractor::extract -> frame_tracker::motion_based_track
      (match_current_and_last_frames [+ widened retry] -> pose_optimizer::optimize -> discard_outliers)
over one batch of independent frames (SURVEY.md section 8(e): frames shard over GPUs with no collective).

  value     : device-resident throughput (images already in HBM when the timed region starts)
  e2e       : same metric through the public batched API with HOST buffers: pinned H2D of the step's images and
              D2H of the step's poses / inlier counts inside the timed region
  roofline  : dominant kernel's algorithmic bytes per launch / its mean launch time (CUDA events on the
              launching stream) vs the measured HBM peak
  cpu_baseline / --impl reference : the CPU oracle port of the same path on the host cores (the reference's
              own binary cannot be built here: no C++ OpenCV / Eigen / g2o), bounded sample.

Launch:  python bench.py --gpus N --steps K --warmup W          (N>1: via torch.distributed.run, one rank per GPU)
"""
from __future__ import annotations

import argparse
import ctypes as C
import importlib.util
import json
import os
import subprocess
import sys
import threading
import time
from concurrent.futures import ThreadPoolExecutor
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT / "tests"))

METRIC = "frames_per_sec_extract_match_poseopt"
UNIT = "frames/s"
ROWS, COLS = 480, 640
WORKLOAD = "ORB extract + Hamming match + pose-opt, 640x480, 8-level pyramid, 1000 kp/frame (BASELINE configs[1]+[2])"
# algorithmic bytes per frame of the extraction path (SURVEY.md section 8(d)); per-kernel split in DESIGN.md
PYR_PX = 950532
ALG_BYTES = {
    "fast_cells_kernel": PYR_PX,  # every pyramid level read once for FAST (+ candidates out, negligible)
    "fast_cells_kernel_v2": PYR_PX,
    "pyr_resize_kernel": None,    # per level, filled below
    "blur_tiles_kernel": 2 * PYR_PX,          # pyramid read + blurred pyramid written
    "blur_tiles_tma_kernel": 2 * PYR_PX,
    "describe_kernel": PYR_PX + 60 * 1200,
    "quadtree_kernel": 8 * 11000 + 8 * 1200,
    # match (per frame) = (M + N) x 48 B: 32 B descriptor + 16 B geometry on each side, N ~ 1200 keypoints, M ~ 1000 queries
    "point_match_kernel": 48 * (1200 + 1000),
    # pose-opt = 41 B per point edge and LM iteration (24 B position + 12 B observation + 4 B weight + 1 B flag), <= 40
    # iterations + 4 re-classification passes per call (SURVEY 8(d)); ~1000 edges per frame
    "pose_opt_kernel": 41 * 1000 * 44,
}


def _load_pkg():
    if "plpslam_b200" in sys.modules:
        return sys.modules["plpslam_b200"]
    pkg = ROOT / "structure-plp-slam_b200"
    spec = importlib.util.spec_from_file_location("plpslam_b200", pkg / "__init__.py",
                                                  submodule_search_locations=[str(pkg)])
    mod = importlib.util.module_from_spec(spec)
    sys.modules["plpslam_b200"] = mod
    spec.loader.exec_module(mod)
    return mod


def _peaks():
    p = ROOT / "MEASURED_PEAKS.json"
    if p.exists():
        d = json.loads(p.read_text())
        return float(d["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region."""

    def __init__(self, device: int):
        self.device = device
        self.samples = []
        self._stop = threading.Event()
        self._t = None

    def _run(self):
        # NVML in-process (a sample every 10 ms, so even a 100 ms timed region yields several samples under load);
        # nvidia-smi as the fallback (one sample per ~150 ms)
        try:
            import pynvml
            pynvml.nvmlInit()
            h = pynvml.nvmlDeviceGetHandleByIndex(self.device)
            mx = pynvml.nvmlDeviceGetMaxClockInfo(h, pynvml.NVML_CLOCK_SM)
            get_reasons = getattr(pynvml, "nvmlDeviceGetCurrentClocksEventReasons", None) or \
                pynvml.nvmlDeviceGetCurrentClocksThrottleReasons
            bits = [(0x8, "hw_slowdown"), (0x40, "hw_thermal_slowdown"), (0x20, "sw_thermal_slowdown"), (0x4, "sw_power_cap")]
            while not self._stop.is_set():
                sm = pynvml.nvmlDeviceGetClockInfo(h, pynvml.NVML_CLOCK_SM)
                r = int(get_reasons(h))
                self.samples.append([str(sm), str(mx)] + ["Active" if r & b else "Not Active" for b, _ in bits])
                self._stop.wait(0.01)
            return
        except Exception:
            pass
        q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        while not self._stop.is_set():
            try:
                out = subprocess.run(["nvidia-smi", f"--id={self.device}", f"--query-gpu={q}",
                                      "--format=csv,noheader,nounits"], capture_output=True, text=True, timeout=5).stdout
                parts = [x.strip() for x in out.strip().split(",")]
                if len(parts) >= 6:
                    self.samples.append(parts)
            except Exception:
                pass
            self._stop.wait(0.2)

    def __enter__(self):
        self._t = threading.Thread(target=self._run, daemon=True)
        self._t.start()
        return self

    def __exit__(self, *a):
        self._stop.set()
        self._t.join(timeout=6)

    def summary(self):
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["unavailable"]}
        sm = sorted(int(s[0]) for s in self.samples if s[0].isdigit())
        mx = max(int(s[1]) for s in self.samples if s[1].isdigit())
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for i, n in enumerate(names) if any(s[2 + i].lower().startswith("active") for s in self.samples)]
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": mx, "reasons": reasons,
                "samples": len(self.samples)}


def build_inputs(batch: int, seed: int):
    """`batch` independent tracking problems from a few rendered planar sequences (tests/scene.py)."""
    import oracle_api
    import scene
    n_seq_frames = 33
    seqs = []
    frames, t_idx = [], []
    s = 0
    while len(frames) < batch:
        seq = scene.PlanarSequence(seed=seed + 17 * s, n_frames=n_seq_frames)
        seqs.append(seq)
        for t in range(1, n_seq_frames):
            if len(frames) < batch:
                frames.append(seq.frames[t])
                t_idx.append((s, t))
        s += 1
    return seqs, np.stack(frames), t_idx


def setup_front_end(pkg, ctx, batch, seed, track_ctx=None):
    """Render frames, extract the 'last' frames once (untimed) to obtain landmark sets, upload everything."""
    import synth
    from plpslam_b200.tracking import FrontEnd
    cam = pkg.capi.make_camera(synth.FX, synth.FY, synth.CX, synth.CY, COLS, ROWS)
    fe = FrontEnd(ctx, ROWS, COLS, cam, max_batch=batch, track_ctx=track_ctx)
    seqs, frames, t_idx = build_inputs(batch, seed)
    # last-frame landmarks: extract frame t-1 of every problem on the GPU (setup, untimed)
    last_imgs = np.stack([seqs[s].frames[t - 1] for (s, t) in t_idx])
    fe.upload_images(last_imgs)
    fe.extract(batch)
    ctx.sync()
    kps = fe.download_keypoints(batch)
    rng = np.random.default_rng(seed)
    lasts = [seqs[s].last_frame_landmarks(t - 1, kps[b][0], kps[b][1]) for b, (s, t) in enumerate(t_idx)]
    preds = np.stack([seqs[s].predicted_pose(t, rng) for (s, t) in t_idx])
    pose_last = np.stack([seqs[s].poses[t - 1] for (s, t) in t_idx])
    fe.set_last_frames(lasts, preds, pose_last)
    fe.upload_images(frames)
    gt = np.stack([seqs[s].poses[t] for (s, t) in t_idx])
    return fe, frames, dict(seqs=seqs, t_idx=t_idx, lasts=lasts, preds=preds, gt=gt)


DUMP_SAMPLE_FRAMES = 64


def dump_outputs(fes, batch, out_dir: Path, seed=0):
    """Write what the last timed step handed its caller, frames in batch order, as float32 / float64 .npy files: per
    frame the pose and counts of every frame; per keypoint (keypoint fields, descriptor bytes, matched landmark index)
    for a fixed seeded sample of DUMP_SAMPLE_FRAMES frames, padded to the extractor's capacity (0, and -1 for matched)."""
    from plpslam_b200 import KP_DTYPE
    kps, trk = [], []
    for fe in fes:
        kps += fe.download_keypoints(batch)
        trk.append(fe.download_tracking(batch))
    matched = [m for t in trk for m in t["matched"]]
    n_frames, cap = len(kps), fes[0].cap
    sample = np.sort(np.random.default_rng(seed).choice(n_frames, min(n_frames, DUMP_SAMPLE_FRAMES), replace=False))
    kp_out = np.zeros((len(sample), cap, len(KP_DTYPE.names)), np.float32)
    desc_out = np.zeros((len(sample), cap, 32), np.float32)
    matched_out = np.full((len(sample), cap), -1, np.float32)
    for i, b in enumerate(sample):
        kp, desc = kps[b]
        kp_out[i, :len(kp)] = np.stack([kp[f].astype(np.float32) for f in KP_DTYPE.names], 1)
        desc_out[i, :len(kp)] = desc
        matched_out[i, :len(kp)] = matched[b]
    out = {k: np.concatenate([t[k] for t in trk]).astype(np.float64)
           for k in ("pose", "num_valid", "n_inliers", "lm_iters", "status")}
    out.update(n_keypoints=np.array([len(kp) for kp, _ in kps], np.float64), sample_frames=sample.astype(np.float64),
               keypoints=kp_out, descriptors=desc_out, matched=matched_out)
    total = sum(a.nbytes for a in out.values())
    assert total <= 64 << 20, f"output dump of {total} bytes exceeds 64 MB"
    out_dir.mkdir(parents=True, exist_ok=True)
    for name, a in out.items():
        np.save(out_dir / f"{name}.npy", a)


def host_cpu_info():
    """Logical CPUs this process may use, physical cores and the CPU model (for the cpu_baseline / reference lines)."""
    import oracle_api
    info = {"logical": oracle_api.Oracle().host_cpus(), "physical": None, "model": None}
    try:
        cores, model = set(), None
        phys, core = None, None
        for ln in open("/proc/cpuinfo"):
            k, _, v = ln.partition(":")
            k, v = k.strip(), v.strip()
            if k == "model name" and model is None:
                model = v
            elif k == "physical id":
                phys = v
            elif k == "core id":
                core = v
            elif not ln.strip():
                if phys is not None and core is not None:
                    cores.add((phys, core))
                phys, core = None, None
        info["physical"] = len(cores) or None
        info["model"] = model
    except OSError:
        pass
    return info


def cpu_port_frames(frames, aux, idxs, threads):
    """The oracle port of the same path (extract -> match [+ widened retry] -> pose-opt -> discard_outliers) on `threads`
    NATIVE host threads (oracle/frontend_mt.cc: a std::thread pool inside liboracle.so, one pinned thread per CPU,
    frames handed out by an atomic counter; the wall time is taken inside the library around the parallel region)."""
    import oracle_api
    import synth
    pkg = _load_pkg()
    orc = oracle_api.Oracle()
    p = oracle_api.orb_params()
    grid = pkg.capi.make_grid(COLS, ROWS)
    cam = pkg.capi.make_camera(synth.FX, synth.FY, synth.CX, synth.CY, COLS, ROWS)
    idxs = list(idxs)
    imgs = np.ascontiguousarray(frames[idxs])
    lasts = [aux["lasts"][b] for b in idxs]
    preds = np.stack([aux["preds"][b] for b in idxs])
    plast = np.stack([aux["seqs"][aux["t_idx"][b][0]].poses[aux["t_idx"][b][1] - 1] for b in idxs])
    r = orc.frontend_track_batch(p, grid, cam, imgs, lasts, preds, plast, 20.0, max(1, threads), pin=True)
    return len(idxs) / r["seconds"], r["seconds"], r["n_inliers"]


def build_line_frames(batch: int, seed: int, rows=ROWS, cols=COLS):
    """`batch` distinct point-and-line-rich frames (tests/synth.make_plp_texture: ~1000 ORB keypoints and ~180 keylines
    >= 60 px per 640x480 frame, BASELINE north_star "~1000 ORB + 200 line features/frame"): a few rendered scenes, each
    shifted by a different offset so that no two frames of a batch are equal."""
    import synth
    n_base = min(batch, 12)
    base = [synth.make_plp_texture(seed + i, rows, cols) for i in range(n_base)]
    rng = np.random.default_rng(seed)
    out = np.empty((batch, rows, cols), np.uint8)
    for b in range(batch):
        dx, dy = (0, 0) if b < n_base else (int(rng.integers(-60, 61)), int(rng.integers(-40, 41)))
        out[b] = np.roll(base[b % n_base], (dy, dx), axis=(0, 1))
    return out


# SURVEY 8(d) line figure with the remap skipped (identity, verified bit-exact): image read by the LSD scale pass (W H) +
# half-resolution image written and read (2 W H / 4) + the LBD blur+Sobel pass (W H read, 2 x int16 per pixel written and
# read back by the descriptor: 2 x 4 W H).  The level-line field is never materialised (DESIGN 3.6), so it is not counted:
# 10.5 W H = 3.2 MB at 640x480 (SURVEY's 3.8 MB includes the remap's read + write).
def line_alg_bytes(rows, cols):
    px, spx = rows * cols, (rows // 2) * (cols // 2)
    return 2 * px + 2 * spx + 2 * 4 * px


def bench_lines(pkg, ctx, stream, rank, world, steps, warmup, batch, seed, cpu_baseline):
    """LSD + LBD extraction (line_extractor.cc:88-160) of `batch` frames per step, device-resident; frames shard over
    ranks with no collective."""
    import torch
    import torch.distributed as dist
    from plpslam_b200.tracking import DeviceBuffer
    lib = pkg.lib()
    frames = build_line_frames(batch, seed + 1000 * rank)
    trk = pkg.LineFeatureTracker(ctx, ROWS, COLS, max_batch=batch)
    cap = trk.capacity
    d_imgs = DeviceBuffer.from_array(ctx, frames)
    d_kl = DeviceBuffer(ctx, batch * cap * pkg.KEYLINE_DTYPE.itemsize)
    d_lbd = DeviceBuffer(ctx, batch * cap * 32)
    d_fn = DeviceBuffer(ctx, batch * cap * 24)
    d_n = DeviceBuffer(ctx, batch * 4)
    d_st = DeviceBuffer(ctx, batch * 4)

    def step():
        ctx._check(lib.plp_line_extract_batch_dev(trk.handle, d_imgs.ptr, C.c_int(batch), C.c_size_t(COLS), d_kl.ptr,
                                                  d_lbd.ptr, d_fn.ptr, d_n.ptr, d_st.ptr))

    def barrier():
        ctx.sync()
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()

    for _ in range(max(warmup, 3)):
        step()
    barrier()
    l0 = ctx.launch_count()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    for _ in range(steps):
        step()
    e1.record(stream)
    barrier()
    launches = ctx.launch_count() - l0
    ms = e0.elapsed_time(e1)
    t = torch.tensor([ms], dtype=torch.float64, device=torch.cuda.current_device())
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms = float(t.item())
    n = d_n.download(np.int32, (batch,))
    st = d_st.download(np.int32, (batch,))
    assert not st.any(), "line extraction capacity overflow"
    # e2e: pinned host frames in, keylines / descriptors / line functions out, through the host entry point
    kl = np.zeros((batch, cap), pkg.KEYLINE_DTYPE)
    lbd = np.zeros((batch, cap, 32), np.uint8)
    fn = np.zeros((batch, cap, 3), np.float64)
    nn = np.zeros(batch, np.int32)

    def e2e_step():
        ctx._check(lib.plp_line_extract_batch(trk.handle, frames.ctypes.data_as(C.c_void_p), C.c_int(batch),
                                              C.c_size_t(COLS), kl.ctypes.data_as(C.c_void_p), lbd.ctypes.data_as(C.c_void_p),
                                              fn.ctypes.data_as(C.c_void_p), nn.ctypes.data_as(C.c_void_p)))

    e2e_step()
    barrier()
    t0 = time.perf_counter()
    for _ in range(steps):
        e2e_step()
    barrier()
    e2e_ms = 1e3 * (time.perf_counter() - t0) / steps
    t = torch.tensor([e2e_ms], dtype=torch.float64, device=torch.cuda.current_device())
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    e2e_ms = float(t.item())
    # one live frame through the host entry point (the region growing then runs its multi-warp, in-order-commit variant)
    lat = []
    for i in range(6):
        t0 = time.perf_counter()
        trk.extract_LSD_LBD(frames[i % batch])
        lat.append(1e3 * (time.perf_counter() - t0))
    batch1_ms = float(np.median(lat[1:]))
    # the same with the out-of-order region growing (opt-in variant 3: tickets, reorder buffer, in-order commit; §3.6)
    batch1_ooo = None
    try:
        trk.grow_variant(3)
        lat = []
        for i in range(6):
            t0 = time.perf_counter()
            trk.extract_LSD_LBD(frames[i % batch])
            lat.append(1e3 * (time.perf_counter() - t0))
        batch1_ooo = float(np.median(lat[1:]))
    except Exception as e:  # an experimental variant must not take the leg down
        batch1_ooo = f"{type(e).__name__}: {e}"
    finally:
        trk.grow_variant(0)
    # per-kernel shares
    ctx._check(lib.plp_ctx_kernel_timing(ctx.handle, 1))
    for _ in range(steps):
        step()
    buf = C.create_string_buffer(1 << 16)
    ctx._check(lib.plp_ctx_kernel_timing_report(ctx.handle, buf, C.c_size_t(len(buf))))
    ctx._check(lib.plp_ctx_kernel_timing(ctx.handle, 0))
    kt = json.loads(buf.value.decode())
    tot = sum(v["total_ms"] for v in kt.values())
    shares = {k: round(v["total_ms"] / tot, 4) for k, v in sorted(kt.items(), key=lambda kv: -kv[1]["total_ms"])}
    per_launch = {k: round(v["total_ms"] / v["count"], 4) for k, v in kt.items()}
    peak, _ = _peaks()
    alg = line_alg_bytes(ROWS, COLS) * batch
    res = {"metric": "frames_per_sec_lsd_lbd_extract", "value": world * batch * steps / (ms * 1e-3), "unit": "frames/s",
           "ms_per_step": ms / steps, "scaling": "weak",
           "config": {"workload": "LSD (refine 1, scale 0.5) + LBD line extraction, 640x480, lines >= 60 px kept",
                      "frames_per_step_per_gpu": batch, "mean_keylines_per_frame": float(n.mean()),
                      "l2": "per-step working set (3.2 MB/frame of intermediates) larger than L2"},
           "e2e": {"value": world * batch / (e2e_ms * 1e-3), "unit": "frames/s", "h2d_bytes_per_step": int(frames.nbytes),
                   "d2h_bytes_per_step": int(kl.nbytes + lbd.nbytes + fn.nbytes + nn.nbytes)},
           "gpu_launches": int(launches), "kernel_time_shares": shares, "ms_per_launch": per_launch,
           "latency_ms_one_frame": batch1_ms, "latency_ms_one_frame_out_of_order": batch1_ooo,
           "out_of_order_fallbacks": trk.ooo_fallbacks(),
           "algorithmic_bytes_per_step": alg, "hbm_roofline_frac": alg / (ms / steps * 1e-3) / 1e9 / peak}
    if cpu_baseline and rank == 0:
        import oracle_api
        orc = oracle_api.Oracle()
        cores = orc.host_cpus()
        ns = int(min(batch, max(32, 4 * cores)))
        _, dt = orc.line_extract_batch_mt(frames[:ns], cores)
        _, d1 = orc.line_extract_batch_mt(frames[:8], 1)
        res["cpu_baseline"] = {"value": ns / dt, "unit": "frames/s", "cores": cores, "kind": "port",
                               "sample": f"{ns} frames over {cores} native host threads ({dt:.2f} s)",
                               "single_thread_value": 8 / d1}
    trk.close()
    for d in (d_imgs, d_kl, d_lbd, d_fn, d_n, d_st):
        d.free()
    return res


def bench_stereo(pkg, ctx, stream, rank, world, steps, warmup, batch, seed, cpu_baseline=False):
    """BASELINE configs[4]: EuRoC-like rectified stereo 752x480, full point + line front end per stereo frame, frames
    sharded over ranks with no collective: ORB left + ORB right (frame.cc:456-457), match::stereo::compute
    (frame.cc:470-480), LSD + LBD left + right (frame.cc:458-463)."""
    import torch
    import torch.distributed as dist
    import synth
    from plpslam_b200.tracking import DeviceBuffer
    lib = pkg.lib()
    H, W = 480, 752
    n_base = min(batch, 6)
    pairs = [synth.make_stereo_pair(seed + 31 * i + 1000 * rank, H, W, plp=True) for i in range(n_base)]
    rng = np.random.default_rng(seed)
    left = np.empty((batch, H, W), np.uint8)
    right = np.empty((batch, H, W), np.uint8)
    for b in range(batch):
        sh = (0, 0) if b < n_base else (int(rng.integers(-40, 41)), int(rng.integers(-60, 61)))
        left[b] = np.roll(pairs[b % n_base][0], sh, axis=(0, 1))
        right[b] = np.roll(pairs[b % n_base][1], sh, axis=(0, 1))
    # two contexts = two streams, like the reference's left / right extraction threads (frame.cc:456-463): the right
    # image's ORB + line extraction runs on the second stream; match::stereo::compute waits for both ORB passes
    ctx_r = pkg.Context(ctx.device)
    el = pkg.OrbExtractor(ctx, H, W, max_batch=batch)
    er = pkg.OrbExtractor(ctx_r, H, W, max_batch=batch)
    ll = pkg.LineFeatureTracker(ctx, H, W, max_batch=batch)
    lr = pkg.LineFeatureTracker(ctx_r, H, W, max_batch=batch)
    cap, lcap = el.capacity, ll.capacity
    d_l, d_r = DeviceBuffer.from_array(ctx, left), DeviceBuffer.from_array(ctx, right)
    kp = [DeviceBuffer(ctx, batch * cap * pkg.KP_DTYPE.itemsize) for _ in range(2)]
    ds = [DeviceBuffer(ctx, batch * cap * 32) for _ in range(2)]
    nk = [DeviceBuffer(ctx, batch * 4) for _ in range(2)]
    st = [DeviceBuffer(ctx, batch * 4) for _ in range(4)]
    d_xr, d_dp = DeviceBuffer(ctx, batch * cap * 4), DeviceBuffer(ctx, batch * cap * 4)
    kl = [DeviceBuffer(ctx, batch * lcap * pkg.KEYLINE_DTYPE.itemsize) for _ in range(2)]
    lb = [DeviceBuffer(ctx, batch * lcap * 32) for _ in range(2)]
    fn = [DeviceBuffer(ctx, batch * lcap * 24) for _ in range(2)]
    nl = [DeviceBuffer(ctx, batch * 4) for _ in range(2)]
    bf, baseline = 47.906, 0.11

    def step():
        ctx._check(lib.plp_orb_extract_batch_dev(er.handle, d_r.ptr, C.c_int(batch), C.c_size_t(W), kp[1].ptr, ds[1].ptr,
                                                 nk[1].ptr, st[1].ptr))
        ctx._check(lib.plp_orb_extract_batch_dev(el.handle, d_l.ptr, C.c_int(batch), C.c_size_t(W), kp[0].ptr, ds[0].ptr,
                                                 nk[0].ptr, st[0].ptr))
        ctx._check(lib.plp_ctx_wait_ctx(ctx.handle, ctx_r.handle))   # the right keypoints / pyramid are ready
        ctx._check(lib.plp_line_extract_batch_dev(lr.handle, d_r.ptr, C.c_int(batch), C.c_size_t(W), kl[1].ptr, lb[1].ptr,
                                                  fn[1].ptr, nl[1].ptr, st[3].ptr))
        ctx._check(lib.plp_stereo_compute_batch_dev(ctx.handle, el.handle, er.handle, C.c_int(batch), kp[0].ptr, ds[0].ptr,
                                                    nk[0].ptr, kp[1].ptr, ds[1].ptr, nk[1].ptr, C.c_float(bf),
                                                    C.c_float(baseline), d_xr.ptr, d_dp.ptr, None))
        ctx._check(lib.plp_line_extract_batch_dev(ll.handle, d_l.ptr, C.c_int(batch), C.c_size_t(W), kl[0].ptr, lb[0].ptr,
                                                  fn[0].ptr, nl[0].ptr, st[2].ptr))
        # the next step's right-image ORB pass overwrites the right pyramid: it must wait for this stereo match
        ctx._check(lib.plp_ctx_wait_ctx(ctx_r.handle, ctx.handle))

    def barrier():
        ctx.sync()
        ctx_r.sync()
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()

    for _ in range(max(warmup, 3)):
        step()
    barrier()
    l0 = ctx.launch_count() + ctx_r.launch_count()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    for _ in range(steps):
        step()
    ctx._check(lib.plp_ctx_wait_ctx(ctx.handle, ctx_r.handle))
    e1.record(stream)
    barrier()
    launches = ctx.launch_count() + ctx_r.launch_count() - l0
    ms = e0.elapsed_time(e1)
    t = torch.tensor([ms], dtype=torch.float64, device=torch.cuda.current_device())
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms = float(t.item())
    xr = d_xr.download(np.float32, (batch, cap))
    n_left = nk[0].download(np.int32, (batch,))
    n_lines = nl[0].download(np.int32, (batch,))
    stereo_ok = float(np.mean([(xr[b, :n_left[b]] >= 0).sum() for b in range(batch)]))
    # e2e: pinned host stereo pairs in (left on the first stream, right on the second), everything frame::frame keeps
    # out (keypoints, descriptors, counts, stereo_x_right, depths, keylines, LBD rows, line functions of both images)
    from plpslam_b200.tracking import PinnedBuffer
    pin_l, pin_r = PinnedBuffer.from_array(ctx, left), PinnedBuffer.from_array(ctx, right)
    outs = [(ctx, d) for d in (kp[0], ds[0], nk[0], d_xr, d_dp, kl[0], lb[0], fn[0], nl[0])] + \
           [(ctx_r, d) for d in (kp[1], ds[1], nk[1], kl[1], lb[1], fn[1], nl[1])]
    pin_out = [PinnedBuffer(ctx, d.nbytes) for _, d in outs]

    def e2e_step():
        ctx._check(lib.plp_dev_upload_async(ctx_r.handle, d_r.ptr, pin_r.ptr, C.c_size_t(pin_r.nbytes)))
        ctx._check(lib.plp_dev_upload_async(ctx.handle, d_l.ptr, pin_l.ptr, C.c_size_t(pin_l.nbytes)))
        step()
        for (cx, d), pb in zip(outs, pin_out):
            cx._check(lib.plp_dev_download_async(cx.handle, pb.ptr, d.ptr, C.c_size_t(d.nbytes)))
        ctx.sync()
        ctx_r.sync()

    e2e_step()
    barrier()
    n_e2e = steps
    t0 = time.perf_counter()
    for _ in range(n_e2e):
        e2e_step()
    barrier()
    e2e_ms = 1e3 * (time.perf_counter() - t0) / n_e2e
    t = torch.tensor([e2e_ms], dtype=torch.float64, device=torch.cuda.current_device())
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    e2e_ms = float(t.item())
    h2d, d2h = int(pin_l.nbytes + pin_r.nbytes), int(sum(pb.nbytes for pb in pin_out))
    for pb in [pin_l, pin_r] + pin_out:
        pb.free()
    cpu = None
    if cpu_baseline and rank == 0:
        import oracle_api
        orc = oracle_api.Oracle()
        cores = orc.host_cpus()
        ns = int(min(batch, max(16, 2 * cores)))
        r = orc.stereo_frontend_batch_mt(oracle_api.orb_params(), left[:ns], right[:ns], bf, baseline, cores)
        cpu = {"value": ns / r["seconds"], "unit": "stereo frames/s", "cores": cores, "kind": "port",
               "sample": f"{ns} stereo frames over {cores} native host threads ({r['seconds']:.2f} s)"}
    ctx._check(lib.plp_ctx_kernel_timing(ctx.handle, 1))
    for _ in range(steps):
        step()
    buf = C.create_string_buffer(1 << 16)
    ctx._check(lib.plp_ctx_kernel_timing_report(ctx.handle, buf, C.c_size_t(len(buf))))
    ctx._check(lib.plp_ctx_kernel_timing(ctx.handle, 0))
    kt = json.loads(buf.value.decode())
    tot = sum(v["total_ms"] for v in kt.values())
    shares = {k: round(v["total_ms"] / tot, 4) for k, v in sorted(kt.items(), key=lambda kv: -kv[1]["total_ms"])}
    for o in (el, er, ll, lr):
        o.close()
    ctx_r.close()
    for d in [d_l, d_r, d_xr, d_dp] + kp + ds + nk + st + kl + lb + fn + nl:
        d.free()
    return {"metric": "stereo_frames_per_sec_point_line_frontend", "value": world * batch * steps / (ms * 1e-3),
            "unit": "stereo frames/s", "ms_per_step": ms / steps, "scaling": "weak",
            "config": {"workload": "rectified stereo 752x480: ORB L+R, match::stereo::compute, LSD+LBD L+R (BASELINE configs[4])",
                       "stereo_frames_per_step_per_gpu": batch, "mean_left_keypoints": float(n_left.mean()),
                       "mean_stereo_matches": stereo_ok, "mean_left_keylines": float(n_lines.mean()),
                       "parallelism": f"stereo frames sharded over {world} GPU(s), no data-path collective"},
            "e2e": {"value": world * batch / (e2e_ms * 1e-3), "unit": "stereo frames/s", "h2d_bytes_per_step": h2d,
                    "d2h_bytes_per_step": d2h},
            "cpu_baseline": cpu, "gpu_launches": int(launches), "kernel_time_shares": shares}


BA_CONFIGS = {
    # BASELINE configs[3]: 20 local + 10 fixed KF, 4000 points + 800 lines + 200 plane-owned points (~29 k edges)
    "config4": dict(seed=42, n_local=20, n_fixed=10, n_points=4000, n_lines=800, n_plane_pts=200),
    # SURVEY 8(e) scaled-up variant where landmark sharding has work to split: 60 KF x 200 k landmarks (~1.2 M edges)
    "large": dict(seed=43, n_local=30, n_fixed=30, n_points=160000, n_lines=40000, n_plane_pts=2000, fast=True),
}


def bench_ba(pkg, ctx, stream, rank, world, steps, warmup, which="config4"):
    """Second BASELINE metric: local-BA LM iterations/s, landmark-sharded over `world` GPUs with the packed reduced
    camera system all-reduced over NCCL (strong scaling: the problem size is fixed)."""
    import torch
    import torch.distributed as dist
    import ba_data
    from plpslam_b200.ba import BaComm, LocalBA, shard_boundaries, shard_edges
    kw = BA_CONFIGS[which]
    prob = ba_data.make_ba_problem(**kw)
    comm = None
    if world > 1:
        uid = [BaComm.unique_id(ctx) if rank == 0 else None]
        dist.broadcast_object_list(uid, src=0)
        comm = BaComm(ctx, uid[0], world, rank)
        sub = prob.shard(world, rank, shard_boundaries, shard_edges)
    else:
        sub = prob
    st = sub.struct()
    ba = LocalBA(ctx, st, (len(sub.kf_fixed), len(sub.pt_pos_w), len(sub.line_plucker), len(sub.pt_edge_kf),
                           len(sub.line_edge_kf)), comm=comm)
    tries_per_step = 15  # one full local BA = 5 + 10 LM iterations
    for _ in range(max(warmup, 3)):
        ba.bench_tries(tries_per_step)
    ctx.sync()
    if world > 1:
        dist.barrier()
    ar0 = comm.allreduce_count() if comm else 0
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    done = 0
    for _ in range(steps):
        it, tr = ba.bench_tries(tries_per_step)
        done += tr
    e1.record(stream)
    ctx.sync()
    ar = (comm.allreduce_count() - ar0) if comm else 0
    collective = ("NVLink peer-memory one-shot kernel" if comm.peer_active() else "ncclAllReduce") if comm else "none"
    ms = e0.elapsed_time(e1)
    t = torch.tensor([ms], dtype=torch.float64, device=torch.cuda.current_device())
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms = float(t.item())
    # full solve latency (upload excluded, result download included)
    t0 = time.perf_counter()
    out = ba.solve()
    solve_ms = 1e3 * (time.perf_counter() - t0)
    ba.close()
    if comm:
        comm.close()
    edges = len(prob.pt_edge_kf) + len(prob.line_edge_kf) + len(prob.plane_edge_lm)
    alg_bytes = edges * 32 + len(prob.pt_pos_w) * 48 + len(prob.line_plucker) * 96 + len(prob.kf_fixed) * 112
    launches_per_try = steps * (tries_per_step + 1)  # bench_tries runs tries + the lambda-init pass
    return {"metric": "local_ba_lm_iterations_per_sec", "value": done / (ms * 1e-3), "unit": "LM iterations/s",
            "scaling": "strong", "lm_tries_timed": done, "ms_per_lm_iteration": ms / max(done, 1),
            "full_solve_ms": solve_ms, "solve_iters": [out["iters_first"], out["iters_second"], out["lm_tries"]],
            "allreduces_per_try": (ar / launches_per_try) if comm else 0.0, "ranks": world, "collective": collective,
            "config": {"workload": f"local_bundle_adjuster {kw['n_local']} local + {kw['n_fixed']} fixed KF, {kw['n_points']} points + "
                                   f"{kw['n_lines']} lines + {kw['n_plane_pts']} plane edges",
                       "edges": edges, "parallelism": f"landmark-sharded over {world} GPU(s), packed all-reduce of the reduced camera system"},
            "algorithmic_bytes_per_iteration": alg_bytes,
            "hbm_roofline_frac": (alg_bytes / (ms * 1e-3 / max(done, 1))) / 1e9 / _peaks()[0]}


def ba_summary(r):
    """The part of a local-BA leg that rides in `config` of the headline line (the driver keeps `config` verbatim)."""
    return {"workload": r["config"]["workload"], "edges": r["config"]["edges"], "lm_iters_per_s": round(r["value"], 1),
            "ms_per_try": round(r["ms_per_lm_iteration"], 4), "ranks": r["ranks"],
            "allreduces_per_try": round(r["allreduces_per_try"], 3), "collective": r.get("collective", "none"),
            "full_solve_ms": round(r["full_solve_ms"], 3),
            "hbm_roofline_frac": float(f"{r['hbm_roofline_frac']:.3g}"), "scaling": "strong"}


def bench_pose_opt_config3(pkg, ctx, stream, rank, world, steps, warmup, batch=296):
    """BASELINE configs[2]: pose_optimizer_extended_line::optimize (pose_optimizer_extended_line.cc:62-305) on 1000 point +
    200 line reprojection edges per frame (SURVEY 8(d) config-3 inputs: 15 % gross outliers, N(0, 1 px x scale) noise,
    initial pose = GT o exp(N(0, diag(0.02 rad, 0.05 m))), seeds 0..batch-1), device-resident, one launch per step;
    frames shard over ranks with no collective."""
    import torch
    import torch.distributed as dist
    import synth
    from plpslam_b200.tracking import DeviceBuffer
    lib = pkg.lib()
    cam = pkg.capi.make_camera(synth.FX, synth.FY, synth.CX, synth.CY, COLS, ROWS)
    n_base = min(batch, 37)
    scenes = [synth.make_pose_opt_scene(1000 * rank + s, n_pts=1000, n_lines=200) for s in range(n_base)]
    T_in = np.stack([scenes[b % n_base][1] for b in range(batch)]).astype(np.float64)
    pts = np.concatenate([np.ascontiguousarray(scenes[b % n_base][2], pkg.PT_OBS_DTYPE) for b in range(batch)])
    lines = np.concatenate([np.ascontiguousarray(scenes[b % n_base][3], pkg.LINE_OBS_DTYPE) for b in range(batch)])
    pt_off = (1000 * np.arange(batch + 1)).astype(np.int32)
    ln_off = (200 * np.arange(batch + 1)).astype(np.int32)
    d_T, d_pts, d_lines = DeviceBuffer.from_array(ctx, T_in), DeviceBuffer.from_array(ctx, pts), DeviceBuffer.from_array(ctx, lines)
    d_po, d_lo = DeviceBuffer.from_array(ctx, pt_off), DeviceBuffer.from_array(ctx, ln_off)
    d_To, d_pout, d_lout = DeviceBuffer(ctx, batch * 128), DeviceBuffer(ctx, batch * 1000), DeviceBuffer(ctx, batch * 200)
    d_ninl, d_it = DeviceBuffer(ctx, batch * 4), DeviceBuffer(ctx, batch * 4)
    cfg = pkg.capi.PoseOptCfg(4, 10)

    def step():
        ctx._check(lib.plp_pose_optimize_batch_dev(ctx.handle, C.byref(cam), C.c_int(batch), d_T.ptr, d_pts.ptr, d_po.ptr,
                                                   d_lines.ptr, d_lo.ptr, C.c_int(1200), C.byref(cfg), d_To.ptr, d_pout.ptr,
                                                   d_lout.ptr, d_ninl.ptr, d_it.ptr))

    for _ in range(max(warmup, 3)):
        step()
    ctx.sync()
    if world > 1:
        dist.barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    for _ in range(steps):
        step()
    e1.record(stream)
    ctx.sync()
    ms = e0.elapsed_time(e1)
    t = torch.tensor([ms], dtype=torch.float64, device=torch.cuda.current_device())
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms = float(t.item()) / steps
    iters = d_it.download(np.int32, (batch,))
    ninl = d_ninl.download(np.int32, (batch,))
    lm_its = int(iters.sum())
    alg = 54800 * lm_its  # SURVEY 8(d): 1000 x 41 + 200 x 69 bytes per LM iteration
    for d in (d_T, d_pts, d_lines, d_po, d_lo, d_To, d_pout, d_lout, d_ninl, d_it):
        d.free()
    return {"workload": "pose_optimizer_extended_line, 1000 point + 200 line edges/frame (BASELINE configs[2])",
            "frames_per_step_per_gpu": batch, "frames_per_s": round(world * batch / (ms * 1e-3), 1), "ms_per_step": round(ms, 4),
            "us_per_frame_latency_bound": round(1e3 * ms, 1), "lm_iterations_per_frame": round(lm_its / batch, 2),
            "lm_iterations_per_s": round(world * lm_its / (ms * 1e-3), 1), "mean_inliers": round(float(ninl.mean()), 1),
            "algorithmic_bytes_per_step": alg, "hbm_roofline_frac": float(f"{alg / (ms * 1e-3) / 1e9 / _peaks()[0]:.3g}")}


def bench_mapping(pkg, ctx, cpu_baseline, reps=10):
    """SURVEY 8(f) rows measured through the C ABI with HOST buffers (the calls the mapping / relocalisation threads make;
    every call includes its H2D/D2H copies): match::fuse search (20 target keyframes x 1000 landmarks,
    mapping_module.cc:711-714), DBoW2 transform on a full-size synthetic vocabulary (k = 10, L = 6, 1 111 110 nodes like the
    shipped orb_vocab.dbow2) and match::bow_tree (one frame x 20 candidate keyframes, relocalizer.cc:79).  Wall clock
    around synchronous calls, median of `reps`; the CPU oracle port (one thread) of the same call beside it."""
    import bow_data
    import fuse_data
    import oracle_api
    import synth
    out = {}

    def med(fn):
        fn()
        ts = []
        for _ in range(reps):
            t0 = time.perf_counter()
            fn()
            ts.append(time.perf_counter() - t0)
        return 1e3 * float(np.median(ts))

    orc = oracle_api.Oracle() if cpu_baseline else None
    # ---- fuse
    grid = pkg.capi.make_grid(COLS, ROWS)
    cam = pkg.capi.make_camera(synth.FX, synth.FY, synth.CX, synth.CY, COLS, ROWS)
    sf, isg = synth.scale_factors(), fuse_data.inv_level_sigma_sq()
    lms, targets = fuse_data.make_point_fuse_scene(77, m=1000, num_targets=20)
    l0 = ctx.launch_count()
    ms = med(lambda: ctx.fuse_search_points(grid, cam, sf, isg, fuse_data.LOG_SF, targets, lms, 3.0, 1))
    pairs = 20 * 1000
    out["fuse_replace_duplication"] = {"ms_per_call": ms, "pairs_per_s": pairs / (ms * 1e-3), "config": "20 target keyframes x 1000 landmarks, ~1200 keypoints each",
                                       "gpu_launches": int(ctx.launch_count() - l0)}
    if orc:
        t0 = time.perf_counter()
        for t in targets:
            orc.fuse_search_points(grid, cam, sf, isg, fuse_data.LOG_SF, t, lms, 3.0, 1)
        out["fuse_replace_duplication"]["cpu_port_ms"] = 1e3 * (time.perf_counter() - t0)
    # ---- DBoW2 transform: full-size complete tree (breadth-first ids: parent(i) = (i - 1) // k)
    k, L = 10, 6
    n_nodes = (k ** (L + 1) - 1) // (k - 1)
    rng = np.random.default_rng(5)
    parent = ((np.arange(1, n_nodes, dtype=np.int64) - 1) // k).astype(np.int32)
    vdesc = rng.integers(0, 256, size=(n_nodes - 1, 32), dtype=np.uint8)
    leaf = (np.arange(1, n_nodes) >= (k ** L - 1) // (k - 1)).astype(np.uint8)
    weight = (rng.uniform(0.1, 9.7, n_nodes - 1) * leaf).astype(np.float32)
    vocab = pkg.BowVocabulary(ctx, k=k, L=L, parent=parent, desc=vdesc, weight=weight, is_leaf=leaf)
    rows = 64 * 1000
    desc = rng.integers(0, 256, size=(rows, 32), dtype=np.uint8)
    l0 = ctx.launch_count()
    ms = med(lambda: vocab.transform(desc, 4))
    alg = rows * (32 + 12 + L * k * 32)   # descriptor in, 3 outputs, k child descriptors per level (L2-resident tree)
    out["bow_transform"] = {"ms_per_call": ms, "descriptors_per_s": rows / (ms * 1e-3), "rows": rows,
                            "config": f"k={k} L={L} {n_nodes} nodes ({(n_nodes * 32) >> 20} MB of descriptors), levelsup 4",
                            "algorithmic_bytes": alg, "gathered_GBps": alg / (ms * 1e-3) / 1e9,
                            "gpu_launches": int(ctx.launch_count() - l0)}
    if orc:
        ov = orc.bow_vocab_create(k, L, parent, vdesc, weight, leaf)
        t0 = time.perf_counter()
        orc.bow_transform(ov, desc[:8000], 4)
        out["bow_transform"]["cpu_port_descriptors_per_s"] = 8000 / (time.perf_counter() - t0)
        orc.bow_vocab_destroy(ov)
    vocab.close()
    # ---- match::bow_tree: one frame x 20 candidate keyframes
    frame, bp = None, []
    for sd in range(20):
        s1, s2, _ = bow_data.make_bow_sides(100 + sd, n1=1000, n2=1000, num_nodes=90)
        if frame is None:
            frame = dict(s2)
            frame.pop("valid")
        bp.append((s1, frame))
    l0 = ctx.launch_count()
    ms = med(lambda: ctx.match_bow_tree(bp, 0.75, True))
    out["bow_tree_match"] = {"ms_per_call": ms, "pairs_per_s": 20 / (ms * 1e-3), "config": "1 frame x 20 keyframes, 1000 keypoints, ~110 nodes",
                             "gpu_launches": int(ctx.launch_count() - l0)}
    if orc:
        t0 = time.perf_counter()
        for a, b in bp:
            orc.bow_tree_match(a, b, 0.75, True)
        out["bow_tree_match"]["cpu_port_ms"] = 1e3 * (time.perf_counter() - t0)
    # ---- solve::essential_solver RANSAC (robust.cc:232: 50 hypotheses over ~500 brute-force matches)
    try:
        import ess_data
        b1, b2, matches, _ = ess_data.make_two_view(10, n=500, outlier_frac=0.3)
        smp = ess_data.draw_samples(1, len(matches), 50)
        l0 = ctx.launch_count()
        ms = med(lambda: ctx.essential_ransac(b1, b2, matches, smp, False))
        out["essential_ransac"] = {"ms_per_call": ms, "config": "500 matches, 50 eight-point hypotheses",
                                   "gpu_launches": int(ctx.launch_count() - l0)}
        if orc:
            t0 = time.perf_counter()
            orc.essential_ransac(b1, b2, matches, smp, False)
            out["essential_ransac"]["cpu_port_ms"] = 1e3 * (time.perf_counter() - t0)
    except Exception as e:
        out["essential_ransac"] = {"error": f"{type(e).__name__}: {e}"}
    # ---- Planar_Mapping_module plane RANSAC (first GPU execution of this path happens at round end, see DESIGN 3.11)
    try:
        import plane_data
        pts, valid, _, _ = plane_data.make_plane_cloud(10, n=400)
        psmp = plane_data.draw_plane_samples(0, valid, 50, 18)
        l0 = ctx.launch_count()
        ms = med(lambda: ctx.plane_ransac(pts, valid, psmp, plane_data.CFG_ESTIMATE))
        out["plane_ransac"] = {"ms_per_call": ms, "config": "400 landmarks, 50 hypotheses of 18 points",
                               "gpu_launches": int(ctx.launch_count() - l0)}
        if orc:
            want = orc.plane_ransac(pts, valid, psmp, plane_data.CFG_ESTIMATE)
            got = ctx.plane_ransac(pts, valid, psmp, plane_data.CFG_ESTIMATE)
            out["plane_ransac"]["matches_oracle"] = bool(got[0] == want[0] and np.array_equal(got[1], want[1]) and
                                                         np.array_equal(got[3], want[3]))
            t0 = time.perf_counter()
            orc.plane_ransac(pts, valid, psmp, plane_data.CFG_ESTIMATE)
            out["plane_ransac"]["cpu_port_ms"] = 1e3 * (time.perf_counter() - t0)
    except Exception as e:
        out["plane_ransac"] = {"error": f"{type(e).__name__}: {e}"}
    return out


def bench_ba_cpu(n_solves=3):
    """CPU oracle port of the same local BA (single thread, like the reference's g2o solve)."""
    import ba_data
    import oracle_api
    orc = oracle_api.Oracle()
    prob = ba_data.make_ba_problem(**BA_CONFIGS["config4"])
    t0 = time.perf_counter()
    tries = 0
    for _ in range(n_solves):
        r = ba_data.oracle_local_ba(orc, prob)
        tries += r.lm_tries
    dt = time.perf_counter() - t0
    return {"value": round(tries / dt, 2), "unit": "LM iterations/s", "cores": 1, "kind": "port",
            "sample": f"{n_solves} full local-BA solves ({tries} LM tries, {dt:.1f} s)"}


def bench_latency(pkg, ctx, n_frames=24, seed=4321, with_lines=False):
    """BASELINE configs[0] (the live-sequence plumbing loop) and SURVEY 8(d)'s batch-1 latency: ONE sequence through the
    host entry points in the order of tracking_module::track (tracking_module.cc:424-570): extract -> motion-based track
    (match_current_and_last_frames + pose_optimizer) -> search_local_landmarks (match_frame_and_landmarks,
    tracking_module.cc:908-984) -> second pose_optimizer (:749-759); frame t uses the pose estimated for frame t-1.  Every
    call takes HOST buffers and synchronises, like the reference's blocking calls.  Wall clock per frame."""
    import scene
    import synth
    from plpslam_b200.sequence import SequentialTracker
    seq = scene.PlanarSequence(seed=seed, n_frames=n_frames, plp=with_lines)
    cam = pkg.capi.make_camera(synth.FX, synth.FY, synth.CX, synth.CY, COLS, ROWS)
    trk = SequentialTracker.for_gpu(pkg, ctx, ROWS, COLS, cam, with_lines=with_lines)
    l0 = ctx.launch_count()
    res = trk.run(seq)
    launches = ctx.launch_count() - l0
    trk.close()
    st = res["stage_ms"]   # per frame, per stage
    tot = np.array([sum(f.values()) for f in st[2:]])  # the first tracked frames include lazy allocations
    med = {k: round(float(np.median([f[k] for f in st[2:]])), 3) for k in st[2]}
    err = [float(np.linalg.norm(res["poses"][t] - seq.poses[t]) / np.linalg.norm(seq.poses[t])) for t in range(1, n_frames)]
    return {"workload": "one live 640x480 sequence through the host entry points, tracking_module::track order "
                        "(extract, motion track, local-map track" + (", points + lines)" if with_lines else ", points)"),
            "frames": n_frames - 1, "ms_per_frame_median": round(float(np.median(tot)), 3),
            "ms_per_frame_p90": round(float(np.percentile(tot, 90)), 3), "frames_per_s": round(1e3 / float(np.median(tot)), 1),
            "stage_ms_median": med, "tracked_frames": int(res["tracked"]), "max_rel_pose_err_vs_gt": float(f"{max(err):.3g}"),
            "gpu_launches_per_frame": round(launches / max(n_frames - 1, 1), 1)}


def run_reference(args, rank, world):
    """--impl reference: the CPU implementation of the path (oracle port; the reference binary cannot be built here) on
    every host CPU this process may use, through the NATIVE thread pool of liboracle.so (oracle/frontend_mt.cc)."""
    if rank != 0:
        return
    import oracle_api
    orc = oracle_api.Oracle()
    hw = host_cpu_info()
    cores = hw["logical"]
    # bounded sample per step: a few frames per host thread (capped), same workload/config as the GPU arm
    per_step = int(min(512, max(16, 4 * cores)))
    seqs, frames, t_idx = build_inputs(per_step, args.seed)
    p = oracle_api.orb_params()
    rng = np.random.default_rng(args.seed)
    pkg = _load_pkg()
    import synth
    grid = pkg.capi.make_grid(COLS, ROWS)
    cam = pkg.capi.make_camera(synth.FX, synth.FY, synth.CX, synth.CY, COLS, ROWS)
    # last-frame landmarks: extract frame t-1 of every problem (setup, untimed, threaded through ctypes)
    with ThreadPoolExecutor(max_workers=min(cores, 64)) as ex:
        kps = list(ex.map(lambda st: orc.orb_extract(p, seqs[st[0]].frames[st[1] - 1]), t_idx))
    lasts = [seqs[s].last_frame_landmarks(t - 1, kps[b]["kps"], kps[b]["desc"]) for b, (s, t) in enumerate(t_idx)]
    preds = np.stack([seqs[s].predicted_pose(t, rng) for (s, t) in t_idx])
    aux = dict(seqs=seqs, t_idx=t_idx, lasts=lasts, preds=preds)
    for _ in range(max(args.warmup, 1)):
        cpu_port_frames(frames, aux, list(range(per_step)), cores)
    per = []
    ok = 0
    for _ in range(args.steps):
        fps_s, dt_s, ninl = cpu_port_frames(frames, aux, list(range(per_step)), cores)
        per.append(dt_s)
        ok = int((ninl >= 20).sum())
    dt = float(sum(per))
    fps = args.steps * per_step / dt
    fps_1, dt_1, _ = cpu_port_frames(frames, aux, list(range(min(8, per_step))), 1)
    line = {
        "impl": "reference", "metric": METRIC, "value": fps, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1e3 * dt / args.steps, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "u8/f64", "data": "synthetic",
        "config": {"workload": WORKLOAD, "frames_per_step": per_step, "tracked_ok_frames": ok,
                   "note": "reference binary unbuildable here (no C++ OpenCV/Eigen/g2o); CPU oracle port, frames spread over "
                           "a native pinned thread pool inside liboracle.so",
                   "cpu_model": hw["model"], "physical_cores": hw["physical"], "logical_cpus": cores,
                   "frames_per_s_per_logical_cpu": round(fps / cores, 3), "single_thread_frames_per_s": round(fps_1, 3),
                   "step_seconds_min_max": [round(min(per), 4), round(max(per), 4)]},
        "cpu_baseline": {"value": fps, "unit": UNIT, "cores": cores, "kind": "port",
                         "sample": f"{per_step} frames/step x {args.steps} steps"},
        "e2e": {"value": fps, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line))


def _round_floats(o, nd=6):
    if isinstance(o, float):
        return float(f"{o:.{nd}g}")
    if isinstance(o, dict):
        return {k: _round_floats(v, nd) for k, v in o.items()}
    if isinstance(o, (list, tuple)):
        return [_round_floats(v, nd) for v in o]
    return o


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--batch", type=int, default=512,
                    help="frames per step per GPU (512 x 307 KB > 126 MB L2); measured r01f: 2 x 296 (whole waves of the "
                         "one-CTA-per-frame kernels) is 1 % slower than 2 x 256 -- the tracking streams already overlap")
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--seed", type=int, default=1234)
    ap.add_argument("--streams", type=int, default=2, help="sub-batches in flight per GPU (one context/stream each)")
    ap.add_argument("--track-streams", type=int, default=1,
                    help="1: matcher / pose optimiser of every sub-batch on a high-priority stream of its own")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-ba", action="store_true", help="skip the local-BA metric")
    ap.add_argument("--no-ba-large", action="store_true", help="skip the scaled-up local-BA problem (60 KF x 200 k landmarks)")
    ap.add_argument("--no-pose3", action="store_true", help="skip the config-3 pose-opt leg (1000 point + 200 line edges)")
    ap.add_argument("--no-latency", action="store_true", help="skip the sequential batch-1 latency leg (config 1)")
    ap.add_argument("--no-lines", action="store_true", help="skip the LSD+LBD line front-end metric")
    ap.add_argument("--only-lines", action="store_true", help="development: run only the line front-end leg")
    ap.add_argument("--no-mapping", action="store_true", help="skip the fuse / BoW legs (SURVEY 8(f) rows)")
    ap.add_argument("--no-stereo", action="store_true", help="skip the stereo point+line front-end leg (configs[4])")
    ap.add_argument("--only-stereo", action="store_true", help="development: run only the stereo leg")
    ap.add_argument("--only-ba", action="store_true", help="development: run only the local-BA legs")
    ap.add_argument("--stereo-batch", type=int, default=148, help="stereo frames per step per GPU")
    ap.add_argument("--line-batch", type=int, default=1776, help="frames per step per GPU of the line front-end leg")
    ap.add_argument("--detail", default=None, help="file for the full per-leg JSON (default: none written)")
    ap.add_argument("--dump-outputs", default=None, metavar="DIR",
                    help="write what the last timed step of the headline path returned (rank 0's frames) to DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    args.warmup = max(args.warmup, 3) if args.impl == "b200" else args.warmup

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))

    if args.impl == "reference":
        run_reference(args, rank, world)
        return

    import torch
    import torch.distributed as dist
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device(f"cuda:{local_rank}"))
    torch.cuda.set_device(local_rank)
    pkg = _load_pkg()
    ctx = pkg.Context(local_rank)
    lib = pkg.lib()
    B = args.batch
    stream = torch.cuda.ExternalStream(lib.plp_ctx_stream(ctx.handle), device=f"cuda:{local_rank}")
    if args.only_lines:
        r = bench_lines(pkg, ctx, stream, rank, world, args.steps, args.warmup, args.line_batch, args.seed,
                        world == 1 and not args.no_cpu_baseline)
        if rank == 0:
            print(json.dumps(r))
        return
    if args.only_stereo:
        r = bench_stereo(pkg, ctx, stream, rank, world, args.steps, args.warmup, args.stereo_batch, args.seed,
                         world == 1 and not args.no_cpu_baseline)
        if rank == 0:
            print(json.dumps(r))
        return
    if args.only_ba:
        out = {"local_ba": bench_ba(pkg, ctx, stream, rank, world, args.steps, args.warmup, "config4")}
        if not args.no_ba_large:
            out["local_ba_large"] = bench_ba(pkg, ctx, stream, rank, world, args.steps, 1, "large")
        if rank == 0:
            print(json.dumps(out))
        if world > 1:
            dist.destroy_process_group()
        return
    # The batch of a step is split into `--streams` sub-batches, each owned by its own context (= CUDA stream) with its
    # own extractor / tracker handles: the H2D copy, the one-CTA-per-frame matcher / pose optimiser and the D2H copy of
    # one sub-batch overlap the extraction kernels of the other (plain stream concurrency, no graph capture).
    S = max(1, min(args.streams, B))
    Bs = B // S
    B = Bs * S
    ctxs = [ctx] + [pkg.Context(local_rank) for _ in range(S - 1)]
    # tracking (one CTA per frame: matcher, pose optimiser) on high-priority streams of its own
    tctxs = [pkg.Context(local_rank, high_priority=True) for _ in range(S)] if args.track_streams else [None] * S
    fes, frames_l, auxs = [], [], []
    for c in range(S):
        fe_c, fr_c, aux_c = setup_front_end(pkg, ctxs[c], Bs, args.seed + 1000 * rank + 37 * c, tctxs[c])
        fes.append(fe_c)
        frames_l.append(fr_c)
        auxs.append(aux_c)
    fe, frames, aux = fes[0], np.concatenate(frames_l), auxs[0]

    all_ctxs = ctxs + [t for t in tctxs if t is not None]

    def barrier():
        for cx in all_ctxs:
            cx.sync()
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()

    def join_streams():  # stream 0 waits for the work enqueued on the other streams
        for cx in all_ctxs[1:]:
            ctx._check(lib.plp_ctx_wait_ctx(ctx.handle, cx.handle))

    def step_all():
        for c in range(S):
            fes[c].step(Bs)

    # ---------------- value: device-resident ------------------------------------------------------------
    for _ in range(args.warmup):
        step_all()
    barrier()
    launches0 = sum(cx.launch_count() for cx in all_ctxs)
    with ClockSampler(local_rank) as clk:
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        for _ in range(args.steps):
            step_all()
        join_streams()
        e1.record(stream)
        barrier()
        ms = e0.elapsed_time(e1)
    launches = sum(cx.launch_count() for cx in all_ctxs) - launches0
    ok = 0
    for c in range(S):
        ok += int((fes[c].download_tracking(Bs)["num_valid"] >= 20).sum())
    t = torch.tensor([ms], dtype=torch.float64, device=f"cuda:{local_rank}")
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_max = float(t.item())
    value = world * B * args.steps / (ms_max * 1e-3)
    if args.dump_outputs and rank == 0:
        dump_outputs(fes, Bs, Path(args.dump_outputs))

    # ---------------- e2e: host buffers, every copy of a step inside the timed region -------------------
    # per step and sub-batch, from / to PINNED host memory: H2D of the images AND of that step's last-frame landmarks
    # (positions, octaves, angles, descriptors, validity, offsets) and predicted / last poses; D2H of everything the
    # host-side data::frame needs: keypoints, descriptors, counts, the landmark index kept on every keypoint, poses,
    # valid / inlier counts, LM iterations, status (full-capacity arrays: the API's fixed per-frame stride).
    for c in range(S):
        fes[c].stage_host_io(frames_l[c])
    h2d_bytes = sum(f.h2d_bytes_per_step for f in fes)
    d2h_bytes = sum(f.d2h_bytes_per_step for f in fes)

    def e2e_step():
        for c in range(S):
            f = fes[c]
            f.upload_inputs_async()
            f.step(Bs)
            f.download_outputs_async()

    for _ in range(2):
        e2e_step()
    barrier()
    f0, f1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    f0.record(stream)
    for _ in range(args.steps):
        e2e_step()
    join_streams()
    f1.record(stream)
    barrier()
    e2e_ms = f0.elapsed_time(f1)
    # the results of the last step are in host memory now: read them (the "loss or metric" of the contract)
    e2e_ok, e2e_kp = 0, 0
    for c in range(S):
        hr = fes[c].host_results()
        e2e_ok += int((hr["num_valid"] >= 20).sum())
        e2e_kp += int(hr["n_kp"].sum())
    t = torch.tensor([e2e_ms], dtype=torch.float64, device=f"cuda:{local_rank}")
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    e2e_value = world * B * args.steps / (float(t.item()) * 1e-3)

    # ---------------- roofline: per-kernel event timing over the same steps ------------------------------
    tim_ctxs = [fe.ctx] + ([fe.track_ctx] if fe.track_ctx is not fe.ctx else [])
    for cx in tim_ctxs:
        cx._check(lib.plp_ctx_kernel_timing(cx.handle, 1))
    for _ in range(args.steps):
        fe.step(Bs)
    kt = {}
    for cx in tim_ctxs:
        buf = C.create_string_buffer(1 << 16)
        cx._check(lib.plp_ctx_kernel_timing_report(cx.handle, buf, C.c_size_t(len(buf))))
        cx._check(lib.plp_ctx_kernel_timing(cx.handle, 0))
        kt.update(json.loads(buf.value.decode()))
    total_ms = sum(v["total_ms"] for v in kt.values())
    shares = {k: round(v["total_ms"] / total_ms, 4) for k, v in sorted(kt.items(), key=lambda kv: -kv[1]["total_ms"])}
    dom = max(kt.items(), key=lambda kv: kv[1]["total_ms"])
    peak, peak_src = _peaks()
    dom_name = dom[0]
    per_launch_ms = dom[1]["total_ms"] / dom[1]["count"]
    launches_per_step = dom[1]["count"] / max(args.steps, 1)
    alg = ALG_BYTES.get(dom_name.split("<")[0])
    if alg is None:
        alg = PYR_PX
    # algorithmic bytes of ONE step of this kernel (all of its launches in a step together process the sub-batch once:
    # the matcher's second launch only revisits the few frames that need the wider margin) over its time per step
    alg_bytes_launch = alg * Bs
    per_step_ms = dom[1]["total_ms"] / max(args.steps, 1)
    achieved = alg_bytes_launch / (per_step_ms * 1e-3) / 1e9
    traffic, traffic_src = None, None
    tf = sorted((ROOT / "profiles").glob("traffic_*.json"))
    if tf:  # dram__bytes_read.sum + dram__bytes_write.sum of the committed `ncu --set full` capture, scaled to this launch
        tj = json.loads(tf[-1].read_text())
        kk = tj["kernels"].get(dom_name) or tj["kernels"].get(dom_name.replace("_v2", ""))
        if kk:
            traffic = (kk["dram_bytes_read"] + kk["dram_bytes_write"]) / tj["frames_per_launch"] * Bs
            traffic_src = f"{tf[-1].name}: {tj['source']}; per-frame bytes x {Bs} frames"
    # whole-step figure beside the dominant kernel's: all algorithmic bytes of a frame over the step time
    step_alg = (2604396 + 48 * 2200 + 41 * 1000 * 44) * B
    roofline = {"bound": "hbm", "kernel": dom_name, "achieved": achieved, "peak": peak, "unit": "GB/s",
                "frac": achieved / peak, "traffic": traffic, "traffic_source": traffic_src, "peak_source": peak_src,
                "algorithmic_bytes_per_launch": alg_bytes_launch, "ms_per_launch": per_launch_ms,
                "launches_per_step": launches_per_step, "ms_per_step_of_this_kernel": per_step_ms,
                "kernel_time_shares": shares, "kernel_ms_per_step": {k: round(v["total_ms"] / max(args.steps, 1), 4) for k, v in kt.items()},
                "frames_per_launch": Bs,
                "whole_step": {"algorithmic_bytes": step_alg, "achieved": step_alg / (ms_max / args.steps * 1e-3) / 1e9,
                               "frac": step_alg / (ms_max / args.steps * 1e-3) / 1e9 / peak},
                "how": "CUDA events around every launch on the launching stream over a repeat of the timed steps "
                       "(one sub-batch, kernels serialised)"}

    detail = {}
    cfg_extra = {}
    if not args.no_ba:
        r = bench_ba(pkg, ctx, stream, rank, world, steps=args.steps, warmup=args.warmup, which="config4")
        if rank == 0 and world == 1 and not args.no_cpu_baseline:
            r["cpu_baseline"] = bench_ba_cpu()
        detail["local_ba"] = r
        cfg_extra["local_ba"] = ba_summary(r)
        if "cpu_baseline" in r:
            cfg_extra["local_ba"]["cpu_port_lm_iters_per_s"] = r["cpu_baseline"]["value"]
        if not args.no_ba_large:
            r = bench_ba(pkg, ctx, stream, rank, world, steps=args.steps, warmup=1, which="large")
            detail["local_ba_large"] = r
            cfg_extra["local_ba_large"] = ba_summary(r)
    if not args.no_pose3:
        r = bench_pose_opt_config3(pkg, ctx, stream, rank, world, args.steps, args.warmup)
        detail["pose_opt_config3"] = r
        cfg_extra["pose_opt_config3"] = r
    if not args.no_latency and rank == 0:
        try:
            r = bench_latency(pkg, ctx)
        except Exception as e:  # an auxiliary leg must not take the headline line down with it; say so loudly
            r = {"error": f"{type(e).__name__}: {e}"}
        detail["latency_batch1"] = r
        cfg_extra["latency_batch1"] = r
    if world > 1:
        dist.barrier()
    if not args.no_lines:
        r = bench_lines(pkg, ctx, stream, rank, world, args.steps, args.warmup, args.line_batch, args.seed,
                        world == 1 and not args.no_cpu_baseline)
        detail["line_frontend"] = r
        cfg_extra["line_frontend"] = {"frames_per_s": round(r["value"], 1), "e2e_frames_per_s": round(r["e2e"]["value"], 1),
                                      "mean_keylines_per_frame": round(r["config"]["mean_keylines_per_frame"], 1),
                                      "hbm_roofline_frac": float(f"{r['hbm_roofline_frac']:.3g}"),
                                      "frames_per_step_per_gpu": args.line_batch,
                                      "latency_ms_one_frame": round(r["latency_ms_one_frame"], 2),
                                      "latency_ms_one_frame_out_of_order": (round(r["latency_ms_one_frame_out_of_order"], 2)
                                                                            if isinstance(r["latency_ms_one_frame_out_of_order"], float)
                                                                            else r["latency_ms_one_frame_out_of_order"])}
        if "cpu_baseline" in r:
            cfg_extra["line_frontend"]["cpu_port_frames_per_s"] = round(r["cpu_baseline"]["value"], 1)
    if not args.no_stereo:
        r = bench_stereo(pkg, ctx, stream, rank, world, args.steps, args.warmup, args.stereo_batch, args.seed,
                         world == 1 and not args.no_cpu_baseline)
        detail["stereo_frontend"] = r
        cfg_extra["stereo_frontend"] = {"stereo_frames_per_s": round(r["value"], 1),
                                        "mean_left_keylines": round(r["config"]["mean_left_keylines"], 1),
                                        "mean_left_keypoints": round(r["config"]["mean_left_keypoints"], 1),
                                        "mean_stereo_matches": round(r["config"]["mean_stereo_matches"], 1),
                                        "stereo_frames_per_step_per_gpu": args.stereo_batch,
                                        "e2e_stereo_frames_per_s": round(r["e2e"]["value"], 1)}
        if r.get("cpu_baseline"):
            cfg_extra["stereo_frontend"]["cpu_port_stereo_frames_per_s"] = round(r["cpu_baseline"]["value"], 1)
    if rank == 0 and world == 1 and not args.no_mapping:
        try:
            detail["mapping_matchers"] = bench_mapping(pkg, ctx, not args.no_cpu_baseline)
        except Exception as e:
            detail["mapping_matchers"] = {"error": f"{type(e).__name__}: {e}"}

    if rank == 0:
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms_max / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "u8/f64", "data": "synthetic",
            "config": {"workload": WORKLOAD, "frames_per_step_per_gpu": B, "image": f"{COLS}x{ROWS}",
                       "orb": {"max_num_keypts": 1000, "scale_factor": 1.2, "num_levels": 8, "ini_fast_thr": 20, "min_fast_thr": 7},
                       "parallelism": f"frames sharded over {world} GPU(s), no data-path collective",
                       "streams_per_gpu": S * (2 if args.track_streams else 1), "frames_per_stream_per_step": Bs,
                       "l2": "inputs larger than L2 (batch x 307 KB images)",
                       "tracked_ok_frames": ok, "tracked_ok_frames_e2e": e2e_ok, "mean_keypoints_e2e": round(e2e_kp / max(B, 1), 1),
                       **cfg_extra},
            "clocks": clk.summary(),
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": int(h2d_bytes), "d2h_bytes_per_step": int(d2h_bytes),
                    "what": "pinned H2D of images + last-frame landmarks/descriptors/poses; D2H of keypoints, descriptors, "
                            "match indices, poses, counts (full-capacity arrays), every step"},
            "gpu_launches": int(launches),
            "roofline": roofline,
        }
        if world == 1 and not args.no_cpu_baseline:
            hw = host_cpu_info()
            cores = hw["logical"]
            n_sample = int(min(Bs, max(32, 4 * cores)))
            fps_mt, dt_mt, _ = cpu_port_frames(frames_l[0], aux, list(range(n_sample)), cores)
            fps_mt2, dt_mt2, _ = cpu_port_frames(frames_l[0], aux, list(range(n_sample)), cores)
            fps_1, dt_1, _ = cpu_port_frames(frames_l[0], aux, list(range(min(8, n_sample))), 1)
            line["cpu_baseline"] = {"value": max(fps_mt, fps_mt2), "unit": UNIT, "cores": cores, "kind": "port",
                                    "sample": f"{n_sample} frames of the same workload over {cores} native pinned host threads, "
                                              f"best of two runs ({dt_mt:.2f} s, {dt_mt2:.2f} s)",
                                    "single_thread_value": fps_1, "cpu_model": hw["model"], "physical_cores": hw["physical"],
                                    "repeat_values": [round(fps_mt, 1), round(fps_mt2, 1)]}
        detail["headline"] = dict(line)
        if args.detail:
            dpath = Path(args.detail)
            try:
                dpath.parent.mkdir(parents=True, exist_ok=True)
                dpath.write_text(json.dumps(detail, indent=1))
                line["detail_file"] = str(dpath)
            except OSError as e:
                line["detail_file"] = f"unwritable: {e}"
        sys.stderr.write("[bench detail] " + json.dumps(_round_floats(detail, 5)) + "\n")
        print(json.dumps(_round_floats(line, 7)))
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
