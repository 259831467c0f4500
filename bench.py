#!/usr/bin/env python
"""bench.py -- frames/s of the 1-point-RANSAC EKF measurement-update path (BASELINE.json metric) on B200.

--gpus 1 (the headline): workload C3 = ONE synthetic 2000-feature inverse-depth map (state dimension 12013, P = 1.15 GB fp64 resident in
  HBM), 1280x960 camera, bounded trajectory; one step = one frame through the whole path (Map::map_management's flag reset +
  ekf_prediction + search_IC_matches incl. the patch warp + ransac_hypotheses + ekf_update_li_inliers + rescue_hi_inliers +
  ekf_update_hi_inliers) via the C ABI (include/rslam.h).
--gpus N > 1: a single filter's update stays on one GPU (north_star), so the headline is the PARTITIONED configuration C5 = 4096
  independent 100-feature filters split over the ranks with no inter-GPU traffic; the sharded hypothesis sweep C4 (NCCL inside the
  library) is reported under "workloads".
  value : frames/s with all inputs (images, uniforms) already resident in HBM, CUDA events on the library's stream
  e2e   : frames/s through the same C-ABI call with HOST (pinned) images/uniforms copied in and the pose copied out every frame
  roofline, cpu_baseline : see DESIGN.md section "Measurement"
`--impl reference` times the reference's OWN sources (oracle/_ref/libref.so) on the host cores on the same workload: whole frames
where they finish in seconds (C5's 100-feature filters), bounded per-stage samples of a frame with the extrapolation stated where one
frame takes hours (C3).
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

from ransac_slam_b200 import synth  # noqa: E402

UNIT = "frames/s"
METRIC_C3 = "frames/s (EKF+1-pt RANSAC) at N=2000 features"
METRIC_C5 = "frames/s (EKF+1-pt RANSAC) at N=100 features, 4096 independent filters (aggregate filter-frames/s)"
C3_N, C3_NU01, C3_SCALE = 2000, 16384, 0.25
C5_FILTERS = int(os.environ.get("RSLAM_C5_FILTERS", "4096"))


def config_for(world):
    """the workload description BOTH arms print (the driver compares it)"""
    if world == 1:
        return dict(workload="C3: synthetic 2000-feature inverse-depth map (state dim 12013, P 1.15 GB fp64), 1280x960 camera (4x pixel density, "
                             "motion and noise scaled 1/4), bounded trajectory, 1-pt RANSAC + li/hi EKF update, patch warp (pred_patch_fc) included",
                    features=C3_N, state_dim=13 + 6 * C3_N, n_u01=C3_NU01, quirks="reference (Q1,Q4,Q6 on)",
                    l2="working set (P 1.15 GB) exceeds L2; nothing to flush", per_gpu="single filter")
    return dict(workload=f"C5: {C5_FILTERS} independent synthetic 100-feature filters (320x240 camera, bounded trajectory, 1-pt RANSAC + li/hi EKF "
                         "update, patch warp included), split over the ranks, no inter-GPU traffic",
                features=100, state_dim=613, filters=C5_FILTERS, n_u01=1000, quirks="reference (Q1,Q4,Q6 on)",
                l2="working set (P 3 MB x filters) exceeds L2; nothing to flush", per_gpu=f"{C5_FILTERS} / n_gpus filters")


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return dict(hbm_gbs=float(d.get("hbm_gbs", 6650.0)), source="measured (MEASURED_PEAKS.json)")
    return dict(hbm_gbs=6650.0, source="fallback (B200_PROFILING.md)")


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)."""

    def __init__(self, index=0):
        self.index = index
        self.proc = None
        self.lines = []

    def start(self):
        q = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), f"--query-gpu={q}", "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if self.proc is None:
            return dict(sm_mhz=None, sm_max_mhz=None, reasons=["nvidia-smi unavailable"])
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            pass
        sm, mx, reasons = [], [], set()
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 8:
                continue
            try:
                sm.append(float(f[0]))
                mx.append(float(f[1]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[4:8]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return dict(sm_mhz=float(np.median(sm)) if sm else None, sm_max_mhz=float(max(mx)) if mx else None, reasons=sorted(reasons),
                    samples=len(sm))


def dist_setup(n_gpus):
    import torch

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world > 1:
        import torch.distributed as dist

        torch.cuda.set_device(local)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    else:
        torch.cuda.set_device(0)
    return world, rank, local


def barrier(world):
    import torch

    torch.cuda.synchronize()
    if world > 1:
        import torch.distributed as dist

        dist.barrier()
    torch.cuda.synchronize()


def max_over_ranks(x, world):
    import torch

    if world == 1:
        return x
    import torch.distributed as dist

    t = torch.tensor([x], dtype=torch.float64, device="cuda")
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return float(t.item())


def sum_over_ranks(x, world):
    import torch

    if world == 1:
        return x
    import torch.distributed as dist

    t = torch.tensor([x], dtype=torch.float64, device="cuda")
    dist.all_reduce(t, op=dist.ReduceOp.SUM)
    return float(t.item())


# ---------------------------------------------------------------------------------------------------------------------
# algorithmic work per kernel and frame (SURVEY.md 8d; DESIGN.md "Kernels"): bytes for the HBM-bound kernels, flops for the fp64
# tensor-core kernels -- each amount belongs to the kernel that executes it
# ---------------------------------------------------------------------------------------------------------------------
def kernel_work(kernel, launches, N, n, st):
    """returns (bound, amount per frame) or (None, None) for latency-only kernels"""
    nic, mid = st["nic"], st["mid"]
    ks = [2.0 * st["m_li"], 2.0 * st["m_hi"]]
    if kernel == "k_predict":  # launched for search_IC_matches and again for rescue_hi_inliers
        return "hbm", launches * (1310.0 * N + 1460.0)
    if kernel == "k_pred_patch":
        return "hbm", launches * N * (41 * 41 + 14 * 8 + 169 * 4.0)
    if kernel == "k_search":
        return "hbm", launches * N * ((2 * 3 + 13) ** 2 + 169 * 4 + 16.0)
    if kernel == "k_ransac_support":
        return "hbm", 288.0 * nic * mid
    if kernel == "k_upd_W":
        return "hbm", sum(8.0 * n * (7 + 3 * k) + 8.0 * n * k for k in ks if k > 0)
    if kernel == "k_ekf_prediction":
        return "hbm", 2 * 13 * n * 8.0 * 2
    if kernel == "k_upd_jnorm":
        return "hbm", launches * 2 * 4 * n * 8.0 * 2
    if kernel == "k_gemm_dmma/syrk_P" or kernel == "k_syrk_rows":
        return "tensor", sum(float(n + 1) * (n + 1) * k for k in ks)  # lower triangle x 2 flop
    if kernel == "k_trsm_small":
        return "tensor", sum(float(n + 1) * k * k for k in ks)
    # large k: two-level TRSM -- the left-looking kernel solves inside 1024-wide outer blocks, K = 1024 GEMMs carry the rest
    if kernel == "k_trsm_ll":
        return "tensor", sum(float(n + 1) * min(1024.0 * k, k * k) for k in ks)
    if kernel == "k_gemm_dmma/trsm_outer":
        return "tensor", sum(float(n + 1) * max(k * k - 1024.0 * k, 0.0) for k in ks)
    if kernel == "cholesky":  # k_chol_panel + k_gemm_dmma/chol_outer + k_chol_trinv (or the single-CTA k_chol_small)
        return "tensor", sum(k**3 / 3.0 for k in ks)
    return None, None


CHOL_KERNELS = ("k_chol_panel", "k_gemm_dmma/chol_outer", "k_chol_trinv", "k_chol_small")
TRSM_KERNELS = ("k_trsm_ll", "k_gemm_dmma/trsm_outer")

# DRAM bytes (read + write) per launch of the dominant kernels from this round's `ncu --set full` captures:
#   profiles/r02_syrk_c3.md      k_gemm_dmma/syrk_P at N = 2000, k = 3608: 8.54 GB read + 1.15 GB written
#   profiles/r02_c5_kernels.md   k_syrk_rows at 1024 filters, k = 186: 2.83 GB read + 3.05 GB written (scaled to the filters of the launch)
NCU_TRAFFIC = {"k_gemm_dmma/syrk_P": 9.70e9, "k_syrk_rows": 5.88e9 / 1024.0}


def roofline_table(prof, frames, N, n, st, fp64_peak):
    """per-kernel CUDA-event times of the instrumented pass -> shares and roofline fractions"""
    pk = peaks()
    tot = sum(v[1] for v in prof.values())
    rows = {}
    chol = [0, 0.0]
    trsm = [0, 0.0]
    for name, (cnt, ms) in sorted(prof.items(), key=lambda kv: -kv[1][1]):
        row = dict(launches_per_frame=cnt / frames, ms_per_frame=ms / frames, share=ms / tot)
        if name in CHOL_KERNELS:
            chol[0] += cnt
            chol[1] += ms
        if name in TRSM_KERNELS:
            trsm[0] += cnt
            trsm[1] += ms
        bound, amount = kernel_work(name, cnt / frames, N, n, st)
        if bound == "hbm" and ms > 0:
            ach = amount / (ms / frames * 1e-3) / 1e9
            row.update(bound="hbm", unit="GB/s", achieved=ach, peak=pk["hbm_gbs"], frac=ach / pk["hbm_gbs"])
        elif bound == "tensor" and ms > 0:
            ach = amount / (ms / frames * 1e-3) / 1e12
            row.update(bound="tensor", unit="TFLOP/s", achieved=ach, peak=fp64_peak, frac=ach / fp64_peak)
        rows[name] = row
    if chol[1] > 0:
        _, amount = kernel_work("cholesky", 0, N, n, st)
        ach = amount / (chol[1] / frames * 1e-3) / 1e12
        rows["cholesky (all of its kernels)"] = dict(launches_per_frame=chol[0] / frames, ms_per_frame=chol[1] / frames, share=chol[1] / tot, bound="tensor",
                                                     unit="TFLOP/s", achieved=ach, peak=fp64_peak, frac=ach / fp64_peak)
    if trsm[1] > 0 and len([k for k in prof if k in TRSM_KERNELS]) > 1:
        amount = sum(float(n + 1) * (2.0 * m) ** 2 for m in (st["m_li"], st["m_hi"]))
        ach = amount / (trsm[1] / frames * 1e-3) / 1e12
        rows["triangular solve (all of its kernels)"] = dict(launches_per_frame=trsm[0] / frames, ms_per_frame=trsm[1] / frames, share=trsm[1] / tot, bound="tensor",
                                                             unit="TFLOP/s", achieved=ach, peak=fp64_peak, frac=ach / fp64_peak)
    return rows


# ---------------------------------------------------------------------------------------------------------------------
# workloads
# ---------------------------------------------------------------------------------------------------------------------
def make_c2(seed, frames, n_u01=1000):
    """a 100-feature filter of C2 / C5: grid-placed smooth-texture features so that the warped predicted patches still match"""
    scene = synth.make_scene(N=100, seed=seed, margin=30, min_sep=18, texture="smooth")
    seq = synth.make_sequence(scene, T=frames, seed=seed + 1, n_u01=n_u01, u01_seed=42 + seed)
    return scene, seq


def make_c3(frames):
    cam = synth.scaled_camera(4)
    scene = synth.make_scene(N=C3_N, seed=1234, cam=cam, margin=30, min_sep=18, assemble_P=False, motion_scale=C3_SCALE, texture="smooth")
    seq = synth.make_sequence(scene, T=frames, seed=1235, n_u01=C3_NU01)
    return cam, scene, seq


def upload_appearance(g, scene, b=0):
    """what Map::initialize_a_features stores per feature (src/Map.cpp:286-294); the predicted patch is warped from it on the device"""
    N = scene.N
    g.upload_feature_init(scene.init_patches, np.tile(scene.x0[:3], (N, 1)), np.tile(np.eye(3).reshape(1, 9), (N, 1)), scene.uv0, b=b)


def new_gpu_filter(scene, batch=1, device=0, quirks=0x7, x=None, P=None, max_features=None):
    from ransac_slam_b200 import capi

    g = capi.Filter(scene.cam.as9(), max_features or scene.N, batch=batch, device=device, quirks=quirks, std_z=scene.std_z)
    for b in range(batch):
        g.upload_state(scene.x0 if x is None else x, scene.P0 if P is None else P, b=b)
        if scene.init_patches is not None:
            upload_appearance(g, scene, b=b)
        else:
            g.upload_patches(scene.templates.astype(np.float64), b=b)
    if scene.init_patches is not None:
        g.set_patch_warp(True)
    return g


def new_c3_filter(cam, scene, P0_dev, device):
    import torch

    from ransac_slam_b200 import capi

    n = scene.x0.size
    g = capi.Filter(cam.as9(), C3_N, batch=1, device=device, std_a=0.007 * C3_SCALE, std_alpha=0.007 * C3_SCALE)
    x0 = torch.from_numpy(scene.x0).to(P0_dev.device)
    g.upload_state_device(x0.data_ptr(), P0_dev.data_ptr(), n, n, C3_N)
    upload_appearance(g, scene)
    g.set_patch_warp(True)
    return g


def run_frames_resident(g, d_images, d_u01, frames, l2_flush, flush_buf, stream):
    """times `frames` (list of frame indices) with CUDA events on the library's stream; returns total ms"""
    import torch

    T, rows, cols = d_images.shape[0], d_images.shape[-2], d_images.shape[-1]
    n_u01 = d_u01.shape[-1]
    img_bytes = rows * cols * (d_images.shape[1] if d_images.dim() == 4 else 1)
    u_bytes = n_u01 * 8 * (d_u01.shape[1] if d_u01.dim() == 3 else 1)
    if l2_flush:
        evs = []
        for k in frames:
            with torch.cuda.stream(stream):
                flush_buf.zero_()
            e0 = torch.cuda.Event(enable_timing=True)
            e1 = torch.cuda.Event(enable_timing=True)
            e0.record(stream)
            g.frame((d_images.data_ptr() + k * img_bytes, rows, cols, cols), (d_u01.data_ptr() + k * u_bytes, n_u01), predict=True)
            e1.record(stream)
            evs.append((e0, e1))
        g.sync()
        return sum(a.elapsed_time(b) for a, b in evs)
    e0 = torch.cuda.Event(enable_timing=True)
    e1 = torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    for k in frames:
        g.frame((d_images.data_ptr() + k * img_bytes, rows, cols, cols), (d_u01.data_ptr() + k * u_bytes, n_u01), predict=True)
    e1.record(stream)
    g.sync()
    return e0.elapsed_time(e1)


def fp64_gemm_peak():
    """cuBLAS fp64 GEMM throughput measured live (MEASURED_PEAKS.json has no fp64 figure); measurement probe only."""
    import torch

    n = 6144
    a = torch.randn(n, n, dtype=torch.float64, device="cuda")
    b = torch.randn(n, n, dtype=torch.float64, device="cuda")
    for _ in range(2):
        a @ b
    torch.cuda.synchronize()
    best = 0.0
    for _ in range(4):
        e0 = torch.cuda.Event(enable_timing=True)
        e1 = torch.cuda.Event(enable_timing=True)
        e0.record()
        a @ b
        e1.record()
        torch.cuda.synchronize()
        best = max(best, 2.0 * n**3 / (e0.elapsed_time(e1) * 1e-3) / 1e12)
    return best


P_SAMPLE, DUMP_SEED = 1 << 20, 2024


def filter_outputs(g, b=0, prefix=""):
    """what a caller of rslam_frame receives for filter b after a frame: the state x, the covariance P, the per-feature predictions,
    matches and inlier flags, and the RANSAC result.  A P of more than 2^20 entries (1.15 GB at C3) is given by its diagonal, its 13
    camera rows and a fixed sample of 2^20 entries drawn with DUMP_SEED (flat column-major indices in P_sample_index)."""
    x, P = g.download_state(b=b)
    n = x.size
    out = dict(x=x)
    if n * n <= P_SAMPLE:
        out["P"] = P
    else:
        flat = np.random.default_rng(DUMP_SEED).integers(0, n * n, P_SAMPLE)
        out.update(P_diag=np.diag(P).copy(), P_camera_rows=np.ascontiguousarray(P[:13]), P_sample=P.reshape(-1, order="F")[flat],
                   P_sample_index=flat.astype(np.float64))
    ft = g.features(b)
    out.update(h=ft["h"], S=ft["S"], z=ft["z"])
    for k in ("has_h", "ic", "li", "hi", "times_predicted", "times_measured"):
        out[k] = ft[k].astype(np.float32)
    r = g.ransac_result(b)
    out["ransac"] = np.array([r[k] for k in ("status", "hyp_run", "best_support", "n_hyp", "num_ic", "winner")], dtype=np.float64)
    return {prefix + k: v for k, v in out.items()}


def dump_outputs(directory, arrays):
    """arrays: name -> float32 / float64 array, written as directory/<name>.npy"""
    total = sum(a.nbytes for a in arrays.values())
    assert total <= 64 << 20, f"{total} bytes of outputs, more than 64 MB"
    os.makedirs(directory, exist_ok=True)
    for name, a in arrays.items():
        assert a.dtype in (np.float32, np.float64), (name, a.dtype)
        np.save(os.path.join(directory, name + ".npy"), a)


def frame_stats(g, b=0):
    ft = g.features(b)
    r = g.ransac_result(b)
    return dict(n_vis=int(ft["has_h"].sum()), nic=int(ft["ic"].sum()), mid=int(ft["ic"].sum()), m_li=int(ft["li"].sum()), m_hi=int(ft["hi"].sum()),
                hyp_run=r["hyp_run"], ransac_status=r["status"])


def cpu_model():
    try:
        for ln in open("/proc/cpuinfo"):
            if ln.startswith("model name"):
                return ln.split(":", 1)[1].strip()
    except Exception:
        pass
    return "unknown"


# ---------------------------------------------------------------------------------------------------------------------
# CPU legs: the reference's OWN sources (oracle/_ref/libref.so = /root/reference/src/{ExtendKF,Tracking,Converter,Map}.cpp compiled
# unmodified over the stand-in Eigen / OpenCV headers of oracle/ref_shim/), single threaded like the reference.
# ---------------------------------------------------------------------------------------------------------------------
def _ref_filter_for(cam, std_scale=1.0):
    from oracle import ref_py as R

    r = R.ReferenceFilter(k1=cam.k1, k2=cam.k2, nRows=cam.nRows, nCols=cam.nCols, d=cam.dx, cx_d=cam.Cx * cam.dx, cy_d=cam.Cy * cam.dy, dx=cam.dx, dy=cam.dy,
                          f=cam.f, std_a=0.007 * std_scale, std_alpha=0.007 * std_scale)
    assert np.allclose(r.camera9(), cam.as9(), rtol=1e-15, atol=0), "the reference parsed a different camera"
    return r


def _draws(u01):
    from oracle import ref_py as R

    return np.minimum((u01 * R.RAND_MAX).astype(np.int64), R.RAND_MAX - 1).astype(np.int32)


class RefC2:
    """whole frames of one 100-feature filter through the reference's own TrackRunning call sequence (map frozen: the flag reset of
    Map::map_management step 2 only), on the same images / uniforms as the GPU arm"""

    def __init__(self, scene, seq):
        from oracle import ref_py as R

        R.set_blocked_gemm(1, 1)  # the stand-in Eigen's dense products through the packed kernel (a fairer stand-in for Eigen's GEBP)
        self.scene, self.seq = scene, seq
        self.r = _ref_filter_for(scene.cam)
        for i in range(scene.N):
            self.r.add_feature(0, scene.init_patches[i], None, scene.x0[:3], np.eye(3), scene.uv0[i])
        self.r.set_state(scene.x0, scene.P0)
        self.k = 0

    def step(self):
        """one frame; returns seconds"""
        r, k = self.r, self.k
        r.set_draws(_draws(self.seq.u01[k]))
        t0 = time.perf_counter()
        r.reset_flags()
        r.ekf_prediction()
        r.search_ic_matches(self.seq.images[k])
        r.ransac_hypotheses()
        r.update_li()
        r.rescue_hi()
        r.update_hi()
        dt = time.perf_counter() - t0
        self.k += 1
        return dt

    def stats(self):
        f = self.r.features()
        return dict(nic=int(f["ic"].sum()), m_li=int(f["li"].sum()), m_hi=int(f["hi"].sum()))


class RefC3Sampler:
    """Bounded samples of ONE reference frame at N = 2000 (a whole frame takes the reference hours: ~9000 dense hypotheses of two passes
    over the 1.15 GB covariance each, 2000 dense H_i P H_i^T, a joint update of 6 n^2 k + 6 n k^2 + 2 k^3 flop).  Every stage is timed
    through the reference's own methods on the full-size state, on a sub-sample of its units, and scaled by the unit count of the
    frame (SURVEY 8d "per-stage sub-sampling with the extrapolation stated"):
      prediction, measurement prediction, Jacobians : whole, as is
      S_i = H_i P H_i^T + R_i (src/Tracking.cpp:39-44) : n_S features, x (predicted features)      [also for rescue_hi_inliers :589]
      patch warp + ZNCC matching : the reference's search_IC_matches on a 16-feature filter, per feature x (predicted features)
      ransac_hypotheses : the reference's loop left after n_hyp hypotheses, per hypothesis x hyp_run
      update : ExtendKF::update at 2 measurement rows measures the size-independent part (by-value copies of P, symmetrisation, Jnorm);
               the dense products of the real k are added at the product rate of the stand-in Eigen measured in the same run:
               (6 n^2 k + 6 n k^2 + 2 k^3) / rate.  NOT included (so the estimate is a lower bound of the reference's time): the
               O(m^2 n) re-allocation of the stacked H (src/ExtendKF.cpp:585-589).
    `blocked` selects the stand-in Eigen's dense product: packed AVX2 kernel (a fair stand-in for Eigen's GEBP; the headline) or the
    plain loops the parity vectors were made with (printed beside it)."""

    def __init__(self, cam, scene, seq, P0, stats):
        from oracle import ref_py as R

        self.R = R
        self.cam, self.scene, self.seq, self.stats = cam, scene, seq, stats
        N = scene.N
        self.n = scene.x0.size
        self.full = _ref_filter_for(cam, C3_SCALE)
        for i in range(N):
            self.full.add_feature(0, scene.init_patches[i], None, scene.x0[:3], np.eye(3), scene.uv0[i])
        self.full.set_state(scene.x0, P0)
        ns = 16
        self.small = _ref_filter_for(cam, C3_SCALE)
        for i in range(ns):
            self.small.add_feature(0, scene.init_patches[i], None, scene.x0[:3], np.eye(3), scene.uv0[i])
        m = 13 + 6 * ns
        self.small.set_state(scene.x0[:m], np.asfortranarray(P0[:m, :m]))
        self.ns = ns
        self.fixed = None
        self.cursor = 0

    def measure_fixed(self):
        """once per run: the whole-frame stages that need no sub-sampling, and the size-independent part of ExtendKF::update"""
        R, f = self.R, self.full
        R.set_blocked_gemm(1, 1)
        t = {}
        t0 = time.perf_counter()
        f.reset_flags()
        f.ekf_prediction()
        t["ekf_prediction"] = time.perf_counter() - t0
        t0 = time.perf_counter()
        f.predict_measurements()
        f.calculate_derivatives()
        t["predict_and_jacobians"] = time.perf_counter() - t0
        ft = f.features()
        self.z = np.rint(ft["h"]) + 1.0
        self.ic = ft["has_h"].astype(np.uint8)
        f.set_matches(self.z, self.ic)
        # ExtendKF::ekf_update_li_inliers on ONE inlier (what quirk Q1 leaves at this workload: m_li = 1): measured whole
        N = self.scene.N
        li = np.zeros(N, np.uint8)
        li[int(np.flatnonzero(self.ic)[0])] = 1
        f.set_inlier_flags(li, np.zeros(N, np.uint8))
        t0 = time.perf_counter()
        f.update_li()
        t["update_at_k2"] = time.perf_counter() - t0
        # the small filter: prediction + search (Jacobians, S_i, patch warp, matching) per feature at a state size where the dense
        # products cost nothing
        s = self.small
        s.reset_flags()
        s.ekf_prediction()
        t0 = time.perf_counter()
        s.search_ic_matches(self.seq.images[0])
        t["search_per_feature"] = (time.perf_counter() - t0) / self.ns
        self.fixed = t
        return t

    def sample(self, n_S=2, n_hyp=2):
        """one bounded sample; returns dict with the per-unit times and the extrapolated frame time for both product kernels"""
        R, f, st = self.R, self.full, self.stats
        N, n = self.scene.N, self.n
        R.set_blocked_gemm(1, 1)
        first = (self.cursor * n_S) % (N - n_S)
        t0 = time.perf_counter()
        done = f.S_subset(first, n_S)
        t_S = (time.perf_counter() - t0) / max(done, 1)
        f.set_draws(_draws(self.seq.u01[0])[(self.cursor * n_hyp) % 8192:])
        t0 = time.perf_counter()
        hyps = f.ransac_limited(n_hyp)
        t_hyp = (time.perf_counter() - t0) / max(hyps, 1)
        self.cursor += 1
        rate = {}
        for name, on in (("blocked", 1), ("plain", 0)):
            R.set_blocked_gemm(on, 1)
            mm, nn, kk = 384, 1536, 1536
            rate[name] = 2.0 * mm * nn * kk / R.gemm_seconds(mm, nn, kk)
        R.set_blocked_gemm(1, 1)
        fx = self.fixed
        k_li, k_hi = 2.0 * st["m_li"], 2.0 * st["m_hi"]

        def upd(k, r):
            if k <= 0:
                return 0.0
            return fx["update_at_k2"] + (6.0 * n * n * k + 6.0 * n * k * k + 2.0 * k**3) / r

        out = dict(t_S_per_feature=t_S, t_per_hypothesis=t_hyp, gemm_gflops=dict(blocked=rate["blocked"] / 1e9, plain=rate["plain"] / 1e9))
        for name in ("blocked", "plain"):
            r = rate[name]
            resc = max(st["nic"] - st["m_li"], 0)
            T = (fx["ekf_prediction"] + fx["predict_and_jacobians"] + st["n_vis"] * t_S + st["n_vis"] * fx["search_per_feature"] + st["hyp_run"] * t_hyp
                 + (fx["update_at_k2"] if k_li <= 4 else upd(k_li, r)) + fx["predict_and_jacobians"] + resc * t_S + upd(k_hi, r))
            out["frame_seconds_" + name] = T
        out["breakdown_seconds_blocked"] = dict(prediction=fx["ekf_prediction"], predict_jacobians=2 * fx["predict_and_jacobians"], S_i=st["n_vis"] * t_S,
                                                patch_warp_and_matching=st["n_vis"] * fx["search_per_feature"], ransac=st["hyp_run"] * t_hyp,
                                                rescue_S_i=max(st["nic"] - st["m_li"], 0) * t_S,
                                                updates=(fx["update_at_k2"] if k_li <= 4 else upd(k_li, rate["blocked"])) + upd(k_hi, rate["blocked"]))
        return out

    def describe(self, n_S, n_hyp):
        st = self.stats
        return (f"per-stage samples of one reference frame at N=2000 (n=12013) through the reference's own methods on the full-size state: {n_S} of "
                f"{st['n_vis']} S_i = H_i P H_i^T, {n_hyp} of {st['hyp_run']} RANSAC hypotheses, prediction / measurement prediction / Jacobians whole, patch "
                f"warp + matching on a 16-feature filter, ExtendKF::update whole at k=2 plus (6n^2k+6nk^2+2k^3)/rate for k_hi={2 * st['m_hi']} at the "
                "dense-product rate of the stand-in Eigen (packed AVX2 kernel) measured in the same run; each sample scaled by its unit count; the O(m^2 n) "
                "re-allocation of the stacked H is left out (lower bound of the reference's time)")


def c3_stats_from_oracle(cam, scene, seq, P0):
    """frame statistics of the C3 workload (predicted / matched features, hypotheses the reference's loop runs, inlier counts) from the CPU
    oracle in sparse mode, all host threads -- set-up of the reference arm, not timed"""
    from oracle import oracle_py as O

    O.set_threads(os.cpu_count() or 1)
    o = O.OracleFilter(cam.as9(), std_a=0.007 * C3_SCALE, std_alpha=0.007 * C3_SCALE, std_z=scene.std_z, quirks=O.Q_ALL, sparse=True, fast_corr=True, warp_patches=True)
    for i in range(scene.N):
        o.add_feature(0, scene.init_patches[i], None, scene.x0[:3], np.eye(3), scene.uv0[i])
    o.set_state(scene.x0, P0)
    o.map_reset_flags()
    o.ekf_prediction()
    o.search_ic_matches(seq.images[0])
    rc, info = o.ransac_hypotheses(seq.u01[0])
    o.update_li()
    o.rescue_hi()
    f = o.features()
    return dict(n_vis=int(f["has_h"].sum()), nic=int(f["ic"].sum()), mid=int(f["ic"].sum()), m_li=int(f["li"].sum()), m_hi=int(f["hi"].sum()),
                hyp_run=int(info["hyp_run"]), ransac_status=int(rc))


# ---------------------------------------------------------------------------------------------------------------------
# --gpus 1: C3, one 2000-feature filter
# ---------------------------------------------------------------------------------------------------------------------
def bench_c3(args, world, rank, local):
    import torch

    K, W = args.steps, args.warmup
    PF = 2  # extra frames for the instrumented pass
    T = W + K + PF
    cam, scene, seq = make_c3(T)
    N, n = scene.N, scene.x0.size
    rows, cols = seq.images.shape[1:]
    dev = torch.device("cuda", local)
    P0 = synth.assemble_P_torch(scene, dev)
    # ---- device-resident throughput ------------------------------------------------------------------------------
    g = new_c3_filter(cam, scene, P0, local)
    stream = torch.cuda.ExternalStream(g.stream)
    d_images = torch.from_numpy(seq.images).to(dev)
    d_u01 = torch.from_numpy(seq.u01).to(dev)
    run_frames_resident(g, d_images, d_u01, range(W), False, None, stream)
    barrier(world)
    sampler = ClockSampler(local)
    sampler.start()
    l0 = g.launches
    ms = run_frames_resident(g, d_images, d_u01, range(W, W + K), False, None, stream)
    launches = g.launches - l0
    barrier(world)
    clocks = sampler.stop()
    value = K / (ms * 1e-3)
    pose_resident = g.download_pose()
    st_last = frame_stats(g)
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, filter_outputs(g))
    # ---- per-kernel breakdown: instrumented pass (CUDA events around every launch on the launching stream, no graph) on the next frames
    g.profile(True)
    stats = []
    for k in range(W + K, T):
        run_frames_resident(g, d_images, d_u01, [k], False, None, stream)
        stats.append(frame_stats(g))
    prof = g.profile_read()
    g.profile(False)
    g.close()
    st = {k: float(np.mean([s_[k] for s_ in stats])) for k in stats[0]}
    fp64_peak = fp64_gemm_peak()
    kernels = roofline_table(prof, PF, N, n, st, fp64_peak)
    top = next(k for k in kernels if "(all of its kernels)" not in k)
    roof = dict(kernel=top, **{k: v for k, v in kernels[top].items()})
    roof["traffic"] = NCU_TRAFFIC.get(top)
    roof["algorithmic_bytes"] = 2.0 * 8.0 * n * (n + 1) / 2 + 8.0 * (n + 1) * 2.0 * st["m_hi"]  # P lower triangle read + written, V read once
    roof["note"] = ("dominant kernel of the step, from the instrumented pass; achieved = algorithmic flops of THIS kernel (covariance downdate P -= V V^T, lower "
                    "triangle: (n+1)^2 k per update) / its time; peak = cuBLAS fp64 GEMM measured live (MEASURED_PEAKS.json has no fp64 figure); "
                    "per-kernel fractions for every kernel of the step are under `kernels`")
    # ---- end to end: host (pinned) image + uniforms copied in, pose copied out, every frame ---------------------------------------
    ge = new_c3_filter(cam, scene, P0, local)
    del P0
    h_images = torch.from_numpy(seq.images).pin_memory()
    h_u01 = torch.from_numpy(seq.u01).pin_memory()
    img_b, u_b = rows * cols, seq.u01.shape[1] * 8

    T_e = h_images.shape[0]

    def e2e_in(k):
        k %= T_e
        return (h_images.data_ptr() + k * img_b, rows, cols, cols), (h_u01.data_ptr() + k * u_b, seq.u01.shape[1])

    def e2e_step(k):
        # the step's own inputs were staged by the previous step's prefetch (the first one copies in line); the NEXT step's host->device
        # copy is started before this step's pose is read back, so it runs beside this step's kernels: one copy per step either way
        ge.frame(*e2e_in(k), predict=True)
        ge.prefetch(*e2e_in(k + 1))
        return ge.download_pose()

    for k in range(W):
        e2e_step(k)
    barrier(world)
    t0 = time.perf_counter()
    for k in range(W, W + K):
        pose = e2e_step(k)
    ge.sync()
    t_e2e = time.perf_counter() - t0
    e2e = dict(value=K / t_e2e, unit=UNIT, h2d_bytes_per_step=img_b + u_b, d2h_bytes_per_step=13 * 8)
    assert np.allclose(pose, pose_resident, rtol=1e-9, atol=1e-12), "resident and end-to-end runs must produce the same trajectory"
    ge.close()
    torch.cuda.empty_cache()
    # ---- CPU baseline: the reference's own sources, bounded per-stage samples of one frame ------------------------------------------
    cpu = None
    if not args.no_cpu:
        try:
            t0 = time.perf_counter()
            P0h = synth.assemble_P_numpy(scene)
            smp = RefC3Sampler(cam, scene, seq, P0h, dict(st_last))
            fixed = smp.measure_fixed()
            one = smp.sample(n_S=4, n_hyp=4)
            cpu = dict(value=1.0 / one["frame_seconds_blocked"], unit=UNIT, cores=1, kind="reference", cpu_model=cpu_model(), host_cores=os.cpu_count(),
                       sample=smp.describe(4, 4) + f"; {time.perf_counter() - t0:.0f} s of CPU work incl. set-up",
                       frame_seconds=one["frame_seconds_blocked"], value_plain_product=1.0 / one["frame_seconds_plain"], frame_stats=st_last,
                       per_unit=dict(fixed, t_S_per_feature=one["t_S_per_feature"], t_per_hypothesis=one["t_per_hypothesis"]),
                       gemm_gflops=one["gemm_gflops"], breakdown_seconds=one["breakdown_seconds_blocked"])
            del smp, P0h
        except Exception as e:  # the baseline must never cost the main line
            cpu = dict(value=None, unit=UNIT, cores=1, kind="reference", error=repr(e))
    line = dict(metric=METRIC_C3, value=value, unit=UNIT, n_gpus=1, steps=K, warmup=W, ms_per_step=ms / K, higher_is_better=True, scaling="weak",
                vs_baseline=None, dtype="f64", data="synthetic", config=config_for(1), e2e=e2e, gpu_launches=int(launches), clocks=clocks, roofline=roof,
                cpu_baseline=cpu, kernels=kernels, frame_stats=st, fp64_gemm_peak_tflops=fp64_peak)
    return line


# ---------------------------------------------------------------------------------------------------------------------
# --gpus N > 1 (and a "workloads" entry at N = 1): C5, independent 100-feature filters split over the ranks, no collective
# ---------------------------------------------------------------------------------------------------------------------
def bench_c5(args, world, rank, local, filters_total=None, steps=None, warmup=None, with_e2e=True, ranks_active=None, dump_dir=None):
    """ranks_active: run on the first `ranks_active` ranks only (the others idle): the same-run single-GPU figure of the scaling line.
    dump_dir: rank 0 writes the outputs of 8 of its filters, evenly spaced over its batch, after the last timed step"""
    import torch

    from ransac_slam_b200 import capi

    Btot = filters_total or C5_FILTERS
    active = ranks_active or world
    K = steps if steps is not None else args.steps
    W = warmup if warmup is not None else args.warmup
    if rank >= active:
        return None
    Bl = (rank + 1) * Btot // active - rank * Btot // active
    NS = 8  # distinct scenes cycled over the batch
    T = W + K + 1
    scenes, seqs = [], []
    for s_ in range(NS):
        sc, sq = make_c2(1234 + s_ + NS * rank, T)
        scenes.append(sc)
        seqs.append(sq)
    cam = scenes[0].cam
    dev = torch.device("cuda", local)
    n = scenes[0].x0.size
    rows, cols = seqs[0].images.shape[1:]
    idx = torch.arange(Bl, device=dev) % NS
    imgs = torch.stack([torch.from_numpy(sq.images) for sq in seqs])  # NS x T x r x c
    u01s = torch.stack([torch.from_numpy(sq.u01) for sq in seqs])

    def new_batch():
        g = capi.Filter(cam.as9(), 100, batch=Bl, device=local)
        for s_ in range(NS):
            xd = torch.from_numpy(scenes[s_].x0).to(dev)
            Pd = torch.from_numpy(np.ascontiguousarray(scenes[s_].P0)).to(dev)
            for b in range(s_, Bl, NS):
                g.upload_state_device(xd.data_ptr(), Pd.data_ptr(), n, n, 100, b=b)
                upload_appearance(g, scenes[s_], b=b)
        g.set_patch_warp(True)
        return g

    g = new_batch()
    d_images = imgs.to(dev)[idx].transpose(0, 1).contiguous()  # T x Bl x r x c
    d_u01 = u01s.to(dev)[idx].transpose(0, 1).contiguous()  # T x Bl x n_u01
    stream = torch.cuda.ExternalStream(g.stream)
    run_frames_resident(g, d_images, d_u01, range(W), False, None, stream)
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    l0 = g.launches
    ms = run_frames_resident(g, d_images, d_u01, range(W, W + K), False, None, stream)
    launches = g.launches - l0
    clocks = sampler.stop() if rank == 0 else None
    pose_resident = g.download_pose(b=Bl - 1)
    if dump_dir and rank == 0:
        arrays = {}
        for b in np.unique(np.linspace(0, Bl - 1, 8).astype(int)):
            arrays.update(filter_outputs(g, b=int(b), prefix=f"filter{b}_"))
        dump_outputs(dump_dir, arrays)
    # instrumented pass (events around every launch, no graph): where the batch frame goes
    g.profile(True)
    run_frames_resident(g, d_images, d_u01, [W + K], False, None, stream)
    prof = g.profile_read()
    g.profile(False)
    ft = [g.features(b=b) for b in range(0, Bl, max(1, Bl // 16))]
    st = dict(n_vis=float(np.mean([f["has_h"].sum() for f in ft])), nic=float(np.mean([f["ic"].sum() for f in ft])), mid=float(np.mean([f["ic"].sum() for f in ft])),
              m_li=float(np.mean([f["li"].sum() for f in ft])), m_hi=float(np.mean([f["hi"].sum() for f in ft])))
    g.close()
    del d_images
    torch.cuda.empty_cache()
    fp64_peak = fp64_gemm_peak()
    # per-kernel work scales with the filters of this rank
    stB = dict(st)
    kernels = roofline_table(prof, 1, 100, n, stB, fp64_peak)
    for row in kernels.values():  # amounts above are per filter: scale to the batch
        if "achieved" in row:
            row["achieved"] *= Bl
            row["frac"] *= Bl
    top = next(k for k in kernels if "(all of its kernels)" not in k)
    roof = dict(kernel=top, **kernels[top])
    roof["traffic"] = NCU_TRAFFIC[top] * Bl if top == "k_syrk_rows" else NCU_TRAFFIC.get(top)
    # whole batch frame against HBM: every filter's P is read and written once per non-empty update, + the P columns W = P H^T gathers
    ldp = (n + 15) // 16 * 16
    upd = (1 if st["m_li"] > 0 else 0) + (1 if st["m_hi"] > 0 else 0)
    bytes_per_filter = upd * 2.0 * n * ldp * 8 + 8.0 * n * (7 * upd + 6 * (st["m_li"] + st["m_hi"]))
    pk = peaks()
    ach = Bl * bytes_per_filter / (ms / K * 1e-3) / 1e9
    out = dict(ms=ms, steps=K, warmup=W, filters_per_gpu=Bl, launches=int(launches), clocks=clocks, frame_stats=st, kernels=kernels, roofline=roof,
               whole_frame_hbm=dict(bound="hbm", unit="GB/s", achieved=ach, peak=pk["hbm_gbs"], frac=ach / pk["hbm_gbs"], bytes_per_filter_frame=bytes_per_filter),
               fp64_gemm_peak_tflops=fp64_peak)
    if with_e2e:
        # end to end: every filter's own host image + uniforms copied in, one pose copied out, every step; bounded number of steps (pinned
        # host memory: rows x cols x filters per step)
        Ke = min(K, 6)
        We = min(W, 2)
        ge = new_batch()
        ih = idx.cpu()
        h_images = imgs[:, :We + Ke][ih].transpose(0, 1).contiguous().pin_memory()  # T x Bl x r x c
        h_u01 = u01s[:, :We + Ke][ih].transpose(0, 1).contiguous().pin_memory()
        img_b, u_b = rows * cols * Bl, seqs[0].u01.shape[1] * 8 * Bl

        def e2e_in(k):
            k %= We + Ke
            return (h_images.data_ptr() + k * img_b, rows, cols, cols), (h_u01.data_ptr() + k * u_b, seqs[0].u01.shape[1])

        def e2e_step(k):
            ge.frame(*e2e_in(k), predict=True)
            ge.prefetch(*e2e_in(k + 1))  # next step's host->device copy beside this step's kernels (one copy per step)
            return ge.download_pose(b=Bl - 1)

        for k in range(We):
            e2e_step(k)
        if ranks_active is None:
            barrier(world)
        t0 = time.perf_counter()
        for k in range(We, We + Ke):
            e2e_step(k)
        ge.sync()
        out["e2e_seconds"] = time.perf_counter() - t0
        out["e2e_steps"] = Ke
        out["e2e_bytes"] = (img_b + u_b, 13 * 8)
        ge.close()
        del h_images
    out["pose_check"] = float(np.abs(pose_resident).sum())
    return out


def c5_line(args, world, rank, local):
    """the headline of --gpus N > 1"""
    import torch

    # same-run single-GPU figure first (rank 0 alone, all filters): what the N-GPU value scales from
    single = bench_c5(args, world, rank, local, steps=min(args.steps, 6), warmup=3, with_e2e=False, ranks_active=1)
    barrier(world)
    torch.cuda.empty_cache()
    r = bench_c5(args, world, rank, local, dump_dir=args.dump_outputs)
    barrier(world)
    ms = max_over_ranks(r["ms"], world)
    K, W = r["steps"], r["warmup"]
    value = C5_FILTERS * K / (ms * 1e-3)
    te = max_over_ranks(r["e2e_seconds"], world)
    h2d = sum_over_ranks(float(r["e2e_bytes"][0]), world)
    e2e = dict(value=C5_FILTERS * r["e2e_steps"] / te, unit=UNIT, h2d_bytes_per_step=int(h2d), d2h_bytes_per_step=13 * 8 * world, steps=r["e2e_steps"],
               note="every filter's own 320x240 image and 1000 uniforms from pinned host memory every step (rslam_prefetch_inputs: step k+1's copy runs beside step k's "
                    "kernels; one pose read back per step); bounded to 6 steps (pinned host memory)")
    launches = int(sum_over_ranks(float(r["launches"]), world))
    if rank != 0:
        return None
    line = dict(metric=METRIC_C5, value=value, unit=UNIT, n_gpus=world, steps=K, warmup=W, ms_per_step=ms / K, higher_is_better=True, scaling="strong",
                vs_baseline=None, dtype="f64", data="synthetic", config=config_for(world), e2e=e2e, gpu_launches=launches, clocks=r["clocks"],
                roofline=dict(r["roofline"], note="dominant kernel of the batch frame on rank 0, instrumented pass; per-kernel fractions under `kernels`"),
                cpu_baseline=None, kernels=r["kernels"], frame_stats=r["frame_stats"], whole_frame_hbm=r["whole_frame_hbm"],
                same_run_1gpu=dict(value=C5_FILTERS * single["steps"] / (single["ms"] * 1e-3), unit=UNIT, ms_per_step=single["ms"] / single["steps"],
                                   steps=single["steps"], note="all filters on rank 0 alone, same process, before the sharded run: what the N-GPU value scales from"))
    return line


# ---------------------------------------------------------------------------------------------------------------------
# reference arm
# ---------------------------------------------------------------------------------------------------------------------
def bench_reference(args, world, rank):
    """the reference's own CPU implementation on the GPU arm's workload; rank 0 only"""
    if rank != 0:
        return None
    from oracle import ref_py as R

    if not R.available():
        return dict(impl="reference", unavailable="oracle/_ref/libref.so missing (it is built from /root/reference by `make -C oracle ref`)")
    K, W = args.steps, args.warmup
    cores = os.cpu_count() or 1
    common = dict(impl="reference", unit=UNIT, n_gpus=world, steps=K, warmup=W, higher_is_better=True, vs_baseline=None, dtype="f64", data="synthetic",
                  config=config_for(world), gpu_launches=0)
    note = ("the reference is single threaded (no OpenMP in its CMakeLists.txt); its sources are compiled unmodified (-O3); third-party arithmetic (Eigen, "
            "OpenCV) is this repository's stand-in (oracle/ref_shim/), dense products through a packed AVX2 kernel; ROS, feature management and "
            "visualisation are not in the timed path")
    if world == 1:
        cam, scene, seq = make_c3(1)
        P0 = synth.assemble_P_numpy(scene)
        stats = c3_stats_from_oracle(cam, scene, seq, P0)
        smp = RefC3Sampler(cam, scene, seq, P0, stats)
        fixed = smp.measure_fixed()
        vals, plain, dts = [], [], []
        last = None
        for k in range(W + K):
            t0 = time.perf_counter()
            last = smp.sample(n_S=2, n_hyp=2)
            if k >= W:
                vals.append(last["frame_seconds_blocked"])
                plain.append(last["frame_seconds_plain"])
                dts.append(time.perf_counter() - t0)
        fs = float(np.mean(vals))
        v = 1.0 / fs
        cb = dict(value=v, unit=UNIT, cores=1, kind="reference", cpu_model=cpu_model(), host_cores=cores, sample=smp.describe(2, 2),
                  frame_seconds=fs, value_plain_product=1.0 / float(np.mean(plain)), frame_stats=stats,
                  per_unit=dict(fixed, t_S_per_feature=last["t_S_per_feature"], t_per_hypothesis=last["t_per_hypothesis"]), gemm_gflops=last["gemm_gflops"],
                  breakdown_seconds=last["breakdown_seconds_blocked"], seconds_of_cpu_work_per_step=float(np.mean(dts)))
        return dict(common, metric=METRIC_C3, value=v, ms_per_step=1e3 * fs, scaling="weak", cpu_baseline=cb,
                    e2e=dict(value=v, unit=UNIT, h2d_bytes_per_step=0, d2h_bytes_per_step=0), note=note)
    # C5: whole frames of 100-feature filters, one filter-frame per step (the filters are independent: frames/s per filter-frame IS the
    # aggregate rate of a single-threaded reference)
    scene, seq = make_c2(1234, W + K)
    rc = RefC2(scene, seq)
    dts = [rc.step() for _ in range(W + K)][W:]
    v = len(dts) / float(np.sum(dts))
    cb = dict(value=v, unit=UNIT, cores=1, kind="reference", cpu_model=cpu_model(), host_cores=cores,
              sample=f"{K} whole frames of ONE of the {C5_FILTERS} filters (after {W} warm-up frames) through the reference's own call sequence; the filters are "
                     "independent, so a single-threaded reference processes them at this rate", frame_stats=rc.stats())
    return dict(common, metric=METRIC_C5, value=v, ms_per_step=1e3 * float(np.mean(dts)), scaling="strong", cpu_baseline=cb,
                e2e=dict(value=v, unit=UNIT, h2d_bytes_per_step=0, d2h_bytes_per_step=0), note=note)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-extras", action="store_true")
    ap.add_argument("--extras", default="c2,c4,c5")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the outputs of the last timed step as DIR/<name>.npy (float32 / float64, at most 64 MB), "
                                                         "to compare two builds output for output")
    args = ap.parse_args()
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the outputs of the CUDA path (--impl b200)")
    if args.warmup < 3 and args.impl == "b200":
        args.warmup = 3
    # stdout carries exactly ONE line, the JSON: everything libraries print while we run (NCCL's version banner ...) goes to stderr
    sys.stdout.flush()
    json_fd = os.dup(1)
    os.dup2(2, 1)

    def emit(obj):
        os.write(json_fd, (json.dumps(obj) + "\n").encode())

    if args.impl == "reference":
        rank = int(os.environ.get("RANK", "0"))
        world = int(os.environ.get("WORLD_SIZE", "1"))
        line = bench_reference(args, world, rank)
        if line is not None:
            emit(line)
        return
    world, rank, local = dist_setup(args.gpus)
    if world == 1:
        line = bench_c3(args, world, rank, local)
    else:
        line = c5_line(args, world, rank, local)
    if not args.no_extras:
        try:
            import bench_extras

            wl = bench_extras.run(args, world, rank, local)
            if line is not None:
                line["workloads"] = wl
        except Exception as e:  # extras must never cost the main line
            if line is not None:
                line["workloads"] = dict(error=repr(e))
    if rank == 0:
        emit(line)
    if world > 1:
        import torch.distributed as dist

        dist.destroy_process_group()


if __name__ == "__main__":
    main()
