"""Time rslam_map_management_batch (Map::map_management for every filter of a batch) against the per-filter path.

  C5 shape   4096 filters of 100 features (max_features 110): every filter deletes 2 features, converts 1 and initialises
             --adds features (no feature blocks the sampling box).  ms per call, and the algorithmic bytes of the covariance pass,
             sum_b 8 (n_old^2 + n_new^2), over that time as a fraction of the HBM figure bench.py uses (MEASURED_PEAKS.json).
  baseline   the per-filter primitives in rslam_map_management's order on --subset of those filters (ms per filter; the 4096
             figure is an extrapolation, labelled as such).
  C3 shape   B = 1, N = 2000 (P 1.15 GB): the batched call against rslam_map_management on the same edits.

CUDA events on the library's stream around the call only; the inputs are restored from device copies between timed calls, outside
the events.  Needs a GPU; writes one JSON file (--out)."""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def gpu_info():
    import torch

    out = dict(name=torch.cuda.get_device_name(0))
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True, timeout=30)
        out["nvidia_smi"] = q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else None
    except Exception as e:  # the card name from torch still identifies the device
        out["nvidia_smi"] = f"unavailable: {e}"
    return out


def hbm_peak():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        return float(json.load(open(p)).get("hbm_gbs", 6650.0)), "measured (MEASURED_PEAKS.json)"
    return 6650.0, "fallback (B200_PROFILING.md)"


class Batch:
    """B copies of one map (device-resident source copies for restoring) on one handle"""

    def __init__(self, B, N, nmax, seed, n_del, cam=None, big=False):
        import torch

        from ransac_slam_b200 import capi, synth

        self.dev = torch.device("cuda", 0)
        if big:
            cam = synth.scaled_camera(4)
            scene = synth.make_scene(N=N, seed=1234, cam=cam, margin=30, min_sep=18, assemble_P=False, motion_scale=0.25)
            P = synth.assemble_P_torch(scene, self.dev)
            x = scene.x0.copy()
        else:
            scene, x, Pn = synth.random_spd_state(N, seed=seed)
            cam = scene.cam
            P = torch.from_numpy(np.ascontiguousarray(Pn.T)).to(self.dev)  # column-major == transpose of a symmetric matrix
        x[13 + 3::6] = np.pi  # every feature faces away: no feature blocks the sampling box
        ip = 13 + 6 * (N // 2)
        s = 1e-3 / torch.sqrt(P[ip + 5, ip + 5])
        P[ip + 5, :] *= s
        P[:, ip + 5] *= s
        self.x = torch.from_numpy(x).to(self.dev)
        self.P = P
        self.n, self.N, self.B = x.size, N, B
        self.tp = np.full(N, 10, np.int32)
        self.tm = np.full(N, 9, np.int32)
        self.tm[np.linspace(N // 10, N // 2, n_del).astype(int)] = 1  # early enough that the reference's run-ahead index stays in range
        self.g = capi.Filter(cam.as9(), nmax, batch=B)
        from tests import golden_npz

        img = golden_npz.load("pgm_frames_all")["frames"][0]
        reps = (cam.nRows // img.shape[0], cam.nCols // img.shape[1])
        self.img = np.tile(img, reps)
        self.cam = cam
        self.restore()
        self.g.set_image(self.img, share=True)

    def restore(self):
        for b in range(self.B):
            self.g.upload_state_device(self.x.data_ptr(), self.P.data_ptr(), self.n, self.n, self.N, b=b)
            self.g.set_counters(self.tp, self.tm, b=b)
        self.g.sync()


def timed(batch, fn, reps):
    import torch

    s = torch.cuda.ExternalStream(batch.g.stream)
    ms = []
    out = None
    for _ in range(reps):
        batch.restore()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(s)
        out = fn()
        e1.record(s)
        e1.synchronize()
        ms.append(e0.elapsed_time(e1))
    return ms, out


def per_filter_sequence(g, bs, step, min_features, u01):
    """rslam_map_management's order with the per-filter primitives on a handle of several filters"""
    meas = []
    for b in bs:
        g.map_delete_features(True, b=b)
        f = g.features(b=b)
        meas.append(int((f["li"] | f["hi"]).sum()))
    g.begin_frame()
    for i, b in enumerate(bs):
        g.map_inversedepth_to_cartesian(b=b)
        t = min_features if meas[i] == 0 else max(min_features - meas[i], 0)
        if t:
            g.map_initialize_features(step, t, u01[b], b=b)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--filters", type=int, default=4096)
    ap.add_argument("--subset", type=int, default=64)
    ap.add_argument("--adds", type=int, default=4)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--skip-c3", action="store_true")
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "map_batch_b200.json"))
    a = ap.parse_args()
    import torch

    if not torch.cuda.is_available():
        sys.exit("bench_map_batch.py needs a CUDA device")
    res = dict(gpu=gpu_info(), torch=torch.__version__)
    peak, peak_src = hbm_peak()
    n_pairs = 60
    rng = np.random.default_rng(3)

    # ---- C5 shape ----
    bt = Batch(a.filters, 100, 110, seed=5, n_del=2)
    u01 = rng.random((a.filters, 2 * n_pairs))
    call = lambda: bt.g.map_management_batch(1, a.adds, u01, True)  # noqa: E731
    timed(bt, call, 1)  # warm-up (first call allocates the spare buffers)
    ms, (rc, status, info) = timed(bt, call, a.reps)
    n_new = np.array([bt.g.L.rslam_state_dim(bt.g.h, b) for b in range(a.filters)], dtype=np.float64)
    nbytes = float(np.sum(8.0 * (bt.n**2 + n_new**2)))
    best = min(ms)
    res["c5_batched"] = dict(filters=a.filters, features=100, max_features=110, n_old=bt.n, n_new_mean=float(n_new.mean()), rc=int(rc),
                             deleted=int(info[:, 0].sum()), converted=int((info[:, 1] >= 0).sum()), initialised=int(info[:, 2].sum()),
                             ms_per_call=ms, ms_best=best, launches_per_call=None, algorithmic_bytes=nbytes,
                             achieved_gbs=nbytes / (best * 1e-3) / 1e9, hbm_peak_gbs=peak, hbm_peak_source=peak_src,
                             frac_of_hbm=nbytes / (best * 1e-3) / 1e9 / peak)
    l0 = bt.g.launches
    bt.restore()
    bt.g.map_management_batch(1, a.adds, u01, True)
    res["c5_batched"]["launches_per_call"] = bt.g.launches - l0
    # ---- per-filter baseline on a subset ----
    bs = list(range(a.subset))
    bt.restore()
    per_filter_sequence(bt.g, [0], 1, a.adds, u01)  # warm-up
    bt.restore()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    per_filter_sequence(bt.g, bs, 1, a.adds, u01)
    bt.g.sync()
    wall = (time.perf_counter() - t0) * 1e3
    res["c5_per_filter_subset"] = dict(filters=a.subset, ms_total=wall, ms_per_filter=wall / a.subset,
                                       ms_extrapolated_to_all=wall / a.subset * a.filters, extrapolation=f"x {a.filters} / {a.subset}, not measured",
                                       timing="host clock around the sequence, ending in a stream synchronise (the primitives synchronise internally)")
    bt.g.close()
    del bt
    torch.cuda.empty_cache()

    # ---- C3 shape ----
    if not a.skip_c3:
        big = Batch(1, 2000, 2001, seed=0, n_del=1, big=True)
        u1 = rng.random((1, 2 * n_pairs))
        out = {}
        for name, fn in (("batched", lambda: big.g.map_management_batch(1, 1, u1, True)),
                         ("per_filter", lambda: big.g.map_management(1, 1, u1[0], True))):
            timed(big, fn, 1)
            ms, r = timed(big, fn, a.reps)
            out[name] = dict(ms_per_call=ms, ms_best=min(ms), n_new=big.g.n)
        nb = 8.0 * (big.n**2 + out["batched"]["n_new"] ** 2)
        out["n_old"] = big.n
        out["algorithmic_bytes_batched"] = nb
        out["batched"]["frac_of_hbm"] = nb / (out["batched"]["ms_best"] * 1e-3) / 1e9 / peak
        res["c3_b1_n2000"] = out
        big.g.close()
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as fh:
        json.dump(res, fh, indent=1)
    print(json.dumps(res))


if __name__ == "__main__":
    main()
