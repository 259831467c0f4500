"""Time rslam_checkpoint_save / rslam_checkpoint_load against the per-filter download calls.

  C5 shape   4096 filters of 100 features (max_features 110): snapshot of the whole batch.
  C3 shape   1 filter of 2000 features (a 577 MB triangle).
  paths      save and load to pinned host memory, to pageable host memory, and device to device (a CUDA buffer on the same GPU).
  rates      snapshot bytes over the call time, against the host link (a plain pinned copy of 1 GiB each way, measured in the same
             run) and against the HBM figure bench.py uses.  For the device path the HBM bytes are counted as the snapshot written
             plus what the pack reads (the whole square of P: each lower tile and its mirror) -- and the reverse for the load.
  baseline   download_state + features + download_patches + one download_feature_init per feature on --subset filters, ms per
             filter; the 4096 figure is an extrapolation, labelled as such.

Host clock around the blocking calls (each returns when its copy is complete); --reps timed calls after one warm-up call per path.
Needs a GPU; writes one JSON file (--out) with the card's name, power limit and max SM clock read in the same run."""
import argparse
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from tools.bench_map_batch import gpu_info, hbm_peak  # noqa: E402


def wall(fn, reps):
    fn()  # warm-up
    ms = []
    for _ in range(reps):
        t0 = time.perf_counter()
        fn()
        ms.append((time.perf_counter() - t0) * 1e3)
    return ms


def host_link(reps):
    """GB/s of a plain pinned 1 GiB copy each way (torch, synchronised)"""
    import torch

    nb = 1 << 30
    h = torch.empty(nb, dtype=torch.uint8, pin_memory=True)
    d = torch.empty(nb, dtype=torch.uint8, device="cuda:0")
    out = {}
    for name, fn in (("h2d", lambda: (d.copy_(h), torch.cuda.synchronize())), ("d2h", lambda: (h.copy_(d), torch.cuda.synchronize()))):
        ms = wall(fn, reps)
        out[name + "_gbs"] = nb / (min(ms) * 1e-3) / 1e9
    del h, d
    return out


def make(B, N, nmax, big):
    import torch

    from ransac_slam_b200 import capi, synth

    dev = torch.device("cuda", 0)
    if big:
        cam = synth.scaled_camera(4)
        scene = synth.make_scene(N=N, seed=1234, cam=cam, margin=30, min_sep=18, assemble_P=False, motion_scale=0.25)
        P = synth.assemble_P_torch(scene, dev)
        x = scene.x0.copy()
    else:
        scene, x, Pn = synth.random_spd_state(N, seed=5)
        cam = scene.cam
        P = torch.from_numpy(np.asfortranarray(Pn).T.copy()).to(dev)
    P = (P + P.T) / 2  # exactly symmetric, as the library keeps it
    xd = torch.from_numpy(x).to(dev)
    g = capi.Filter(cam.as9(), nmax, batch=B)
    rng = np.random.default_rng(1)
    for b in range(B):
        g.upload_state_device(xd.data_ptr(), P.data_ptr(), x.size, x.size, N, b=b)
        g.set_counters(rng.integers(0, 20, N).astype(np.int32), rng.integers(0, 20, N).astype(np.int32), b=b)
    g.sync()
    del P
    torch.cuda.empty_cache()
    return g, cam, x.size


def bench_shape(B, N, nmax, big, reps, link, peak):
    import torch

    from ransac_slam_b200 import capi

    g, cam, n = make(B, N, nmax, big)
    nb = g.checkpoint_bytes()
    tri = B * 8 * (n * (n + 1) // 2)
    t = capi.Filter(cam.as9(), nmax, batch=B)
    pinned = torch.empty(nb, dtype=torch.uint8, pin_memory=True)
    pinned_np = pinned.numpy()
    pageable = np.empty(nb, dtype=np.uint8)
    device = torch.empty(nb, dtype=torch.uint8, device="cuda:0")
    res = dict(filters=B, features=N, max_features=nmax, n=n, snapshot_bytes=nb, triangle_bytes=tri, records_and_states_bytes=nb - tri,
               full_square_bytes=B * 8 * n * n)
    hbm_save = nb + B * 8 * n * n  # snapshot written + the square read (lower tiles and their mirrors)
    for path, buf in (("pinned", pinned_np), ("pageable", pageable), ("device", device)):
        l0 = g.launches
        g.save(out=buf)
        launches = g.launches - l0
        ms_s = wall(lambda: g.save(out=buf), reps)
        ms_l = wall(lambda: t.load(buf), reps)
        r = dict(save_ms=ms_s, load_ms=ms_l, save_ms_best=min(ms_s), load_ms_best=min(ms_l), save_launches=launches,
                 save_gbs=nb / (min(ms_s) * 1e-3) / 1e9, load_gbs=nb / (min(ms_l) * 1e-3) / 1e9)
        if path == "device":
            r["hbm_bytes_per_call"] = hbm_save
            r["save_frac_of_hbm"] = hbm_save / (min(ms_s) * 1e-3) / 1e9 / peak
            r["load_frac_of_hbm"] = hbm_save / (min(ms_l) * 1e-3) / 1e9 / peak
        else:
            r["save_frac_of_host_link_d2h"] = r["save_gbs"] / link["d2h_gbs"]
            r["load_frac_of_host_link_h2d"] = r["load_gbs"] / link["h2d_gbs"]
        res[path] = r
    assert np.array_equal(device.cpu().numpy(), pageable) and np.array_equal(pinned_np, pageable)  # every path wrote the same bytes
    del pinned, pinned_np, pageable, device
    t.close()
    return g, res


def per_filter_baseline(g, subset):
    """the existing per-filter reads of everything a snapshot holds, host clock"""

    def one(b):
        g.download_state(b=b)
        g.download_state(b=b, prior=True, want_P=False)
        g.features(b=b)
        g.H_sparse(b=b)
        g.download_patches(b=b)
        for i in range(g.L.rslam_num_features(g.h, b)):
            g.feature_init(i, b=b)

    one(0)
    t0 = time.perf_counter()
    for b in range(subset):
        one(b)
    ms = (time.perf_counter() - t0) * 1e3
    return dict(filters=subset, ms_total=ms, ms_per_filter=ms / subset, ms_extrapolated_to_4096=ms / subset * 4096,
                extrapolation=f"x 4096 / {subset}, not measured",
                calls="download_state (x, P) + download_state (x_k_km1) + download_features + download_H + download_patches + N download_feature_init")


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--filters", type=int, default=4096)
    ap.add_argument("--subset", type=int, default=64)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r04_checkpoint_b200.json"))
    a = ap.parse_args()
    import torch

    if not torch.cuda.is_available():
        sys.exit("bench_checkpoint.py needs a CUDA device")
    res = dict(gpu=gpu_info(), torch=torch.__version__, timing="host clock around each blocking call, best of --reps after one warm-up")
    peak, peak_src = hbm_peak()
    res["hbm_peak_gbs"], res["hbm_peak_source"] = peak, peak_src
    res["host_link"] = link = host_link(a.reps)
    g, res["c5"] = bench_shape(a.filters, 100, 110, False, a.reps, link, peak)
    res["c5_per_filter_baseline"] = per_filter_baseline(g, a.subset)
    res["c5_per_filter_baseline"]["speedup_vs_pinned_save_extrapolated"] = res["c5_per_filter_baseline"]["ms_extrapolated_to_4096"] / res["c5"]["pinned"]["save_ms_best"]
    g.close()
    del g
    torch.cuda.empty_cache()
    g, res["c3"] = bench_shape(1, 2000, 2000, True, a.reps, link, peak)
    g.close()
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as fh:
        json.dump(res, fh, indent=1)
    print(json.dumps(res))


if __name__ == "__main__":
    main()
