"""k_gemm_dmma on the shapes of the C3 high-innovation update (N = 2000 features, n = 12013), against cuBLAS on the same operands.

One call measures, for each library given with --lib (they alternate --rounds times: base, new, base, new, ...):
  * per-kernel ms per update from the instrumented pass (rslam_profile_enable / rslam_profile_read) over --updates updates after
    --warmup, for k = 3260 and k = 3976 (rslam_upload_state_device + rslam_upload_linearisation + rslam_update_hi; the state and
    covariance are restored before every update, outside the kernels' events);
  * with a library built with -DRSLAM_PHASE_CLOCKS (--clock-lib), the per-CTA timeline of syrk_P and of the first trsm_outer launch:
    main-loop cycles per k-chunk, prologue (until the first chunk has landed) and epilogue cycles, the gap between one CTA's end and
    the next CTA's start on an SM slot, and the wave tail;
and, once: cuBLAS fp64 (torch.mm) on the syrk_P operand shape (n+1) x k . k x (n+1) and on the trsm_outer shapes
(n+1) x 1024 . 1024 x (k - 1024 (J + 1)), the register-only DMMA probe tools/ubench/dmma_peak (--dmma-peak, a binary built with
the command in its header), and the card's name, power limit and SM clocks.

Rates: syrk_P does the lower triangle, (n+1)^2 k flop (bench.py's convention); cuBLAS does the full product, 2 (n+1)^2 k flop.
Needs a GPU; writes one JSON file (--out)."""
import argparse
import json
import os
import re
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

N_FEAT, KS, OB = 2000, (3260, 3976), 1024


def gpu_info():
    q = "name,power.limit,clocks.sm,clocks.max.sm"
    try:
        r = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader"], capture_output=True, text=True, timeout=30)
        return dict(query=q, value=r.stdout.strip().splitlines()[0] if r.returncode == 0 and r.stdout.strip() else None)
    except Exception as e:  # the torch device name below still identifies the card
        return dict(query=q, value=f"unavailable: {e}")


def problem(dev, seed=5):
    """x, P (device, n x n column-major) and the linearisation of N_FEAT inverse-depth features; each H row scaled so that its
    H P H^T entry is 10..100 px^2, as in tests/test_gpu_update_kernels.py."""
    import torch

    rng = np.random.default_rng(seed)
    N = N_FEAT
    n = 13 + 6 * N
    sd = np.concatenate([[0.004] * 3, [0.001] * 4, [0.01] * 3, [0.003] * 3, np.tile([0.002, 0.002, 0.002, 0.001, 0.001, 0.03], N)])
    U = rng.standard_normal((n, 6)) * np.sqrt(0.1 / 6)
    d = rng.uniform(0.5, 1.5, n)
    x = np.zeros(n)
    q = np.array([0.97, 0.06, -0.2, 0.04])
    x[3:7] = q / np.linalg.norm(q)
    x[13 + 5::6] = 0.1
    Hc = rng.standard_normal((N, 2, 7))
    Hf = rng.standard_normal((N, 2, 6))
    for i in range(N):
        idx = np.r_[0:7, 13 + 6 * i:19 + 6 * i]
        Ps = (U[idx] @ U[idx].T + np.diag(d[idx])) * np.outer(sd[idx], sd[idx])
        for r in range(2):
            gr = np.r_[Hc[i, r], Hf[i, r]]
            s = np.sqrt(rng.uniform(10.0, 100.0) / (gr @ Ps @ gr))
            Hc[i, r] *= s
            Hf[i, r] *= s
    h = np.column_stack([rng.uniform(5, 1275, N), rng.uniform(5, 955, N)])
    z = h + rng.standard_normal((N, 2))
    Ud, sdd = torch.from_numpy(U).to(dev), torch.from_numpy(sd).to(dev)
    P = Ud @ Ud.T
    P.diagonal().add_(torch.from_numpy(d).to(dev))
    P.mul_(sdd[:, None]).mul_(sdd[None, :])
    P = (P + P.T) * 0.5  # exactly symmetric: the row-major storage is the column-major matrix
    return torch.from_numpy(x).to(dev), P.contiguous(), (h, Hc, Hf, z)


def timeline(rows):
    """per-CTA stamps (start_ns, end_ns, clk_start, clk_first_chunk, clk_loop_end, clk_end, smid, chunks) -> summary"""
    r = rows[rows[:, 0] != 0].astype(np.float64)
    if r.size == 0:
        return None
    t0, t1, c0, c1, c2, c3, sm, nk = r.T
    out = dict(ctas=int(r.shape[0]), sms=int(np.unique(sm).size), chunks_median=float(np.median(nk)))
    loop = c2 - c1
    out["main_loop_cycles_per_chunk"] = dict(median=float(np.median(loop / np.maximum(nk - 1, 1))), p10=float(np.percentile(loop / np.maximum(nk - 1, 1), 10)),
                                             p90=float(np.percentile(loop / np.maximum(nk - 1, 1), 90)))
    # one 128 x 64 x 16 chunk = 2 * 128 * 64 * 16 flop; two CTAs share an SM
    fpc = 2.0 * 128 * 64 * 16 / out["main_loop_cycles_per_chunk"]["median"]
    out["main_loop_flop_per_cycle_per_cta"] = fpc
    ghz = float(np.median((c3 - c0) / np.maximum(t1 - t0, 1)))  # the SM clock while the kernel ran, from the stamps themselves
    out["sm_ghz_from_stamps"] = ghz
    out["main_loop_tflops_two_ctas_per_sm_all_sms"] = 2 * fpc * 148 * ghz * 1e9 / 1e12
    out["prologue_cycles"] = dict(median=float(np.median(c1 - c0)), p90=float(np.percentile(c1 - c0, 90)))
    out["epilogue_cycles"] = dict(median=float(np.median(c3 - c2)), p90=float(np.percentile(c3 - c2, 90)))
    out["cta_ns"] = dict(median=float(np.median(t1 - t0)))
    # slots: on each SM, a CTA takes the slot that ended most recently at or before its start
    gaps, slot_last_end = [], []
    for s in np.unique(sm):
        sel = np.argsort(t0[sm == s])
        st, en = t0[sm == s][sel], t1[sm == s][sel]
        slots = []
        for a, b in zip(st, en):
            free = [i for i, e in enumerate(slots) if e <= a]
            if free:
                i = max(free, key=lambda i: slots[i])
                gaps.append(a - slots[i])
                slots[i] = b
            else:
                slots.append(b)
        slot_last_end += slots
    span0, span1 = t0.min(), t1.max()
    out["slot_gap_ns"] = dict(median=float(np.median(gaps)) if gaps else None, mean=float(np.mean(gaps)) if gaps else None, count=len(gaps))
    out["span_ns"] = float(span1 - span0)
    le = np.array(slot_last_end)
    out["tail_ns"] = dict(end_minus_median_slot_end=float(span1 - np.median(le)), idle_slot_fraction=float(np.sum(span1 - le) / (le.size * (span1 - span0))),
                          slots=int(le.size))
    ts = np.unique(np.concatenate([t0, t1]))
    out["globaltimer_step_ns"] = float(np.min(np.diff(ts))) if ts.size > 1 else None
    return out


def worker(args):
    """one library (RSLAM_LIB is set by the caller): per-kernel ms per update for each k, and the stamps if the library has them"""
    import ctypes as C

    import torch

    from ransac_slam_b200 import capi, synth

    dev = torch.device("cuda", 0)
    x, P, (h, Hc, Hf, z) = problem(dev)
    n = x.numel()
    g = capi.Filter(synth.Camera().as9(), N_FEAT)
    stamps_fn = getattr(g.L, "rslam_debug_gemm_stamps", None)
    if stamps_fn is not None:
        stamps_fn.argtypes = [C.c_int, C.c_void_p, C.c_int]
    res = {}
    for k in KS:
        flags = np.zeros((N_FEAT, 4), np.uint8)
        flags[:, :2] = 1
        flags[np.random.default_rng(k).choice(N_FEAT, k // 2, replace=False), 3] = 1

        def one():
            g.upload_state_device(x.data_ptr(), P.data_ptr(), n, n, N_FEAT)
            g.upload_linearisation(h, Hc, Hf, z, flags)
            g.update_hi()

        for _ in range(args.warmup):
            one()
        g.sync()
        g.profile(True)
        g.profile_read()
        tot = {}
        for _ in range(args.updates):
            one()
            for name, (cnt, ms) in g.profile_read().items():  # read per update: the event list stays short
                c0, m0 = tot.get(name, (0, 0.0))
                tot[name] = (c0 + cnt, m0 + ms)
        g.profile(False)
        r = {name: dict(launches=cnt / args.updates, ms=ms / args.updates) for name, (cnt, ms) in tot.items()}
        if stamps_fn is not None:
            one()
            g.sync()
            st = {}
            for rec, name in ((0, "syrk_P"), (1, "trsm_outer_first")):
                buf = np.zeros((16384, 8), np.uint64)
                cnt = stamps_fn(rec, buf.ctypes.data, 16384)
                st[name] = buf[:max(cnt, 0)]
            if args.stamp_dir:
                np.savez_compressed(os.path.join(args.stamp_dir, f"stamps_k{k}.npz"), **st)
            r["_stamps"] = {name: timeline(v) for name, v in st.items()}
        res[str(k)] = r
    g.close()
    print(json.dumps(res))


def cublas(reps=5):
    import torch

    n1 = 13 + 6 * N_FEAT + 1
    out = {}

    def timed(a, b):
        for _ in range(2):
            torch.mm(a, b)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(reps):
            torch.mm(a, b)
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) / reps

    for k in KS:
        a = torch.randn(n1, k, dtype=torch.float64, device="cuda")
        b = torch.randn(k, n1, dtype=torch.float64, device="cuda")
        ms = timed(a, b)
        d = dict(syrk_shape=dict(ms=ms, tflops=2.0 * n1 * n1 * k / (ms * 1e-3) / 1e12))
        del b
        tr = []
        for J in range(k // OB + 1):
            w = k - OB * (J + 1)
            if w <= 0:
                break
            bb = torch.randn(OB, w, dtype=torch.float64, device="cuda")
            ms = timed(a[:, :OB].contiguous(), bb)
            tr.append(dict(J=J, cols=w, ms=ms, tflops=2.0 * n1 * OB * w / (ms * 1e-3) / 1e12))
        d["trsm_outer_shapes"] = tr
        d["trsm_outer_total_ms"] = sum(t["ms"] for t in tr)
        out[str(k)] = d
        del a
        torch.cuda.empty_cache()
    return out


def rates(per_k):
    """algorithmic TFLOP/s of syrk_P and trsm_outer from one library's per-kernel ms"""
    n1 = 13 + 6 * N_FEAT + 1
    out = {}
    for k, r in per_k.items():
        k = int(k)
        row = {}
        if "k_gemm_dmma/syrk_P" in r:
            row["syrk_P"] = dict(ms=r["k_gemm_dmma/syrk_P"]["ms"], tflops=float(n1) * n1 * k / (r["k_gemm_dmma/syrk_P"]["ms"] * 1e-3) / 1e12)
        if "k_gemm_dmma/trsm_outer" in r:
            fl = sum(2.0 * n1 * OB * (k - OB * (J + 1)) for J in range(k // OB + 1) if k > OB * (J + 1))
            row["trsm_outer"] = dict(ms=r["k_gemm_dmma/trsm_outer"]["ms"], tflops=fl / (r["k_gemm_dmma/trsm_outer"]["ms"] * 1e-3) / 1e12)
        out[str(k)] = row
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--lib", action="append", default=[], metavar="NAME=PATH", help="library to time (repeatable); default: the tree's own")
    ap.add_argument("--clock-lib", metavar="PATH", help="a build with -DRSLAM_PHASE_CLOCKS: per-CTA timelines (one pass, after the timed rounds)")
    ap.add_argument("--dmma-peak", metavar="PATH", help="the tools/ubench/dmma_peak binary")
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--updates", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--out", default="profiles/r05_gemm_dmma_b200.json")
    ap.add_argument("--worker", action="store_true", help=argparse.SUPPRESS)
    ap.add_argument("--stamp-dir", help=argparse.SUPPRESS)
    args = ap.parse_args()
    if args.worker:
        return worker(args)
    import torch

    libs = [tuple(s.split("=", 1)) for s in args.lib] or [("tree", os.path.join(ROOT, "ransac_slam_b200", "lib", "librslam_b200.so"))]
    info = dict(gpu=gpu_info(), torch_device=torch.cuda.get_device_name(0))

    def run(path, extra=()):
        env = dict(os.environ, RSLAM_LIB=os.path.abspath(path))
        cmd = [sys.executable, os.path.abspath(__file__), "--worker", "--updates", str(args.updates), "--warmup", str(args.warmup)] + list(extra)
        p = subprocess.run(cmd, env=env, capture_output=True, text=True)
        if p.returncode != 0:
            raise RuntimeError(f"{path}: {p.stderr[-3000:]}")
        return json.loads(p.stdout.strip().splitlines()[-1])

    runs = []
    for rnd in range(args.rounds):
        for name, path in libs:
            r = run(path)
            runs.append(dict(lib=name, round=rnd, per_kernel=r, rates=rates(r)))
            print(f"round {rnd} {name}: " + "  ".join(f"k={k} syrk_P {v['syrk_P']['ms']:.3f} ms trsm_outer {v.get('trsm_outer', {}).get('ms', 0):.3f} ms"
                                                       for k, v in runs[-1]["rates"].items()), file=sys.stderr)
    summary = {}
    for name, _ in libs:
        mine = [r for r in runs if r["lib"] == name]
        summary[name] = {k: {kern: dict(ms_min=min(r["rates"][k][kern]["ms"] for r in mine), ms_max=max(r["rates"][k][kern]["ms"] for r in mine),
                                        tflops_best=max(r["rates"][k][kern]["tflops"] for r in mine))
                             for kern in mine[0]["rates"][k]} for k in mine[0]["rates"]}
    out = dict(info, n=13 + 6 * N_FEAT, ks=list(KS), updates=args.updates, rounds=args.rounds, libs=dict(libs), runs=runs, summary=summary)
    out["cublas"] = cublas()
    for name in summary:
        for k, v in summary[name].items():
            if "syrk_P" in v:
                v["syrk_P"]["vs_cublas"] = v["syrk_P"]["tflops_best"] / out["cublas"][k]["syrk_shape"]["tflops"]
            if "trsm_outer" in v:
                v["trsm_outer"]["vs_cublas"] = out["cublas"][k]["trsm_outer_total_ms"] / v["trsm_outer"]["ms_min"]
    if args.clock_lib:
        sd = os.path.join(os.path.dirname(os.path.abspath(args.out)), "gemm_dmma_stamps")
        os.makedirs(sd, exist_ok=True)
        extra = ["--stamp-dir", sd]
        out["timelines"] = {k: v.get("_stamps") for k, v in run(args.clock_lib, extra).items()}
    if args.dmma_peak:
        p = subprocess.run([args.dmma_peak], capture_output=True, text=True, timeout=600)
        vals = [float(v) for v in re.findall(r"([\d.]+) TFLOP/s", p.stdout) if float(v) < 1000]
        out["dmma_peak"] = dict(best_tflops=max(vals) if vals else None, log=p.stdout)
    out["gpu_after"] = gpu_info()
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(out, f, indent=1)
    print(json.dumps(dict(summary=summary, cublas={k: v["syrk_shape"] for k, v in out["cublas"].items()}, gpu=info["gpu"]["value"])))


if __name__ == "__main__":
    main()
