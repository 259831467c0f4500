"""Writes tests/golden/checkpoint_v1.bin: a snapshot (rslam_checkpoint_save, format version 1) of a small deterministic state --
two filters of N = 5 and N = 12 features, feature 3 of the second one cartesian, with counters, flags, linearisation, templates
and initialisation records set.  state() builds the arrays from uniform draws with element-wise numpy only (no BLAS product, no
libm call), so they are the same bits on any machine and tests can compare the committed file against them without a GPU; writing
the file needs one.

    python tests/golden/make_checkpoint_vectors.py [out.bin]
"""
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
OUT = os.path.join(ROOT, "tests", "golden", "checkpoint_v1.bin")
NMAX = 16


def _filter_state(seed, N, cartesian=()):
    """Uniform draws and IEEE additions / multiplications only -- no BLAS product, no libm call -- so the arrays are the same bits on
    every machine (a format pin needs no physically meaningful state, only an exactly symmetric P)."""
    from ransac_slam_b200 import synth

    rng = np.random.default_rng(500 + seed)
    types = np.zeros(N, np.int32)
    types[list(cartesian)] = 1
    n = 13 + int(np.sum(np.where(types == 0, 6, 3)))
    x = rng.uniform(-2.0, 2.0, n)
    A = rng.uniform(-1.0, 1.0, (n, n))
    P = np.asfortranarray((A + A.T) / 2)  # exactly symmetric, as the library keeps it
    flags = (rng.random((N, 4)) < 0.5).astype(np.uint8)
    return dict(cam9=synth.Camera().as9(), std_z=1.0, x=x, x_k_km1=x + rng.uniform(-1e-3, 1e-3, n), P=P, types=types,
                times_predicted=rng.integers(0, 20, N).astype(np.int32), times_measured=rng.integers(0, 20, N).astype(np.int32), flags=flags,
                h=rng.uniform(0, 320, (N, 2)), Hc=rng.uniform(-3, 3, (N, 2, 7)), Hf=rng.uniform(-3, 3, (N, 2, 6)), z=rng.uniform(0, 320, (N, 2)),
                templates=rng.integers(0, 256, (N, 13, 13)).astype(np.float64), patch41=rng.integers(0, 256, (N, 41, 41)).astype(np.uint8),
                r_wc=rng.uniform(-2, 2, (N, 3)), R_wc=rng.uniform(-1, 1, (N, 9)), uv=rng.uniform(20, 300, (N, 2)))


def state():
    """the two filters' arrays (numpy only)"""
    return [_filter_state(3, 5), _filter_state(4, 12, cartesian=(3,))]


def expected(m):
    """what read_checkpoint returns for filter m (S is not uploadable and stays zero)"""
    N = m["types"].size
    pose14 = np.concatenate([m["r_wc"], m["R_wc"], m["uv"]], axis=1)
    Hf = m["Hf"].copy()
    return dict(n=m["x"].size, N=N, types=m["types"], x=m["x"], x_k_km1=m["x_k_km1"], P=m["P"], times_predicted=m["times_predicted"],
                times_measured=m["times_measured"], has_h=m["flags"][:, 0].astype(bool), ic=m["flags"][:, 1].astype(bool), li=m["flags"][:, 2].astype(bool),
                hi=m["flags"][:, 3].astype(bool), h=m["h"], S=np.zeros((N, 2, 2)), z=m["z"], Hc=m["Hc"], Hf=Hf,
                patches=m["templates"].astype(np.float32), patch41=m["patch41"], pose14=pose14)


def load_into(g, b, m):
    """the uploads that put filter m into slot b of handle g"""
    g.upload_state(m["x"], m["P"], feat_types=m["types"], b=b, prior=False)
    g.upload_state(m["x_k_km1"], None, feat_types=m["types"], b=b, prior=True)  # same shape: nothing is cleared
    g.set_counters(m["times_predicted"], m["times_measured"], b=b)
    g.upload_linearisation(m["h"], m["Hc"], m["Hf"], m["z"], m["flags"], b=b)
    g.upload_patches(m["templates"], b=b)
    g.upload_feature_init(m["patch41"], m["r_wc"], m["R_wc"], m["uv"], b=b)


def make_handle(batch=2, nmax=NMAX):
    from ransac_slam_b200 import capi

    ms = state()
    return capi.Filter(ms[0]["cam9"], nmax, batch=batch, std_z=ms[0]["std_z"]), ms


def main(out=OUT):
    g, ms = make_handle()
    for b, m in enumerate(ms):
        load_into(g, b, m)
    buf = g.save()
    with open(out, "wb") as fh:
        fh.write(buf.tobytes())
    print(f"wrote {out}: {buf.size} bytes")


if __name__ == "__main__":
    main(*sys.argv[1:])
