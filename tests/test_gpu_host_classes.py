"""The drop-in C++ host classes (ExtendKF / Map / Tracking, reference method names) driven in System::TrackRunning's call order by
ransac_slam_b200/lib/rslam_replay must reproduce the direct C-ABI run bit for bit (same kernels, same order)."""
import os
import struct
import subprocess

import numpy as np
import pytest

from ransac_slam_b200 import synth
from tests import helpers as H

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_host_classes_replay(tmp_path):
    exe = os.path.join(ROOT, "ransac_slam_b200", "lib", "rslam_replay")
    assert os.path.exists(exe), "run __graft_entry__.build() first"
    scene = synth.make_scene(N=50, seed=33)
    T = 5
    seq = synth.make_sequence(scene, T=T, seed=34)
    n = scene.x0.size
    dump = tmp_path / "dump.bin"
    with open(dump, "wb") as f:
        f.write(struct.pack("<6i", scene.N, n, T, scene.cam.nRows, scene.cam.nCols, seq.u01.shape[1]))
        f.write(scene.cam.as9().tobytes())
        f.write(scene.x0.tobytes())
        f.write(np.asfortranarray(scene.P0).tobytes(order="F"))
        f.write(scene.templates.astype(np.float64).tobytes())
        for k in range(T):
            f.write(seq.images[k].tobytes())
            f.write(seq.u01[k].tobytes())
    out = tmp_path / "out.bin"
    r = subprocess.run([exe, str(dump), str(out)], capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stderr
    raw = open(out, "rb").read()
    rec = 13 * 8 + 12
    assert len(raw) == T * rec
    g = H.gpu_from(scene, scene.x0, scene.P0, prior=False)
    g.set_graph(False)
    for k in range(T):
        g.frame(seq.images[k][None], seq.u01[k][None])
        x13 = np.frombuffer(raw[k * rec:k * rec + 104], dtype=np.float64)
        cnt = np.frombuffer(raw[k * rec + 104:(k + 1) * rec], dtype=np.int32)
        ft = g.features()
        assert np.array_equal(x13, g.download_pose()), k
        assert list(cnt) == [int(ft["ic"].sum()), int(ft["li"].sum()), int(ft["hi"].sum())]


def test_pgm_replay_through_host_classes_matches_the_reference(tmp_path):
    """configuration C1 end to end: frames of the reference's bundled sequence written as P5 files, replayed by the C++ drop-in
    classes in System::System / System::TrackRunning order (rslam_replay_pgm), against the outputs of the reference's own sources
    (tests/golden/ref_vectors.*.npz) fed the same libc draws."""
    from oracle import ref_py as R  # only for the settings template (numbers of examples/Monocular/initialize_param.yaml)
    from tests import ref_cases as RC

    exe = os.path.join(ROOT, "ransac_slam_b200", "lib", "rslam_replay_pgm")
    assert os.path.exists(exe), "run __graft_entry__.build() first"
    g = RC.load()
    frames = np.load(os.path.join(RC.GOLD, "pgm_frames.npz"))["frames"]
    nf = int(g["bundled_frames"])
    yaml = tmp_path / "settings.yaml"
    yaml.write_text(R.YAML_TEMPLATE.format(**R.BUNDLED_YAML))
    names = []
    with open(tmp_path / "draws.bin", "wb") as d:
        for k in range(nf):
            p = tmp_path / f"rawoutput{k:04d}.pgm"
            with open(p, "wb") as f:
                f.write(b"P5\n# bundled frame\n320 240\n255\n")
                f.write(frames[k].tobytes())
            names.append(str(p))
            d.write(g[f"bundled_k{k}_draws_map"][:100].astype("<i4").tobytes())
            d.write(g[f"bundled_k{k}_draws_ransac"].astype("<i4").tobytes())
    out = tmp_path / "out.bin"
    r = subprocess.run([exe, str(yaml), str(out), "--draws", str(tmp_path / "draws.bin")] + names, capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stderr
    raw = open(out, "rb").read()
    rec = 13 * 8 + 6 * 4
    assert len(raw) == nf * rec
    for k in range(nf):
        x13 = np.frombuffer(raw[k * rec:k * rec + 104], dtype=np.float64)
        cnt = np.frombuffer(raw[k * rec + 104:(k + 1) * rec], dtype=np.int32)
        pre = f"bundled_k{k}_"
        H.assert_x_close(x13, g[pre + "x"][:13], what=f"camera state after frame {k}")
        assert cnt[0] == g[pre + "types"].size and cnt[1] == g[pre + "ic"].sum() and cnt[2] == g[pre + "li"].sum() and cnt[3] == g[pre + "hi"].sum(), (k, cnt)


_UPDATE_SRC = r'''
#include <cstdio>
#include <cstdlib>
#include <vector>
#include "ransac_slam/ExtendKF.h"
using namespace ransac_slam;
// reads n, k, x(n), P(n x n col-major), H(k x n col-major), z(k), h(k) as doubles from argv[1]; writes x_k_k (n) and p_k_k (n x n) to argv[2]
int main(int argc, char** argv) {
    FILE* f = fopen(argv[1], "rb");
    double hdr[2];
    if (fread(hdr, 8, 2, f) != 2) return 2;
    const int n = (int)hdr[0], k = (int)hdr[1];
    Eigen::VectorXd x(n), z(k), h(k);
    Eigen::MatrixXd P(n, n), H(k, n), R(k, k);
    if (fread(x.data(), 8, n, f) != (size_t)n || fread(P.data(), 8, (size_t)n * n, f) != (size_t)n * n || fread(H.data(), 8, (size_t)k * n, f) != (size_t)k * n ||
        fread(z.data(), 8, k, f) != (size_t)k || fread(h.data(), 8, k, f) != (size_t)k)
        return 3;
    fclose(f);
    for (int i = 0; i < k; i++) for (int j = 0; j < k; j++) R(i, j) = i == j ? 1.0 : 0.0;
    CamParam cam;
    cam.k1 = 0.06333; cam.k2 = 0.01390; cam.nRows = 240; cam.nCols = 320; cam.dx = cam.dy = 0.0112; cam.f = 2.1735;
    cam.Cx = 1.7945 / 0.0112; cam.Cy = 1.4433 / 0.0112;
    ExtendKF kf("", &cam, "constant_velocity");
    const int N = (n - 13) / 6;
    kf.features_info.resize(N);  // inverse-depth features (the default type)
    kf.update(x, P, H, R, z, h);
    if (kf.last_status() != 0) { fprintf(stderr, "update failed: %d %s\n", kf.last_status(), rslam_last_error()); return 4; }
    // a Jacobian without the measurement structure must be refused, not silently mangled
    Eigen::MatrixXd Hbad = H;
    Hbad(0, 8) = 1.0;  // velocity column
    Eigen::VectorXd xk = kf.x_k_k;
    kf.update(x, P, Hbad, R, z, h);
    if (kf.last_status() == 0) return 5;
    kf.x_k_k = xk;
    FILE* o = fopen(argv[2], "wb");
    fwrite(kf.x_k_k.data(), 8, n, o);
    fwrite(kf.p_k_k.data(), 8, (size_t)n * n, o);
    fclose(o);
    return 0;
}
'''


def test_host_extendkf_update_runs_on_the_device(tmp_path):
    """ExtendKF::update(x, P, H, R, z, h) of the C++ drop-in class (src/ExtendKF.cpp:597-639): dense caller-built H with the structure of
    stacked measurement Jacobians goes through rslam_upload_linearisation + the device update; against the numpy restatement."""
    from oracle import np_oracle as NP

    host = os.path.join(ROOT, "ransac_slam_b200", "host")
    lib = os.path.join(ROOT, "ransac_slam_b200", "lib")
    src = tmp_path / "upd.cpp"
    src.write_text(_UPDATE_SRC)
    exe = str(tmp_path / "upd")
    gxx = "/usr/bin/g++" if os.path.exists("/usr/bin/g++") else "g++"
    r = subprocess.run([gxx, "-std=c++17", "-O1", "-w", "-I", host, str(src), os.path.join(host, "host_classes.cpp"), "-o", exe, "-L", lib, "-lrslam_b200",
                        "-Wl,-rpath," + lib], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr[-3000:]
    # a prior and a linearisation from a real prediction (oracle), measurements for features 1, 4, 5 of 8
    scene, x, P = synth.random_spd_state(8, seed=141)
    o = H.oracle_from(scene, x, P, sparse=False)
    o.search_ic_matches(None)
    fo = o.features()
    sel = [1, 4, 5]
    assert fo["has_h"][sel].all()
    n = x.size
    Hd = np.vstack([o.H_dense(i) for i in sel])
    h = fo["h"][sel].reshape(-1)
    z = np.rint(h) + np.tile([0.6, -0.4], len(sel))
    with open(tmp_path / "in.bin", "wb") as f:
        f.write(np.array([n, len(z)], dtype=np.float64).tobytes())
        f.write(x.tobytes())
        f.write(np.asfortranarray(P).tobytes(order="F"))
        f.write(np.asfortranarray(Hd).tobytes(order="F"))
        f.write(z.tobytes())
        f.write(h.tobytes())
    r = subprocess.run([exe, str(tmp_path / "in.bin"), str(tmp_path / "out.bin")], capture_output=True, text=True, timeout=120)
    assert r.returncode == 0, (r.returncode, r.stderr)
    raw = np.fromfile(tmp_path / "out.bin", dtype=np.float64)
    xg, Pg = raw[:n], raw[n:].reshape(n, n, order="F")
    xn, Pn = NP.ekf_update(x, P, Hd, z, h)
    H.assert_x_close(xg, xn)
    H.assert_P_close(Pg, Pn)
