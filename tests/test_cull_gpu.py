"""GPU: icg_ba_outlier_culling_resident (updateParametersFromOptimizer + gvinsOutlierCulling on the device, IG/ic_gvins.cc:1299-1389,
1035-1128) against the CPU restatement (tests/cull_oracle.py), and its effect on the resident marginalization."""
import copy
import os
import shutil
import subprocess
import tempfile

import numpy as np
import pytest

from datagen import synth_cull
from tests import cull_cases as cc
from tests import cull_oracle as co
from tests import oracle_api as oa
from tests.test_marg_gpu import compare

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def olib(oracle):
    oa.declare_ba(oracle)
    return oracle


@pytest.fixture(scope="module")
def solver():
    from ic_gvins_b200.ba import WindowSolver
    s = WindowSolver(max_windows=4, max_K=10, max_L=300, max_F=2700, max_gnss=16, max_marg_r=160)
    yield s
    s.close()


def windows(olib, seeds):
    return [synth_cull.make_cull_window(lambda *a: oa.preintegrate(olib, *a), seed=s) for s in seeds]


def same(g, o, tol=1e-12):
    assert g["ext_updated"] == o["ext_updated"]
    for k in ("counts", "f_outlier", "lm_ref_outlier", "lm_outlier"):
        assert np.array_equal(np.asarray(g[k]), np.asarray(o[k])), k
    for k in ("R_bc", "t_bc", "cam_pose", "lm_pos", "lm_depth"):
        x, y = np.asarray(g[k], np.float64).reshape(-1), np.asarray(o[k], np.float64).reshape(-1)
        assert x.size == y.size and (x.size == 0 or np.abs(x - y).max() <= tol * max(1.0, np.abs(y).max())), k


def test_gpu_culling_matches_oracle_on_the_solved_parameters(olib, solver):
    ws = windows(olib, [5, 6])
    probs, cins = [w[0] for w in ws], [w[1] for w in ws]
    solver.gvins_optimization_batch(probs, 20)  # parameters + chi2 mask written back
    chi2 = [p["f_active"].copy() for p in probs]
    ref = [co.outlier_culling(p, c) for p, c in zip(probs, cins)]
    got = solver.outlier_culling(probs, cins)
    for p, g, o, m in zip(probs, got, ref, chi2):
        same(g, o)
        assert np.array_equal(p["f_active"], o["f_active"]) and not np.array_equal(p["f_active"], m)
        assert g["counts"][2] > 0 and g["counts"][4] > 0


def test_gpu_solve_and_cull_matches_the_oracle_chain(olib, solver):
    prob, cin, _ = windows(olib, [7])[0]
    pg, po = copy.deepcopy(prob), copy.deepcopy(prob)
    solver.gvins_optimization_batch([pg], 20)
    g = solver.outlier_culling([pg], [cin])[0]
    cc.two_pass(olib, po)
    assert synth_cull.decision_margin(po, cin) > 1e-6
    o = co.outlier_culling(po, cin)
    for k in ("counts", "f_outlier", "lm_ref_outlier", "lm_outlier"):
        assert np.array_equal(g[k], o[k]), k
    assert np.array_equal(pg["f_active"], o["f_active"])
    assert np.abs(g["lm_pos"] - o["lm_pos"]).max() <= 1e-6 * np.abs(o["lm_pos"]).max()


def test_batch_equals_one_window_per_call(olib, solver):
    ws = windows(olib, [11, 12, 13, 14])
    base = [w[0] for w in ws]
    solver.gvins_optimization_batch(copy.deepcopy(base), 20)  # warm
    single = []
    for p, c in zip(base, [w[1] for w in ws]):
        q = copy.deepcopy(p)
        solver.gvins_optimization_batch([q], 20)
        single.append((solver.outlier_culling([q], [c])[0], q))
    batch = copy.deepcopy(base)
    solver.gvins_optimization_batch(batch, 20)
    got = solver.outlier_culling(batch, [w[1] for w in ws])
    for g, (s, q), b in zip(got, single, batch):
        same(g, s, tol=0.0)
        assert np.array_equal(b["f_active"], q["f_active"])


def test_hand_built_windows(olib, solver):
    prob, cin = cc.hand_window()
    o = co.outlier_culling(copy.deepcopy(prob), cin)
    solver.upload([prob])
    g = solver.outlier_culling([prob], [cin])[0]
    same(g, o)
    assert list(g["counts"]) == cc.EXPECT_COUNTS and np.array_equal(prob["f_active"], o["f_active"])
    for q, t, est in ((cc.rot([0.3, 1.0, 0.2], 9.0), [0.1, 0, 0], 1), (cc.rot([0.3, 1.0, 0.2], 11.0), [0, 0, 0], 1), (cc.rot([1, 0, 0], 1.0), [1.2, 0, 0], 1),
                      (cc.rot([0.3, 1.0, 0.2], 2.0), [0.1, 0, 0], 0)):
        pw, cw = cc.gate_window(np.array(q), np.array(t, np.float64), est)
        solver.upload([pw])
        same(solver.outlier_culling([pw], [cw])[0], co.outlier_culling(pw, cw), tol=0.0)


def test_cfg4_handle(olib):
    from ic_gvins_b200.ba import WindowSolver
    prob, cin, _ = synth_cull.make_cull_window(lambda *a: oa.preintegrate(olib, *a), K=20, L=2000, seed=21)
    sv = WindowSolver(max_windows=1, max_K=20, max_L=2000, max_F=prob["F"], max_gnss=16, max_marg_r=1)
    try:
        sv.gvins_optimization_batch([prob], 20)
        o = co.outlier_culling(prob, cin)
        same(sv.outlier_culling([prob], [cin])[0], o)
        assert o["counts"][0] > 0
    finally:
        sv.close()


def test_resident_marginalization_after_culling(olib, solver):
    """cull -> icg_ba_marginalize_resident == icg_ba_marginalize of the same dict with f_active = the culling mask (bit for bit), and the oracle"""
    ws = windows(olib, [5, 8])
    probs, cins = [w[0] for w in ws], [w[1] for w in ws]
    solver.gvins_optimization_batch(probs, 20)
    solver.outlier_culling(probs, cins)
    res = solver.marginalize(probs, 1, resident=True)
    up = solver.marginalize([copy.deepcopy(p) for p in probs], 1)
    for a, b, p in zip(res, up, probs):
        assert a["m"] == b["m"] and a["r"] == b["r"]
        for key in ("block_type", "block_node", "x0", "J0", "e0", "Hp", "bp"):
            assert np.array_equal(a[key], b[key]), key
        compare(a, oa.ba_marginalize(olib, copy.deepcopy(p), 1), tol_sqrt=1e-8)


def test_argument_errors_leave_the_handle_usable(olib, solver):
    from ic_gvins_b200 import IcgError
    prob, cin, _ = windows(olib, [5])[0]
    solver.gvins_optimization_batch([prob], 20)
    bad = []
    c = dict(cin, lm_ref_node=cin["lm_ref_node"].copy())
    c["lm_ref_node"][prob["f_lm"][0]] += 1  # f_ref != lm_ref_node[f_lm]
    bad.append(([prob], [c]))
    c = dict(cin, lm_ref_pos=cin["lm_ref_pos"].copy())
    c["lm_ref_pos"][0] = 99  # outside [0, factors]
    bad.append(([prob], [c]))
    bad.append(([prob], [dict(cin, f_kp=None)]))  # required array NULL
    bad.append(([prob, prob], [cin, cin]))  # n_windows != uploaded count
    for p, c in bad:
        with pytest.raises(IcgError, match="code -1"):
            solver.outlier_culling(p, c)
    s2 = type(solver)(max_windows=1, max_K=10, max_L=300, max_F=2700)
    try:
        s2.shard_export(0, 2)  # rank 0 of a two-rank landmark-shard group (nothing connected or run): a sharded handle
        with pytest.raises(IcgError, match="code -4"):
            s2.outlier_culling([prob], [cin])
    finally:
        s2.close()
    q = copy.deepcopy(prob)
    q["f_active"][:] = 1
    info = solver.gvins_optimization_batch([q], 20)[0]
    assert info["pass2"]["iterations"] > 0
    assert solver.outlier_culling([q], [cin])[0]["counts"][0] > 0


SRC = r'''
#include <cstdio>
#include <vector>
#include "ic_gvins_b200/host/icg_shims.hpp"
static std::vector<double> rd(FILE *f) {
    long long n = 0;
    if (fread(&n, 8, 1, f) != 1) throw std::runtime_error("short input");
    std::vector<double> v((size_t) n);
    if (n && fread(v.data(), 8, (size_t) n, f) != (size_t) n) throw std::runtime_error("short input");
    return v;
}
static void wr(FILE *f, const std::vector<double> &v) {
    long long n = (long long) v.size();
    fwrite(&n, 8, 1, f);
    if (n) fwrite(v.data(), 8, (size_t) n, f);
}
template <typename T, typename U> static std::vector<T> as(const std::vector<U> &v) { return std::vector<T>(v.begin(), v.end()); }
int main(int argc, char **argv) {
    try {
        FILE *in = fopen(argv[1], "rb"), *out = fopen(argv[2], "wb");
        if (!in || !out) return 2;
        std::vector<double> dim = rd(in), pose = rd(in), ext = rd(in), rho = rd(in), flm = rd(in), fref = rd(in), fobs = rd(in), fact = rd(in),
                            fkp = rd(in), lkp = rd(in), lnode = rd(in), lpos = rd(in), cam = rd(in);
        const int K = (int) dim[0], L = (int) dim[1], F = (int) dim[2];
        std::vector<int32_t> f_lm = as<int32_t>(flm), f_ref = as<int32_t>(fref), f_obs = as<int32_t>(fobs), ln = as<int32_t>(lnode), lp = as<int32_t>(lpos);
        std::vector<uint8_t> f_active = as<uint8_t>(fact);
        std::vector<float> f_kp = as<float>(fkp), l_kp = as<float>(lkp);
        std::vector<double> mix((size_t) 9 * K, 0.0), fc((size_t) 14 * F, 0.0);
        icg_ba_problem p{};
        p.K = K, p.L = L, p.F = F, p.pose = pose.data(), p.mix = mix.data(), p.ext = ext.data(), p.invdepth = rho.data(), p.ext_const = 1, p.td_const = 1;
        p.f_lm = f_lm.data(), p.f_ref = f_ref.data(), p.f_obs = f_obs.data(), p.f_const = fc.data(), p.f_active = f_active.data(), p.reproj_std = 1.5 / 787.0;
        icg_ba_cull_input c{};
        c.cam.fx = cam[0], c.cam.fy = cam[1], c.cam.cx = cam[2], c.cam.cy = cam[3], c.reprojection_error_std = 1.5, c.estimate_extrinsic = 1;
        c.R_bc[0] = c.R_bc[4] = c.R_bc[8] = 1.0;
        c.f_kp = f_kp.data(), c.lm_ref_kp = l_kp.data(), c.lm_ref_node = ln.data(), c.lm_ref_pos = lp.data();
        icg_b200::WindowSolver solver(K, L, F);
        icg_b200::WindowSolver::Culling r = solver.outlierCulling(p, c, false);
        wr(out, std::vector<double>(r.out.counts, r.out.counts + 5));
        wr(out, as<double>(r.f_outlier)), wr(out, as<double>(r.lm_outlier)), wr(out, as<double>(f_active)), wr(out, r.lm_pos), wr(out, r.cam_pose);
        fclose(in), fclose(out);
        return 0;
    } catch (const std::exception &e) {
        fprintf(stderr, "shim test: %s\n", e.what());
        return 1;
    }
}
'''


@pytest.mark.skipif(shutil.which("g++") is None, reason="g++ not available")
def test_cpp_shim_outlier_culling():
    from tests.test_shims_gpu import _rd, _wr
    prob, cin = cc.hand_window()
    o = co.outlier_culling(copy.deepcopy(prob), cin)
    lib = os.path.join(ROOT, "ic_gvins_b200", "libicgvins_b200.so")
    with tempfile.TemporaryDirectory() as td:
        cpp, exe, fin, fout = (os.path.join(td, x) for x in ("cull.cpp", "cull", "in.bin", "out.bin"))
        open(cpp, "w").write(SRC)
        r = subprocess.run(["g++", "-std=c++17", "-O1", "-Wall", "-I", ROOT, cpp, "-o", exe, lib, "-Wl,-rpath," + os.path.dirname(lib)], capture_output=True, text=True)
        assert r.returncode == 0, r.stderr
        with open(fin, "wb") as fh:
            for a in ([prob["K"], prob["L"], prob["F"]], prob["pose"], prob["ext"], prob["invdepth"], prob["f_lm"], prob["f_ref"], prob["f_obs"], prob["f_active"],
                      cin["f_kp"], cin["lm_ref_kp"], cin["lm_ref_node"], cin["lm_ref_pos"], cin["cam"][:4]):
                _wr(fh, a)
        r = subprocess.run([exe, fin, fout], capture_output=True, text=True, timeout=300)
        assert r.returncode == 0, (r.returncode, r.stderr)
        with open(fout, "rb") as fh:
            counts, fo, lo, act, pos, cp = (_rd(fh) for _ in range(6))
    assert list(counts.astype(int)) == cc.EXPECT_COUNTS
    assert np.array_equal(fo.astype(np.uint8), o["f_outlier"]) and np.array_equal(lo.astype(np.uint8), o["lm_outlier"])
    assert np.array_equal(act.astype(np.uint8), o["f_active"])
    assert np.abs(pos - o["lm_pos"].ravel()).max() <= 1e-12 * np.abs(o["lm_pos"]).max()
    assert np.abs(cp - o["cam_pose"].ravel()).max() <= 1e-12 * max(1.0, np.abs(o["cam_pose"]).max())
