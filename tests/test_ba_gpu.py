"""GPU parity tests for path B (factor evaluation + LM/Schur window solve) through the C ABI, against the CPU oracle.

Bar (north_star): pose / landmark solution within 1e-6 relative of the reference path.  The reference path here is the
oracle restatement (Ceres is absent: parity unpinned at that boundary, stated in DESIGN.md)."""
import copy

import numpy as np
import pytest

from datagen import synth_ba
from tests import oracle_api as oa

pytestmark = pytest.mark.gpu
REL = 1e-6


@pytest.fixture(scope="module")
def olib(oracle):
    oa.declare_ba(oracle)
    return oracle


@pytest.fixture(scope="module")
def solver():
    from ic_gvins_b200.ba import WindowSolver
    s = WindowSolver(max_windows=4, max_K=10, max_L=300, max_F=2700, max_gnss=16, max_marg_r=64)
    yield s
    s.close()


def make(olib, **kw):
    return synth_ba.make_window(lambda *a: oa.preintegrate(olib, *a), **kw)


def rel_err(a, b):
    a, b = np.asarray(a), np.asarray(b)
    return float(np.abs(a - b).max() / max(1e-300, np.abs(b).max()))


def test_preintegration_host_matches_oracle(olib):
    """B3 (host side in both implementations): blob equality to 1e-12 relative."""
    from ic_gvins_b200.ba import imu_preintegrate
    rng = np.random.default_rng(5)
    imu = synth_ba.imu_samples(0.0, 0.5, 200.0, rng, np.zeros(3), np.zeros(3))
    p, v, _, psi = synth_ba.trajectory(0.0)
    st = np.concatenate([p, synth_ba.q_yaw(psi), v, [1e-4, -2e-4, 3e-4], [1e-3, 2e-3, -1e-3]])
    blob_o, pn, end_o = oa.preintegrate(olib, st, synth_ba.IEWN, synth_ba.GRAVITY, synth_ba.NOISE5, imu)
    blob_g, end_g = imu_preintegrate(st, synth_ba.IEWN, synth_ba.GRAVITY, synth_ba.NOISE5, imu)
    assert np.abs(blob_g[:27] - blob_o[:27]).max() <= 1e-12 * max(1.0, np.abs(blob_o[:27]).max())
    assert rel_err(blob_g[27:252], blob_o[27:252]) <= 1e-12
    assert rel_err(blob_g[252:477], blob_o[252:477]) <= 1e-10
    assert rel_err(end_g, end_o) <= 1e-13


def test_reprojection_evaluate_matches_oracle(olib, solver):
    prob, _ = make(olib, K=10, L=60, seed=11)
    pose = prob["pose"].reshape(-1, 7)
    for f in (0, 3, 50, 111):
        c = prob["f_const"][14 * f:14 * f + 14]
        i, j, l = prob["f_ref"][f], prob["f_obs"][f], prob["f_lm"][f]
        args = (pose[i], pose[j], prob["ext"][:7], prob["invdepth"][l], prob["ext"][7], c, prob["reproj_std"])
        r_o, J_o = oa.reproj_eval(olib, *args)
        r_g, J_g = solver.reproj_evaluate(*args)
        assert rel_err(r_g, r_o) <= 1e-12
        for a, b in zip(J_g, J_o):
            assert np.abs(a - b).max() <= 1e-11 * max(1.0, np.abs(b).max())


def test_imu_evaluate_matches_oracle(olib, solver):
    prob, _ = make(olib, K=6, L=30, seed=12)
    pose, mix = prob["pose"].reshape(-1, 7), prob["mix"].reshape(-1, 9)
    off, pn = prob["pn_off"], prob["pn"].reshape(-1, 4)
    for k in (0, 2, 4):
        blob = prob["imu_blob"][480 * k:480 * (k + 1)]
        r_o, J_o = oa.imu_eval(olib, blob, pn[off[k]:off[k + 1]], pose[k], mix[k], pose[k + 1], mix[k + 1])
        r_g, J_g = solver.imu_evaluate(blob, pose[k], mix[k], pose[k + 1], mix[k + 1])
        assert np.abs(r_g - r_o).max() <= 1e-7 * max(1.0, np.abs(r_o).max())  # whitening amplifies 1e-16 by cond(cov) ~ 1e8
        for a, b in zip(J_g, J_o):
            assert np.abs(a - b).max() <= 1e-7 * max(1.0, np.abs(b).max())


CASES = {
    "cfg3_const_ext": dict(K=10, L=300, seed=2024, const_ext=True),
    "cfg3_marg_prior": dict(K=10, L=300, seed=2025, with_marg=True),
    "small_full_vis": dict(K=5, L=40, seed=7, full_visibility=True, const_ext=True),
    "no_huber": dict(K=8, L=120, seed=9, const_ext=True, huber=False),
    # ImuPosePriorFactor + ImuMixPriorFactor inside the solve (imu_pose_prior_factor.h:42-68, imu_mix_prior_factor.h:40-75; ic_gvins.cc:1880-1887)
    "cfg3_first_window_priors": dict(K=10, L=300, seed=2026, with_priors=True),
    "priors_and_marg": dict(K=6, L=60, seed=41, with_priors=True, with_marg=True, pixel_noise=1.5),
    # windows without landmarks: addReprojectionParameters returns early (ic_gvins.cc:1698) and Ceres solves IMU + GNSS + priors
    "camera_only": dict(K=10, L=0, seed=4),
}


@pytest.mark.parametrize("name", list(CASES))
@pytest.mark.parametrize("iters", [5, 20])
def test_window_solve_matches_oracle(olib, solver, name, iters):
    kw = dict(CASES[name])
    const_ext = kw.pop("const_ext", False)
    hub = kw.pop("huber", True)
    prob, _ = make(olib, **kw)
    if const_ext:
        prob["ext_const"], prob["td_const"] = 1, 1
    if not hub:
        prob["reproj_huber"], prob["gnss_huber"] = 0, 0
    po, pg = copy.deepcopy(prob), copy.deepcopy(prob)
    so = oa.ba_solve(olib, po, iters)
    sg = solver.solve(pg, iters)[0]
    assert sg["iterations"] == so["iterations"] and sg["num_successful_steps"] == so["num_successful_steps"]
    assert sg["termination"] == so["termination"]
    assert abs(sg["initial_cost"] - so["initial_cost"]) <= 1e-9 * so["initial_cost"]
    assert abs(sg["final_cost"] - so["final_cost"]) <= 1e-7 * so["final_cost"]
    _compare_solution(pg, po)  # velocity / bias groups have very different magnitudes: compared per group


def test_batched_windows_are_independent(olib, solver):
    """Four different windows in one call == the same windows solved one by one (bitwise)."""
    probs = [make(olib, K=10, L=100 + 20 * i, seed=30 + i)[0] for i in range(4)]
    for p in probs:
        p["ext_const"], p["td_const"] = 1, 1
    single = []
    for p in probs:
        q = copy.deepcopy(p)
        solver.solve(q, 8)
        single.append(q)
    batch = copy.deepcopy(probs)
    solver.solve(batch, 8)
    for a, b in zip(batch, single):
        for key in ("pose", "mix", "invdepth", "ext"):
            assert np.array_equal(a[key], b[key]), key


def test_two_pass_protocol_matches_oracle(olib, solver):
    """GVINS::gvinsOptimization: 5 iterations, chi2 culling (GNSS re-weighting + reprojection removal), 15 iterations."""
    prob, _ = make(olib, K=10, L=300, seed=77)
    prob["ext_const"], prob["td_const"] = 1, 1
    fc = prob["f_const"].reshape(-1, 14)
    fc[10, 3] += 0.2      # gross visual outliers
    fc[500, 4] -= 0.15
    prob["gnss_blh"][3:6] += np.array([1.0, -0.8, 0.5])  # a GNSS outlier on the second fix
    pg, po = copy.deepcopy(prob), copy.deepcopy(prob)
    info = solver.gvins_optimization(pg, 20)
    # the same protocol on the oracle
    po["gnss_huber"] = 1
    oa.ba_solve(olib, po, 5)
    rc, gc = oa.ba_residual_costs(olib, po)
    std = po["gnss_std"].reshape(-1, 3)
    for g in range(po["n_gnss"]):
        if 2 * gc[g] > 7.815:
            std[g] *= np.sqrt(2 * gc[g] / 7.815)
    po["gnss_std"] = std.reshape(-1)
    out = (2 * rc > 5.991)
    po["f_active"][out] = 0
    po["gnss_huber"] = 0
    oa.ba_solve(olib, po, 15)
    assert info["reproj_removed"] == int(out.sum()) and out[10] and out[500]
    assert np.array_equal(pg["f_active"], po["f_active"])
    assert rel_err(pg["gnss_std"], po["gnss_std"]) <= 1e-9
    for key in ("pose", "invdepth"):
        assert rel_err(pg[key], po[key]) <= REL, key


def test_capacity_errors(solver, olib):
    from ic_gvins_b200 import IcgError
    prob, _ = make(olib, K=10, L=40, seed=1)
    prob["K"] = 11
    with pytest.raises(IcgError):
        solver.solve(prob, 2)


def test_device_resident_two_pass_equals_host_protocol(olib, solver):
    """icg_ba_gvins_optimization (culling on the device, no host round trip) == the host-driven protocol, bitwise."""
    probs = []
    for i in range(3):
        p, _ = make(olib, K=10, L=200, seed=90 + i)
        p["ext_const"], p["td_const"] = 1, 1
        fc = p["f_const"].reshape(-1, 14)
        fc[7 + i, 3] += 0.2
        p["gnss_blh"][3:6] += np.array([1.0, -0.8, 0.5])
        probs.append(p)
    host = copy.deepcopy(probs)
    infos_h = [solver.gvins_optimization(p, 20) for p in host]
    dev = copy.deepcopy(probs)
    infos_d = solver.gvins_optimization_batch(dev, 20)
    for a, b, ia, ib in zip(dev, host, infos_d, infos_h):
        assert ia["reproj_removed"] == ib["reproj_removed"] >= 1 and ia["gnss_reweighted"] == ib["gnss_reweighted"] >= 1
        assert np.array_equal(a["f_active"], b["f_active"])
        assert ia["pass1"]["iterations"] == ib["pass1"]["iterations"] and ia["pass2"]["iterations"] == ib["pass2"]["iterations"]
        for key in ("pose", "mix", "invdepth", "ext", "gnss_std"):
            assert np.array_equal(a[key], b[key]), key


def _compare_solution(pg, po, rel=REL):
    for key in ("pose", "mix", "invdepth", "ext"):
        a, b = pg[key], po[key]
        if a.size == 0:
            continue
        if key == "mix":
            a, b = a.reshape(-1, 9), b.reshape(-1, 9)
            for sl in (slice(0, 3), slice(3, 6), slice(6, 9)):
                assert rel_err(a[:, sl], b[:, sl]) <= rel, (key, sl)
        else:
            assert rel_err(a, b) <= rel, key


def test_initialization_solve_shape_matches_oracle(olib):
    """GVINS::gvinsInitializationOptimization (IG/ic_gvins.cc:698-718): states + GNSS (Huber) + IMU factors + ImuErrorFactor + first-window
    priors, no landmarks, max_num_iterations = 50.  (SPARSE_NORMAL_CHOLESKY there: same normal equations, different factorisation.)"""
    from ic_gvins_b200.ba import WindowSolver
    s = WindowSolver(max_windows=1, max_K=4, max_L=0, max_F=0, max_gnss=8, max_marg_r=0)
    try:
        for K, seed in ((2, 3), (3, 5), (4, 8)):
            prob, _ = make(olib, K=K, L=0, seed=seed, with_priors=True, gnss_every=1)
            pg, po = copy.deepcopy(prob), copy.deepcopy(prob)
            so = oa.ba_solve(olib, po, 50)
            sg = s.solve(pg, 50)[0]
            assert sg["iterations"] == so["iterations"] and sg["termination"] == so["termination"] == 1
            assert abs(sg["final_cost"] - so["final_cost"]) <= 1e-7 * so["final_cost"]
            _compare_solution(pg, po)
    finally:
        s.close()


@pytest.fixture(scope="module")
def solver_cfg4():
    from ic_gvins_b200.ba import WindowSolver
    s = WindowSolver(max_windows=2, max_K=20, max_L=2000, max_F=12000, max_gnss=16, max_marg_r=64)
    yield s
    s.close()


CFG4 = {
    "free_ext_td": dict(K=20, L=2000, seed=2027),
    "marg_prior": dict(K=20, L=2000, seed=2028, with_marg=True),
    "const_ext_priors": dict(K=20, L=2000, seed=2029, with_priors=True, const_ext=True),
}


@pytest.mark.parametrize("name", list(CFG4))
def test_cfg4_window_solve_matches_oracle(olib, solver_cfg4, name):
    """BASELINE.json cfg 4 on one GPU: 20-KF / 2000-landmark window (n = 307 camera-side columns: the reduced system no longer fits one
    CTA's shared memory -- a different solve kernel than cfg 3).  Solution within 1e-6 relative of the oracle, same LM trajectory."""
    kw = dict(CFG4[name])
    const_ext = kw.pop("const_ext", False)
    prob, _ = make(olib, **kw)
    if const_ext:
        prob["ext_const"], prob["td_const"] = 1, 1
    assert prob["F"] <= 12000
    po, pg = copy.deepcopy(prob), copy.deepcopy(prob)
    so = oa.ba_solve(olib, po, 20)
    sg = solver_cfg4.solve(pg, 20)[0]
    assert sg["iterations"] == so["iterations"] and sg["num_successful_steps"] == so["num_successful_steps"]
    assert sg["termination"] == so["termination"]
    assert abs(sg["initial_cost"] - so["initial_cost"]) <= 1e-9 * so["initial_cost"]
    assert abs(sg["final_cost"] - so["final_cost"]) <= 1e-7 * so["final_cost"]
    _compare_solution(pg, po)


def test_cfg4_two_pass_protocol_matches_oracle(olib, solver_cfg4):
    prob, _ = make(olib, K=20, L=2000, seed=2030)
    fc = prob["f_const"].reshape(-1, 14)
    fc[10, 3] += 0.2
    fc[5000, 4] -= 0.15
    prob["gnss_blh"][3:6] += np.array([1.0, -0.8, 0.5])
    pg, po = copy.deepcopy(prob), copy.deepcopy(prob)
    info = solver_cfg4.gvins_optimization_batch([pg], 20)[0]
    po["gnss_huber"] = 1
    s1 = oa.ba_solve(olib, po, 5)
    rc, gc = oa.ba_residual_costs(olib, po)
    std = po["gnss_std"].reshape(-1, 3)
    for g in range(po["n_gnss"]):
        if 2 * gc[g] > 7.815:
            std[g] *= np.sqrt(2 * gc[g] / 7.815)
    po["gnss_std"] = std.reshape(-1)
    out = (2 * rc > 5.991)
    po["f_active"][out] = 0
    po["gnss_huber"] = 0
    s2 = oa.ba_solve(olib, po, 15)
    assert info["pass1"]["iterations"] == s1["iterations"] and info["pass2"]["iterations"] == s2["iterations"]
    assert info["reproj_removed"] == int(out.sum()) and out[10] and out[5000]
    assert np.array_equal(pg["f_active"], po["f_active"])
    _compare_solution(pg, po)


def test_restart_resolves_the_uploaded_problem(olib, solver):
    """icg_ba_run_gvins(restart = 1) after a completed two-pass call must re-solve the problems AS UPLOADED (factor activity and GNSS
    std restored), not the culled / re-weighted ones: two restarted runs give bit-identical results and the same culling counts."""
    prob, _ = make(olib, K=10, L=200, seed=91)
    prob["ext_const"], prob["td_const"] = 1, 1
    prob["f_const"].reshape(-1, 14)[7, 3] += 0.2
    prob["gnss_blh"][3:6] += np.array([1.0, -0.8, 0.5])
    ref = copy.deepcopy(prob)
    info0 = solver.gvins_optimization_batch([ref], 20)[0]   # upload + run + end (writes culled data into the staging buffers)
    assert info0["reproj_removed"] >= 1 and info0["gnss_reweighted"] >= 1
    again = copy.deepcopy(prob)
    solver.upload([again])
    solver.run_gvins(20, restart=False)
    a = solver.download()
    first = {k: again[k].copy() for k in ("pose", "mix", "invdepth")}
    solver.run_gvins(20, restart=True)
    b = solver.download()
    for k in first:
        assert np.array_equal(first[k], again[k]) and np.array_equal(first[k], ref[k]), k
    assert a[0]["iterations"] == b[0]["iterations"] == info0["pass2"]["iterations"]
    assert abs(a[0]["final_cost"] - b[0]["final_cost"]) == 0.0


def _solve_sharded_in_process(probs, world, iters, K, two_pass=False):
    """`world` solver handles in THIS process (all on cuda:0), connected over the peer-memory transport, each driven by its own host
    thread -- the code path of one-process-per-GPU landmark sharding (ba_split.cuh), runnable on a single GPU."""
    import threading
    from ic_gvins_b200.ba import WindowSolver, shard_window
    n = len(probs)
    shards = [[shard_window(p, r, world) for p in probs] for r in range(world)]
    solvers = [WindowSolver(max_windows=n, max_K=K, max_L=max(1, max(s["L"] for s in shards[r])), max_F=max(1, max(s["F"] for s in shards[r])),
                            max_gnss=16, max_marg_r=64) for r in range(world)]
    try:
        blobs = [solvers[r].shard_export(r, world) for r in range(world)]
        for sv in solvers:
            sv.shard_connect(blobs)
        out, errs = [None] * world, []

        def run(r):
            try:
                out[r] = solvers[r].gvins_optimization_batch(shards[r], iters) if two_pass else solvers[r].solve(shards[r], iters)
            except Exception as e:  # noqa: BLE001
                errs.append((r, repr(e)))
        th = [threading.Thread(target=run, args=(r,)) for r in range(world)]
        for t in th:
            t.start()
        for t in th:
            t.join(300)
        assert not errs, errs
    finally:
        for sv in solvers:
            sv.close()
    merged = []
    for w, p in enumerate(probs):
        full = copy.deepcopy(p)
        for r in range(world):
            sh = shards[r][w]
            full["invdepth"][sh["lm_lo"]:sh["lm_hi"]] = sh["invdepth"]
            full["f_active"][sh["f_index"]] = sh["f_active"]
            for key in ("pose", "mix", "ext", "gnss_std"):
                assert np.array_equal(sh[key], shards[0][w][key]), (w, r, key, "camera-side blocks differ between shards")
        for key in ("pose", "mix", "ext", "gnss_std"):
            full[key] = shards[0][w][key]
        merged.append(full)
    return merged, out


@pytest.mark.parametrize("world,K,L,nwin", [(2, 10, 300, 3), (3, 10, 300, 4), (2, 20, 2000, 2)])
def test_landmark_sharded_p2p_in_process_matches_oracle(olib, world, K, L, nwin):
    """Landmark shards over the peer-memory transport (window w owned by rank w mod world) == the oracle's solve of the whole window:
    same LM trajectory, solution within 1e-6.  Every rank ends with bit-identical camera-side blocks."""
    probs = []
    for w in range(nwin):
        p, _ = make(olib, K=K, L=L, seed=3000 + 10 * K + w, with_marg=(w % 2 == 1), with_priors=(w == 2))
        if w % 3 == 1:
            p["ext_const"], p["td_const"] = 1, 1
        probs.append(p)
    merged, out = _solve_sharded_in_process(probs, world, 20, K)
    for w, p in enumerate(probs):
        po = copy.deepcopy(p)
        so = oa.ba_solve(olib, po, 20)
        for r in range(world):
            sg = out[r][w]
            assert sg["iterations"] == so["iterations"] and sg["num_successful_steps"] == so["num_successful_steps"], (w, r, sg, so)
            assert sg["termination"] == so["termination"]
            assert abs(sg["final_cost"] - so["final_cost"]) <= 1e-7 * so["final_cost"]
        _compare_solution(merged[w], po)


def test_landmark_sharded_two_pass_in_process(olib):
    """gvinsOptimization (5 + chi2 culling + 15) on landmark shards: culling is local to the shard that owns the factor, GNSS re-weighting
    is replicated; merged result == the single-handle two-pass result (identical LM decisions; solution within 1e-8: the shard partials
    are summed in a different order than the single-handle Gram products, and 20 LM iterations on the weakly observed camera-IMU
    extrinsic carry that rounding to ~1e-9 relative)."""
    from ic_gvins_b200.ba import WindowSolver
    probs = []
    for w in range(2):
        p, _ = make(olib, K=10, L=300, seed=3100 + w)
        p["f_const"].reshape(-1, 14)[10 + w, 3] += 0.2
        p["gnss_blh"][3:6] += np.array([1.0, -0.8, 0.5])
        probs.append(p)
    merged, out = _solve_sharded_in_process(probs, 2, 20, 10, two_pass=True)
    single = copy.deepcopy(probs)
    s = WindowSolver(max_windows=2, max_K=10, max_L=300, max_F=2700, max_gnss=16, max_marg_r=64)
    try:
        info = s.gvins_optimization_batch(single, 20)
    finally:
        s.close()
    for w in range(2):
        assert sum(out[r][w]["reproj_removed"] for r in range(2)) == info[w]["reproj_removed"] >= 1
        assert out[0][w]["gnss_reweighted"] == info[w]["gnss_reweighted"] >= 1
        assert out[0][w]["pass2"]["iterations"] == info[w]["pass2"]["iterations"]
        assert np.array_equal(merged[w]["f_active"], single[w]["f_active"])
        _compare_solution(merged[w], single[w], rel=1e-8)


def test_preintegration_normal_matches_oracle(olib, solver):
    """PreintegrationNormal (`iswithearth: false`, preintegration_normal.cc): host propagation, device factor evaluation and a window solve."""
    from ic_gvins_b200.ba import imu_preintegrate
    rng = np.random.default_rng(6)
    imu = synth_ba.imu_samples(0.0, 0.5, 200.0, rng, np.zeros(3), np.zeros(3), earth=False)
    p, v, _, psi = synth_ba.trajectory(0.0)
    st = np.concatenate([p, synth_ba.q_yaw(psi), v, [1e-4, -2e-4, 3e-4], [1e-3, 2e-3, -1e-3]])
    blob_o, _, end_o = oa.preintegrate(olib, st, None, synth_ba.GRAVITY, synth_ba.NOISE5, imu)
    blob_g, end_g = imu_preintegrate(st, None, synth_ba.GRAVITY, synth_ba.NOISE5, imu)
    assert blob_g[477] == blob_o[477] == 1.0
    assert np.abs(blob_g[:27] - blob_o[:27]).max() <= 1e-12 * max(1.0, np.abs(blob_o[:27]).max())
    assert rel_err(blob_g[27:252], blob_o[27:252]) <= 1e-12 and rel_err(blob_g[252:477], blob_o[252:477]) <= 1e-10
    assert rel_err(end_g, end_o) <= 1e-13
    prob, _ = make(olib, K=6, L=60, seed=77, earth=False)
    pose, mix = prob["pose"].reshape(-1, 7), prob["mix"].reshape(-1, 9)
    for k in (0, 3):
        blob = prob["imu_blob"][480 * k:480 * (k + 1)]
        r_o, J_o = oa.imu_eval(olib, blob, np.zeros((0, 4)), pose[k], mix[k], pose[k + 1], mix[k + 1])
        r_g, J_g = solver.imu_evaluate(blob, pose[k], mix[k], pose[k + 1], mix[k + 1])
        assert np.abs(r_g - r_o).max() <= 1e-7 * max(1.0, np.abs(r_o).max())
        for a, b in zip(J_g, J_o):
            assert np.abs(a - b).max() <= 1e-7 * max(1.0, np.abs(b).max())
    po, pg = copy.deepcopy(prob), copy.deepcopy(prob)
    so = oa.ba_solve(olib, po, 20)
    sg = solver.solve(pg, 20)[0]
    assert sg["iterations"] == so["iterations"] and sg["num_successful_steps"] == so["num_successful_steps"]
    assert abs(sg["final_cost"] - so["final_cost"]) <= 1e-7 * so["final_cost"]
    _compare_solution(pg, po)


def test_small_factor_seams_match_oracle(olib, solver):
    """CostFunction::Evaluate seams for GnssFactor, ImuPosePriorFactor, ImuMixPriorFactor, ImuErrorFactor, MarginalizationFactor."""
    import math
    prob, _ = make(olib, K=6, L=60, seed=41, with_priors=True, with_marg=True)
    pose, mix = prob["pose"].reshape(-1, 7), prob["mix"].reshape(-1, 9)
    # GNSS
    g = 1
    nd = int(prob["gnss_node"][g])
    r_o, J_o = np.zeros(3), np.zeros((3, 7))
    a = [pose[nd].copy(), prob["gnss_blh"][3 * g:3 * g + 3].copy(), prob["gnss_std"][3 * g:3 * g + 3].copy(), np.array(prob["lever"], np.float64)]
    olib.icgo_gnss_eval(oa._p(a[0]), oa._p(a[1]), oa._p(a[2]), oa._p(a[3]), oa._p(r_o), oa._p(J_o))
    r_g, J_g = solver.gnss_evaluate(*a)
    assert np.abs(r_g - r_o).max() <= 1e-12 * max(1.0, np.abs(r_o).max()) and np.abs(J_g - J_o).max() <= 1e-12 * np.abs(J_o).max()
    # pose prior
    r_o, J_o = np.zeros(6), np.zeros((6, 7))
    a = [pose[0].copy(), np.asarray(prob["pose_prior"], float).copy(), np.asarray(prob["pose_prior_std"], float).copy()]
    olib.icgo_pose_prior_eval(oa._p(a[0]), oa._p(a[1]), oa._p(a[2]), oa._p(r_o), oa._p(J_o))
    r_g, J_g = solver.pose_prior_evaluate(*a)
    assert np.abs(r_g - r_o).max() <= 1e-11 * max(1.0, np.abs(r_o).max()) and np.abs(J_g - J_o).max() <= 1e-11 * np.abs(J_o).max()
    # mix prior / bias-magnitude factor: closed forms (imu_mix_prior_factor.h:40-75, imu_error_factor.h:45-91)
    sd = np.asarray(prob["mix_prior_std"], float)
    r_g, J_g = solver.mix_prior_evaluate(mix[0], prob["mix_prior"], sd)
    assert np.allclose(r_g, (mix[0] - prob["mix_prior"]) / sd, rtol=1e-14) and np.allclose(J_g, np.diag(1.0 / sd), rtol=1e-14)
    gb, ab = 7200 / 3600.0 * math.pi / 180.0, 2.0e4 * 1.0e-5
    r_g, J_g = solver.imu_error_evaluate(mix[5])
    assert np.allclose(r_g, np.concatenate([mix[5][3:6] / gb, mix[5][6:9] / ab]), rtol=1e-14)
    J_ref = np.zeros((6, 9))
    for q in range(3):
        J_ref[q, 3 + q], J_ref[3 + q, 6 + q] = 1.0 / gb, 1.0 / ab
    assert np.allclose(J_g, J_ref, rtol=1e-14)
    # marginalization factor vs the numpy restatement (e = e0 + J0 dx)
    from tests.test_oracle_lm_trajectory import quat_mul
    rr = prob["marg_r"]
    J0 = np.asarray(prob["marg_J0"], float).reshape(rr, rr)
    x0 = np.asarray(prob["marg_x0"], float)
    params, dx, xo = [], [], 0
    for t, ndx in zip(prob["marg_block_type"], prob["marg_block_node"]):
        if t in (0, 2):
            x = pose[ndx] if t == 0 else prob["ext"][:7]
            xl = x0[xo:xo + 7]
            dq = quat_mul(np.array([-xl[3], -xl[4], -xl[5], xl[6]]) / (xl[3:7] @ xl[3:7]), x[3:7])
            dx += list(x[:3] - xl[:3]) + list(2.0 * dq[:3] * (1.0 if dq[3] >= 0 else -1.0))
            xo += 7
        elif t == 1:
            x = mix[ndx]
            dx += list(x - x0[xo:xo + 9])
            xo += 9
        else:
            x = prob["ext"][7:8]
            dx.append(float(x[0] - x0[xo]))
            xo += 1
        params.append(np.array(x, copy=True))
    e_ref = np.asarray(prob["marg_e0"], float) + J0 @ np.array(dx)
    res, Js = solver.marg_factor_evaluate(prob["marg_block_type"], params, x0, J0, prob["marg_e0"])
    assert np.abs(res - e_ref).max() <= 1e-11 * max(1.0, np.abs(e_ref).max())
    col = 0
    for t, J in zip(prob["marg_block_type"], Js):
        l = {0: 6, 1: 9, 2: 6, 3: 1}[int(t)]
        assert np.array_equal(J[:, :l], J0[:, col:col + l]) and (J.shape[1] == l or np.all(J[:, l:] == 0))
        col += l
