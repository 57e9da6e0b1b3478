"""GPU parity tests (run with `-m gpu` on the B200 box): the sm_100a path, called through the C ABI, against
(a) the reference's own CUDA kernels (recorded runs, tests/golden/reference), (b) the CPU oracle and (c) the committed
golden fixtures.

Tolerances (BASELINE.json north_star): 1e-4 relative on residual sums / normal-equation coefficients,
1e-5 m / 1e-5 rad on poses; counts are integers and must match exactly unless noted.
"""
import copy
import os

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

REL = 1e-4
POSE_T, POSE_R = 1e-5, 1e-5
GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def rel(a, b):
    a, b = np.asarray(a, np.float64), np.asarray(b, np.float64)
    return float(np.max(np.abs(a - b)) / (np.max(np.abs(b)) + 1e-30))


@pytest.fixture(scope="module")
def mods():
    import torch
    assert torch.cuda.is_available()
    from badslam_b200 import scene as S
    from badslam_b200.direct_ba import DirectBA
    from oracle import cpu_oracle, ref_cuda
    return S, DirectBA, cpu_oracle, ref_cuda


def test_pose_coefficients_three_way(mods, small_scene):
    S, DirectBA, O, R = mods
    sc = small_scene
    ba, ref, orc = DirectBA.from_scene(sc), R.reference(sc), O.Oracle(sc)
    for k in range(sc.cfg.num_keyframes):
        pc = ba.AccumulatePoseEstimationCoeffs(k, sc.poses_init[k])
        H, b, cnt, cost = ref.pose_coeffs(k, sc.poses_init[k])
        st = orc.pose_coeffs(k)
        # counters: exact against the reference's debug counter and the oracle's stage counters
        assert pc.n_assoc + pc.n_photo == cnt
        assert (pc.n_pair, pc.n_inimg, pc.n_depthok, pc.n_assoc, pc.n_photo) == (st.n_pair, st.n_inimg, st.n_depthok, st.n_assoc, st.n_photo)
        assert pc.n_pair >= pc.n_inimg >= pc.n_depthok >= pc.n_assoc >= pc.n_photo
        # normal equations and residual sums: 1e-4 relative to the reference
        assert rel(pc.H[:], H) < REL and rel(pc.b[:], b) < REL
        assert abs(pc.cost_depth + pc.cost_desc1 - cost) < REL * cost
        # and the CPU oracle agrees with both (its texture filter is an emulation: slightly looser on b)
        assert rel(pc.H[:], st.H[:]) < REL and rel(pc.b[:], st.b[:]) < 3 * REL
        # (the Tukey cost 1 - (1 - q^2)^3 cancels in fp32 for small residuals; -use_fast_math vs libm differ there)
        assert abs(pc.cost_depth - st.cost_depth) < 5 * REL * max(st.cost_depth, 1.0)
        assert abs(pc.cost_desc1 - st.cost_desc1) < 3 * REL * st.cost_desc1
        assert abs(pc.cost_desc2 - st.cost_desc2) < 3 * REL * st.cost_desc2


@pytest.mark.parametrize("use_depth,use_desc", [(True, False), (False, True)])
def test_single_residual_type(mods, tiny_scene, use_depth, use_desc):
    S, DirectBA, O, R = mods
    sc = tiny_scene
    ba = DirectBA.from_scene(sc, use_depth_residuals=use_depth, use_descriptor_residuals=use_desc)
    ref = R.reference(sc, use_depth, use_desc)
    for k in range(sc.cfg.num_keyframes):
        pc = ba.AccumulatePoseEstimationCoeffs(k, sc.poses_init[k])
        H, b, cnt, cost = ref.pose_coeffs(k, sc.poses_init[k])
        assert rel(pc.H[:], H) < REL and rel(pc.b[:], b) < REL
        expect = (pc.n_assoc if use_depth else 0) + (pc.n_photo if use_desc else 0)
        assert expect == cnt
    ba.UpdateSurfelActivation(); ref.update_activation()
    ba.OptimizeGeometryIteration(); ref.optimize_geometry_iteration()
    a, b_ = R.same_sample(ba.GetSurfelsHost(), ref.surfels())
    d = np.max(np.abs(a[:3] - b_[:3]), axis=0)
    if use_depth:
        assert d.max() < 2e-6
    else:
        # photometric-only position updates are ill-conditioned for low-texture surfels (H00 ~ 1e-6 regulariser,
        # kernel_opt_geometry.cu:292-295): round-off differences are amplified for a handful of surfels
        assert np.mean(d) < 2e-6 and (d > 2e-6).mean() < 0.1 and d.max() < 2e-3
    assert np.array_equal(a[3].view(np.uint32), b_[3].view(np.uint32))
    dd = np.abs(a[6:8] - b_[6:8])
    assert dd.max() < (2e-3 if use_depth else 5.0) and dd.mean() < (1e-4 if use_depth else 5e-3)


def test_estimate_frame_pose(mods, small_scene):
    S, DirectBA, O, R = mods
    sc = small_scene
    ba, ref, orc = DirectBA.from_scene(sc), R.reference(sc), O.Oracle(sc)
    for k in range(sc.cfg.num_keyframes):
        pp, ip, cp = ba.EstimateFramePose(None, sc.poses_init[k], k)
        pr, ir, cr = ref.estimate_frame_pose(k, sc.poses_init[k])
        po, io, co = orc.estimate_frame_pose(k)
        dt, dr = S.pose_error(pp, pr)
        assert dt < POSE_T and dr < POSE_R, (k, dt, dr)
        assert ip == ir and cp == cr
        dt, dr = S.pose_error(po, pr)      # the oracle is pinned by the reference as well
        assert dt < POSE_T and dr < POSE_R, (k, dt, dr)
    # EstimateFramePose does not change the stored keyframe pose (direct_ba.h:122-129 returns the estimate)
    assert np.allclose(ba.keyframes()[0].global_T_frame(), sc.poses_init[0])


def test_activation_and_geometry(mods, small_scene):
    S, DirectBA, O, R = mods
    sc = small_scene
    ba, ref, orc = DirectBA.from_scene(sc), R.reference(sc), O.Oracle(sc)
    # make keyframe 1 inactive and 2 covisible-active to exercise the activation rules
    for obj_set in (lambda k, a: ba.keyframes()[k].SetActivation(a), ref.set_activation):
        obj_set(1, 2)
        obj_set(2, 1)
    orc.activation[1], orc.activation[2] = 2, 1
    ba.UpdateSurfelActivation(); ref.update_activation(); orc.update_activation()
    fa, fr, fo = ba.GetActiveHost(), ref.active(), orc.active[:sc.num_surfels]
    assert R.identical(fa, fr) and R.identical(fo, fr)
    assert 0 < fa.sum() <= sc.num_surfels
    ba.OptimizeGeometryIteration(); ref.optimize_geometry_iteration(); orc.optimize_geometry_iteration()
    a, b_, c = ba.GetSurfelsHost(), ref.surfels(), orc.surfels[:8, :sc.num_surfels]
    assert np.array_equal(a[4:6].view(np.uint32), sc.surfels[4:6, :sc.num_surfels].view(np.uint32))   # radius / colour untouched
    (a, b_), (c, _), (s0, _) = (R.same_sample(x, b_) for x in (a, c, sc.surfels[:8, :sc.num_surfels]))
    assert np.max(np.abs(a[:3] - b_[:3])) < 2e-6                      # positions (m)
    assert (a[3].view(np.uint32) != b_[3].view(np.uint32)).sum() == 0  # packed normals
    assert np.max(np.abs(a[6:8] - b_[6:8])) < 2e-3                    # descriptors (range +-180)
    assert np.max(np.abs(c[:3] - b_[:3])) < 5e-4 and (c[3].view(np.uint32) != b_[3].view(np.uint32)).mean() < 1e-3
    moved = np.abs(b_[:3] - s0[:3]).max()
    assert moved > 1e-4      # the step did something


def test_bundle_adjustment_against_reference(mods, small_scene):
    S, DirectBA, O, R = mods
    sc = small_scene
    K = sc.cfg.num_keyframes
    ba, ref, ref2 = DirectBA.from_scene(sc), R.reference(sc), R.reference(sc)
    ro = ba.BundleAdjustment(None, False, False, False, True, True, 3, 3)
    rr = ref.bundle_adjust(True, True, 3, 3)
    rr2 = ref2.bundle_adjust(True, True, 3, 3)
    assert ro.iterations_done == rr.iterations_done == 3
    # a keyframe whose last update sits at the 1e-6 convergence threshold may take one Gauss-Newton iteration more or
    # less (the reference's float atomics make its own count vary from run to run)
    assert abs(ro.pose_iterations_total - rr.pose_iterations_total) <= 2
    ours_pairs = ro.depth_residual_count + ro.descriptor_residual_count // 2
    assert abs(ours_pairs - rr.n_count) <= max(2, 1e-5 * rr.n_count)      # association flips near thresholds
    # cost at the start of the LAST iteration's pose step: the inputs already differ by two iterations of round-off, the
    # Tukey cost 1 - (1 - q^2)^3 cancels in fp32 for the small residuals of a converged scene (see the three-way test), and ONE
    # pair whose association flips at a threshold moves the sum by up to 100 / 6 (a saturated Tukey residual) -- 2 % of this
    # converged scene's total of ~800 (seen once in ~10 hardware runs: 1.56).  The cost at a FIXED state is compared to 1e-4 in
    # test_pose_coefficients_three_way; here the bound is the reference's own run-to-run difference plus that allowance.
    flips = abs(ours_pairs - rr.n_count) + abs(ro.pose_iterations_total - rr.pose_iterations_total) + 1
    assert abs(ro.cost - rr.cost) < 5 * REL * rr.cost + 3 * abs(rr.cost - rr2.cost) + (100.0 / 6.0) * flips, (ro.cost, rr.cost, rr2.cost)
    self_noise = max(max(S.pose_error(ref.pose(k), ref2.pose(k))) for k in range(K))
    for k in range(K):
        dt, dr = S.pose_error(ba.keyframes()[k].global_T_frame(), ref.pose(k))
        assert dt < POSE_T + 2 * self_noise and dr < POSE_R + 2 * self_noise, (k, dt, dr, self_noise)
    assert np.array_equal(ba.GetKeyframeStates()[1], ref.activation())
    a, b_ = R.same_sample(ba.GetSurfelsHost(), ref.surfels())
    assert np.mean(np.abs(a[:3] - b_[:3])) < 1e-6


def test_windowed_bundle_adjustment(mods, small_scene):
    """active_keyframe_window != all keyframes: fixed activation + all surfels active (direct_ba_alternating.cc:354-372,444-446)."""
    S, DirectBA, O, R = mods
    sc = small_scene
    ba, ref = DirectBA.from_scene(sc), R.reference(sc)
    ro = ba.BundleAdjustment(None, False, False, False, True, True, 2, 2, active_keyframe_window_start=1, active_keyframe_window_end=3)
    rr = ref.bundle_adjust(True, True, 2, 2, window_start=1, window_end=3)
    # (a keyframe whose last update sits at the 1e-6 convergence threshold may take one Gauss-Newton iteration more or less: the
    #  reference's float atomics make its own count vary from run to run, see test_bundle_adjustment_against_reference)
    assert abs(ro.pose_iterations_total - rr.pose_iterations_total) <= 2
    assert ba.GetActiveHost().all() and ref.active().all()
    ref2 = R.reference(sc)
    ref2.bundle_adjust(True, True, 2, 2, window_start=1, window_end=3)
    self_noise = max(max(S.pose_error(ref.pose(k), ref2.pose(k))) for k in range(sc.cfg.num_keyframes))
    for k in range(sc.cfg.num_keyframes):
        dt, dr = S.pose_error(ba.keyframes()[k].global_T_frame(), ref.pose(k))
        assert dt < POSE_T + 2 * self_noise and dr < POSE_R + 2 * self_noise, (k, dt, dr, self_noise)


def test_edge_cases(mods, tiny_scene):
    S, DirectBA, O, R = mods
    # ragged sizes: 1 surfel, tile-size +- 1, exactly one tile
    for n in (1, 255, 256, 257, 1023, 1025):
        sc = copy.copy(tiny_scene)
        sc.num_surfels = n
        ba, orc = DirectBA.from_scene(sc), O.Oracle(sc)
        pc, st = ba.AccumulatePoseEstimationCoeffs(0, sc.poses_init[0]), orc.pose_coeffs(0)
        assert (pc.n_inimg, pc.n_assoc, pc.n_photo) == (st.n_inimg, st.n_assoc, st.n_photo), n
        if st.n_assoc:
            assert rel(pc.H[:], st.H[:]) < 2 * REL
        r = ba.BundleAdjustment(None, False, False, False, True, True, 1, 2)
        assert r.iterations_done >= 1
    # empty surfel set: H = 0 -> x = 0 -> converged immediately (direct_ba_alternating.cc:147-150)
    sc = copy.copy(tiny_scene)
    sc.num_surfels = 0
    ba = DirectBA.from_scene(sc)
    p, it, conv = ba.EstimateFramePose(None, sc.poses_init[0], 0)
    assert np.allclose(p, sc.poses_init[0]) and it == 1 and conv
    assert ba.BundleAdjustment(None, False, False, False, True, True, 1, 3).converged
    # surfels behind the cameras: nothing associates, nothing is activated, geometry is a no-op
    sc = copy.copy(tiny_scene)
    sc.surfels = tiny_scene.surfels.copy()
    sc.surfels[2] = -5.0
    ba = DirectBA.from_scene(sc)
    pc = ba.AccumulatePoseEstimationCoeffs(0, sc.poses_init[0])
    assert pc.n_inimg == 0 and not any(pc.H[:])
    ba.UpdateSurfelActivation()
    assert not ba.GetActiveHost().any()
    before = ba.GetSurfelsHost()
    ba.OptimizeGeometryIteration()
    assert np.array_equal(before.view(np.uint32), ba.GetSurfelsHost().view(np.uint32))
    # invalid options fail loudly instead of silently doing something else
    from badslam_b200._lib import BadBAError
    with pytest.raises(BadBAError):   # gauge keyframe out of range / more keyframes than pcg_max_keyframes (direct_ba_pcg.cc:232)
        ba.BundleAdjustment(None, False, False, False, True, True, 1, 1, use_pcg=True, pcg_gauge_keyframe=sc.cfg.num_keyframes)
    with pytest.raises(BadBAError):
        ba.BundleAdjustment(None, False, False, False, True, True, 1, 1, use_pcg=True, pcg_max_keyframes=1)


def test_host_buffer_entry_points(mods, tiny_scene):
    """The *_host path (library-owned device memory) gives the same results as caller-owned device buffers."""
    S, DirectBA, O, R = mods
    sc = tiny_scene
    a, b_ = DirectBA.from_scene(sc), DirectBA.from_scene(sc, host_owned=True)
    ra = a.BundleAdjustment(None, False, False, False, True, True, 2, 2)
    b_.UpdateKeyframeHost(1, sc.depth[1], sc.normals[1], sc.radius[1], sc.color[1])
    rb = b_.BundleAdjustment(None, False, False, False, True, True, 2, 2)
    assert ra.depth_residual_count == rb.depth_residual_count and ra.pose_iterations_total == rb.pose_iterations_total
    pa, pb = a.GetKeyframeStates()[0], b_.GetKeyframeStates()[0]
    assert max(max(S.pose_error(pa[k], pb[k])) for k in range(sc.cfg.num_keyframes)) < 2e-6
    assert np.max(np.abs(a.GetSurfelsHost()[:3] - b_.GetSurfelsHost()[:3])) < 2e-6


@pytest.mark.parametrize("name,tag,use_depth,use_desc", [("cfg1", "", True, True), ("tiny", "", True, True),
                                                          ("tiny", "_depth_only", True, False), ("tiny", "_desc_only", False, True)])
def test_against_golden_fixtures(mods, name, tag, use_depth, use_desc):
    S, DirectBA, O, R = mods
    path = os.path.join(GOLDEN, f"{name}{tag}.npz")
    if not os.path.exists(path):
        pytest.skip("golden fixture not generated yet (tools/make_golden.py)")
    g = np.load(path)
    sc = S.make_scene(S.config_by_name(name))
    assert abs(float(np.sum(sc.surfels[:3, :sc.num_surfels].astype(np.float64))) - float(g["surfel_checksum"])) < 1e-6
    ba = DirectBA.from_scene(sc, use_depth_residuals=use_depth, use_descriptor_residuals=use_desc)
    for k in range(sc.cfg.num_keyframes):
        pc = ba.AccumulatePoseEstimationCoeffs(k, sc.poses_init[k])
        assert rel(pc.H[:], g["pose_H"][k]) < REL and rel(pc.b[:], g["pose_b"][k]) < REL
        assert (pc.n_assoc if use_depth else 0) + (pc.n_photo if use_desc else 0) == g["pose_count"][k]
        p, it, conv = ba.EstimateFramePose(None, sc.poses_init[k], k)
        dt, dr = S.pose_error(p, g["efp_pose"][k])
        assert dt < POSE_T and dr < POSE_R and it == g["efp_iterations"][k]
    ba.UpdateSurfelActivation()
    assert np.array_equal(np.packbits(ba.GetActiveHost()), g["activation_flags"])
    ba.OptimizeGeometryIteration()
    rows = ba.GetSurfelsHost()[[0, 1, 2, 3, 6, 7]]
    d = np.max(np.abs(rows[:3] - g["geometry_rows"][:3]), axis=0)
    if use_depth:
        assert d.max() < 2e-6
    else:   # photometric-only position updates are ill-conditioned for low-texture surfels (see test_single_residual_type)
        assert np.mean(d) < 2e-6 and (d > 2e-6).mean() < 0.1 and d.max() < 2e-3
    assert (rows[3].view(np.uint32) != g["geometry_rows"][3].view(np.uint32)).sum() == 0


def test_full_size_properties(mods):
    """cfg2 (20 keyframes x 200k surfels, 640x480): size-independent properties + oracle spot checks."""
    S, DirectBA, O, R = mods
    sc = S.make_scene(S.config_by_name("cfg2"))
    ba, orc = DirectBA.from_scene(sc), O.Oracle(sc)
    for k in (0, 7, 19):
        pc, st = ba.AccumulatePoseEstimationCoeffs(k, sc.poses_init[k]), orc.pose_coeffs(k)
        assert (pc.n_inimg, pc.n_depthok, pc.n_assoc, pc.n_photo) == (st.n_inimg, st.n_depthok, st.n_assoc, st.n_photo)
        assert rel(pc.H[:], st.H[:]) < REL
        # idempotence: the accumulators are consumed and re-armed by every call
        pc2 = ba.AccumulatePoseEstimationCoeffs(k, sc.poses_init[k])
        assert rel(pc2.H[:], pc.H[:]) < 1e-6 and pc2.n_assoc == pc.n_assoc
        # H is symmetric positive semi-definite
        H = np.zeros((6, 6))
        H[np.triu_indices(6)] = pc.H[:]
        H = H + H.T - np.diag(H.diagonal())
        assert np.linalg.eigvalsh(H).min() > -1e-3 * np.abs(H).max()
    r1 = ba.BundleAdjustment(None, False, False, False, True, True, 1, 1)
    r5 = ba.BundleAdjustment(None, False, False, False, True, True, 4, 4)
    assert r5.cost < r1.cost                      # BA lowers the robust cost
    assert r5.depth_residual_count > 0.3 * 20 * sc.num_surfels
    poses, act = ba.GetKeyframeStates()
    assert np.allclose(np.linalg.norm(poses[:, :4], axis=1), 1.0, atol=1e-5)     # unit quaternions
    errs = [S.pose_error(poses[k], sc.poses_true[k])[0] for k in range(20)]
    errs0 = [S.pose_error(sc.poses_init[k], sc.poses_true[k])[0] for k in range(20)]
    assert np.mean(errs) < np.mean(errs0)


def _distorted_scene(S, name):
    """Depth-distorted raw depth (true a / cfactor != the model's zeros) and perturbed camera estimates."""
    import dataclasses
    sc = S.make_scene(dataclasses.replace(S.config_by_name(name), depth_a=0.03, cfactor=0.005))
    sc.depth_K = (np.asarray(sc.depth_K, np.float32) * np.float32([1.003, 0.998, 1.002, 0.997])).astype(np.float32)
    sc.color_K = (np.asarray(sc.color_K, np.float32) * np.float32([0.998, 1.002, 1.001, 0.999])).astype(np.float32)
    return sc


@pytest.mark.parametrize("opt_depth,opt_color", [(True, True), (True, False), (False, True)])
def test_intrinsics_step_three_way(mods, opt_depth, opt_color):
    """OptimizeIntrinsicsCUDA (kernel_opt_intrinsics.cc:39-281): one step, ours vs the reference kernels vs the oracle."""
    S, DirectBA, O, R = mods
    sc = _distorted_scene(S, "small")
    ba, ref, ref2, orc = DirectBA.from_scene(sc), R.reference(sc), R.reference(sc), O.Oracle(sc)
    # a non-zero deformation model, so that the d/da and d/dcfactor terms (kernel_opt_intrinsics.cu:97-113) are exercised
    a_init = 0.02
    cf_init = (np.random.default_rng(5).standard_normal(sc.cfactor.shape) * 0.003).astype(np.float32)
    ba.SetA(a_init); ba.SetCFactorBuffer(cf_init)
    ref.set_depth_params(a_init, cf_init)
    ref2.set_depth_params(a_init, cf_init)
    orc.model.a = a_init; orc.cfactor[:] = cf_init
    for _ in range(2):
        ba.OptimizeIntrinsics(opt_depth, opt_color)
        ref.optimize_intrinsics(opt_depth, opt_color)
        ref2.optimize_intrinsics(opt_depth, opt_color)
        orc.optimize_intrinsics(opt_depth, opt_color)
    d0, c0, a0 = ba._intrinsics()
    d1, c1, a1 = ref.intrinsics()
    # `a` is the weakly constrained unknown of this step (hence the reference's prior, kernel_opt_intrinsics.cc:146-155): the
    # reference's own run-to-run difference (unordered fp32 atomics on the per-cell terms) sets the scale of what can be asked
    a_noise = abs(a1 - ref2.intrinsics()[2])
    d2, c2, a2 = np.array(orc.model.depth_K[:], np.float32), np.array(orc.model.color_K[:], np.float32), orc.model.a
    # the UPDATE (new - old, up to ~0.5 px here) must agree to 1e-4 relative of the parameter scale + fp32 atomics noise
    tol_d = REL * np.abs(d1) + 1e-3
    assert np.all(np.abs(d0 - d1) < tol_d), (d0, d1)
    assert np.all(np.abs(c0 - c1) < REL * np.abs(c1) + 1e-3), (c0, c1)
    assert abs(a0 - a1) < 1e-5 + 5 * a_noise, (a0, a1, a_noise)
    assert np.all(np.abs(d0 - d2) < tol_d) and np.all(np.abs(c0 - c2) < REL * np.abs(c2) + 1e-3) and abs(a0 - a2) < 1e-4
    cf0, cf1 = ba.cfactor_buffer(), ref.cfactor()
    cs0, cf1 = R.same_sample(cf0, cf1)
    if opt_depth:
        assert np.any(d0 != np.asarray(sc.depth_K, np.float32)) and np.any(cf0 != cf_init) and abs(a0 - a_init) > 1e-3
        assert (cs0 != 0).sum() == (cf1 != 0).sum()
        assert np.abs(cs0 - cf1).max() < 1e-4 and np.abs(cf0 - orc.cfactor).max() < 1e-3
    else:
        assert np.array_equal(d0, np.asarray(sc.depth_K, np.float32)) and np.array_equal(cf0, cf_init) and a0 == np.float32(a_init)
    if not opt_color:
        assert np.array_equal(c0, np.asarray(sc.color_K, np.float32))


def test_bundle_adjustment_with_intrinsics(mods):
    """BundleAdjustment(optimize_depth_intrinsics, optimize_color_intrinsics) against the reference's alternation."""
    S, DirectBA, O, R = mods
    sc = _distorted_scene(S, "small")
    K = sc.cfg.num_keyframes
    ba, ref, ref2 = DirectBA.from_scene(sc), R.reference(sc), R.reference(sc)
    ro = ba.BundleAdjustment(None, True, True, False, True, True, 3, 3)
    rr = ref.bundle_adjust(True, True, 3, 3, optimize_depth_intrinsics=True, optimize_color_intrinsics=True)
    ref2.bundle_adjust(True, True, 3, 3, optimize_depth_intrinsics=True, optimize_color_intrinsics=True)
    assert ro.iterations_done == rr.iterations_done == 3 and ro.ms_intrinsics_optimization > 0
    d0, c0, a0 = ba._intrinsics()
    d1, c1, a1 = ref.intrinsics()
    d2, c2, a2 = ref2.intrinsics()
    noise_d, noise_c = np.abs(d1 - d2).max(), np.abs(c1 - c2).max()
    assert np.abs(d0 - d1).max() < 5e-3 + 3 * noise_d and np.abs(c0 - c1).max() < 5e-3 + 3 * noise_c, (d0, d1, c0, c1)
    # `a` is only weakly constrained (hence the reference's prior, kernel_opt_intrinsics.cc:146-155): the alternation
    # amplifies round-off differences in it (the single steps agree to 1e-6, test_intrinsics_step_three_way)
    assert abs(a0 - a1) < 0.02 + 3 * abs(a1 - a2)
    self_noise = max(max(S.pose_error(ref.pose(k), ref2.pose(k))) for k in range(K))
    for k in range(K):
        dt, dr = S.pose_error(ba.keyframes()[k].global_T_frame(), ref.pose(k))
        assert dt < 2e-4 + 3 * self_noise and dr < 2e-4 + 3 * self_noise, (k, dt, dr, self_noise)
    assert np.any(d0 != np.asarray(sc.depth_K, np.float32)) and np.any(c0 != np.asarray(sc.color_K, np.float32))


def _segments(K, n, stride, total):
    segs = {"pose": (0, 6 * (K - 1)), "surfel": (6 * (K - 1), 6 * (K - 1) + stride * n)}
    if total > segs["surfel"][1]:
        segs["intr"] = (segs["surfel"][1], total)
    return segs


@pytest.mark.parametrize("name,distort,intr,use_desc,a_init", [("tiny", False, False, True, 0.0), ("tiny", False, False, False, 0.0),
                                                                ("small", True, True, True, 0.02)])
def test_pcg_building_blocks_three_way(mods, name, distort, intr, use_desc, a_init):
    """PCGInit / PCGInit2 / PCGStep1 (kernel_pcg.cu:179-1037): r, M, p0, g = J^T W J p0, alpha_n, alpha_d."""
    import dataclasses
    S, DirectBA, O, R = mods
    cfg = S.config_by_name(name)
    if distort:
        cfg = dataclasses.replace(cfg, depth_a=0.03, cfactor=0.005)
    sc = S.make_scene(cfg)
    K, n = cfg.num_keyframes, sc.num_surfels
    ba = DirectBA.from_scene(sc, use_descriptor_residuals=use_desc)
    ref, orc = R.reference(sc, True, use_desc), O.Oracle(sc, True, use_desc)
    if a_init:
        cf = (np.random.default_rng(5).standard_normal(sc.cfactor.shape) * 0.003).astype(np.float32)
        ba.SetA(a_init); ba.SetCFactorBuffer(cf)
        ref.set_depth_params(a_init, cf)
        orc.model.a = a_init; orc.cfactor[:] = cf
    kw = dict(optimize_depth_intrinsics=intr, optimize_color_intrinsics=intr, gauge_keyframe=1)
    ours, theirs, cpu = ba.PCGDebug(**kw), ref.pcg_debug(**kw), orc.pcg_debug(**kw)
    size = len(ours[0])
    assert size == R.shape_of(theirs[0])[0] == len(cpu[0]) == 6 * (K - 1) + (3 if use_desc else 1) * n + ((5 + sc.cfactor.size + 4) if intr else 0)
    for idx, what in enumerate(("r", "M", "p", "g")):
        at, t = R.same_sample(np.arange(size), theirs[idx])     # (the entries the reference's vector was recorded at)
        for seg, (lo, hi) in _segments(K, n, 3 if use_desc else 1, size).items():
            sel = at[(at >= lo) & (at < hi)]
            ts = t[(at >= lo) & (at < hi)]
            scale = np.abs(ts).max()
            d = np.abs(ours[idx][sel].astype(np.float64) - ts).max() / scale
            assert d < 5e-5, (what, seg, d)      # vs the reference's kernels: fp32 summation order only
            if seg != "surfel":                  # oracle (software texture filter, threshold flips): aggregated entries only
                dc = np.abs(cpu[idx][sel].astype(np.float64) - ts).max() / scale
                assert dc < 1e-3, (what, seg, dc)
    assert np.all(np.abs(ours[4] - theirs[4]) < 1e-5 * np.abs(theirs[4]))
    assert np.all(np.abs(cpu[4] - theirs[4]) < 1e-4 * np.abs(theirs[4]))
    assert np.all(ours[1] >= 0) and ours[4][1] > 0   # M = diag(J^T W J) >= 0, p^T A p > 0


def test_pcg_bundle_adjustment_against_reference(mods, small_scene):
    """use_pcg = true (direct_ba_pcg.cc:43-819).  A few inner steps: tight parity.  Full solve: CG in fp32 is not reproducible
    across summation orders (loss of conjugacy amplifies 1e-7 differences), so the bar is the quality of the solution."""
    S, DirectBA, O, R = mods
    sc = small_scene
    K = sc.cfg.num_keyframes
    # (1) 4 inner steps per outer iteration
    ba, ref, ref2 = DirectBA.from_scene(sc), R.reference(sc), R.reference(sc)
    ro = ba.BundleAdjustment(None, False, False, False, True, True, 2, 2, use_pcg=True, pcg_max_inner_iterations=4, pcg_gauge_keyframe=2)
    rr = ref.bundle_adjust_pcg(min_iterations=2, max_iterations=2, max_inner_iterations=4, gauge_keyframe=2)
    ref2.bundle_adjust_pcg(min_iterations=2, max_iterations=2, max_inner_iterations=4, gauge_keyframe=2)
    assert ro.iterations_done == rr.iterations_done == 2 and ro.pcg_inner_iterations_total == rr.inner_iterations_total == 8
    assert abs(ro.pcg_last_r_norm - rr.last_r_norm) < 1e-3 * rr.last_r_norm
    noise = max(max(S.pose_error(ref.pose(k), ref2.pose(k))) for k in range(K))
    pa = ba.GetKeyframeStates()[0]
    assert np.array_equal(pa[2], sc.poses_init[2])     # the gauge keyframe does not move
    for k in range(K):
        dt, dr = S.pose_error(pa[k], ref.pose(k))
        assert dt < 1e-5 + 3 * noise and dr < 1e-5 + 3 * noise, (k, dt, dr, noise)
    a, b_ = R.same_sample(ba.GetSurfelsHost(), ref.surfels())
    assert np.abs(a[:3] - b_[:3]).max() < 1e-4 and np.abs(a[:3] - b_[:3]).mean() < 1e-6      # 8 fp32 CG steps
    assert (a[3].view(np.uint32) != b_[3].view(np.uint32)).mean() < 1e-4   # second normals update sees 1e-6-different positions
    # (2) full solves: same quality as the reference
    ba, ref = DirectBA.from_scene(sc), R.reference(sc)
    ro = ba.BundleAdjustment(None, False, False, False, True, True, 3, 3, use_pcg=True, pcg_gauge_keyframe=0)
    rr = ref.bundle_adjust_pcg(min_iterations=3, max_iterations=3, gauge_keyframe=0)
    def rel_err(poses):
        e = []
        for k in range(1, K):
            x = O.se3_mul(O.se3_inverse(poses[0]), poses[k])
            y = O.se3_mul(O.se3_inverse(sc.poses_true[0]), sc.poses_true[k])
            e.append(max(S.pose_error(x, y)))
        return max(e)
    e0, eo, er = rel_err(sc.poses_init), rel_err(ba.GetKeyframeStates()[0]), rel_err(ref.poses())
    assert eo < 0.5 * e0 and eo < 1.5 * er + 1e-4, (e0, eo, er)
    assert ro.kernel_launches < rr.kernel_launches / 3


def test_intrinsics_and_pcg_against_golden_fixture(mods):
    """The CUDA path against tests/golden/tiny_intrinsics_pcg.npz (outputs of the reference's kernels, tools/make_golden.py)."""
    from test_oracle_pcg import distorted_scene
    S, DirectBA, O, R = mods
    g = np.load(os.path.join(GOLDEN, "tiny_intrinsics_pcg.npz"))
    sc, a_init, cf_init = distorted_scene("tiny")
    K, n = sc.cfg.num_keyframes, sc.num_surfels

    def fresh():
        ba = DirectBA.from_scene(sc)
        ba.SetA(a_init); ba.SetCFactorBuffer(cf_init)
        return ba

    ba = fresh()
    for step in range(2):
        ba.OptimizeIntrinsics(True, True)
        d, c, a = ba._intrinsics()
        assert np.abs(d - g[f"intr{step}_depth_K"]).max() < 1e-3 and np.abs(c - g[f"intr{step}_color_K"]).max() < 1e-3
        assert abs(a - float(g[f"intr{step}_a"])) < 1e-5 and np.abs(ba.cfactor_buffer() - g[f"intr{step}_cfactor"]).max() < 1e-5
    for intr in (False, True):
        tag = "pcgi" if intr else "pcg"
        ba = fresh()
        r, M, p, gv, scal = ba.PCGDebug(optimize_depth_intrinsics=intr, optimize_color_intrinsics=intr, gauge_keyframe=1)
        lo, hi = 6 * (K - 1), 6 * (K - 1) + 3 * n
        for nm, v in (("r", r), ("M", M), ("p", p), ("g", gv)):
            ref = g[f"{tag}_{nm}_pose"]
            assert np.abs(v[:lo] - ref).max() < 5e-5 * np.abs(ref).max(), (tag, nm)
            assert abs(v[lo:hi].astype(np.float64).sum() - float(g[f"{tag}_{nm}_surfel_sum"])) < 1e-5 * float(g[f"{tag}_{nm}_surfel_abs"])
            if intr:
                ref = g[f"{tag}_{nm}_intr"]
                assert np.abs(v[hi:] - ref).max() < 5e-5 * np.abs(ref).max(), (tag, nm)
        assert np.all(np.abs(scal - g[f"{tag}_scalars"]) < 1e-5 * np.abs(g[f"{tag}_scalars"]))
        res = ba.BundleAdjustment(None, intr, intr, False, True, True, 2, 2, use_pcg=True, pcg_max_inner_iterations=4, pcg_gauge_keyframe=1)
        assert res.pcg_inner_iterations_total == 8
        noise = max(max(S.pose_error(g[f"{tag}_ba_poses"][k], g[f"{tag}_ba_poses_rerun"][k])) for k in range(K))
        pa = ba.GetKeyframeStates()[0]
        for k in range(K):
            dt, dr = S.pose_error(pa[k], g[f"{tag}_ba_poses"][k])
            assert dt < 2e-5 + 3 * noise and dr < 2e-5 + 3 * noise, (tag, k, dt, dr, noise)
        assert abs(res.pcg_last_r_norm - float(g[f"{tag}_ba_r_norm"])) < 5e-3 * float(g[f"{tag}_ba_r_norm"])
        if intr:
            d, c, a = ba._intrinsics()
            assert np.abs(d - g["pcgi_ba_depth_K"]).max() < 2e-3 and np.abs(c - g["pcgi_ba_color_K"]).max() < 2e-3
            assert abs(a - float(g["pcgi_ba_a"])) < 5e-4


def test_progress_function_stops_the_iterations(mods, tiny_scene):
    """direct_ba_alternating.cc:346-348 / direct_ba_pcg.cc:174-176: progress_function(iteration) is asked before every iteration;
    false ends the optimisation there."""
    S, DirectBA, O, R = mods
    for use_pcg in (False, True):
        ba = DirectBA.from_scene(tiny_scene)
        seen = []
        r = ba.BundleAdjustment(None, False, False, False, True, True, 5, 5, use_pcg=use_pcg, pcg_gauge_keyframe=0,
                                progress_function=lambda it: (seen.append(it), it < 2)[1])
        assert seen == [0, 1, 2] and r.iterations_done == 2
        r = ba.BundleAdjustment(None, False, False, False, True, True, 2, 2, use_pcg=use_pcg, pcg_gauge_keyframe=0)
        assert r.iterations_done == 2


def test_residual_types_can_be_switched_at_runtime(mods, tiny_scene):
    """DirectBA::SetUseDepthResiduals / SetUseDescriptorResiduals (direct_ba.h:317-328; main.cc:853 turns the descriptor residuals
    off for the final BA): the same numbers as a backend created with those flags."""
    S, DirectBA, O, R = mods
    sc = tiny_scene
    ba = DirectBA.from_scene(sc)
    assert ba.use_depth_residuals() and ba.use_descriptor_residuals()
    for use_depth, use_desc in ((True, False), (False, True), (True, True)):
        ba.SetUseDepthResiduals(True)          # keep one type enabled while switching the other
        ba.SetUseDescriptorResiduals(use_desc)
        ba.SetUseDepthResiduals(use_depth)
        assert (ba.use_depth_residuals(), ba.use_descriptor_residuals()) == (use_depth, use_desc)
        fixed = DirectBA.from_scene(sc, use_depth_residuals=use_depth, use_descriptor_residuals=use_desc)
        for k in range(sc.cfg.num_keyframes):
            p, q = ba.AccumulatePoseEstimationCoeffs(k, sc.poses_init[k]), fixed.AccumulatePoseEstimationCoeffs(k, sc.poses_init[k])
            assert (p.n_assoc, p.n_photo) == (q.n_assoc, q.n_photo)
            assert rel(p.H[:], q.H[:]) < 1e-6 and rel(p.b[:], q.b[:]) < 1e-6
    from badslam_b200._lib import BadBAError
    ba.SetUseDescriptorResiduals(False)
    with pytest.raises(BadBAError):
        ba.SetUseDepthResiduals(False)


def test_estimate_frame_pose_from_buffers_equals_the_keyframe_form(mods, small_scene):
    """DirectBA::EstimateFramePose takes a frame's buffers (direct_ba.h:122-129); a frame that is not a keyframe must be
    tracked exactly like the same images stored as a keyframe, and must leave no trace in the backend."""
    import torch
    S, DirectBA, O, R = mods
    sc = small_scene
    K = sc.cfg.num_keyframes
    ba = DirectBA.from_scene(sc, max_keyframes=K + 1)
    k = 2
    up = lambda a: torch.from_numpy(np.ascontiguousarray(a).view(np.int16)).cuda()
    depth, normals = up(sc.depth[k]), up(sc.normals[k])
    color = torch.from_numpy(np.ascontiguousarray(sc.color[k])).cuda()
    want, it_w, conv_w = ba.EstimateFramePose(None, sc.poses_init[k], k)
    got, it_g, conv_g = ba.EstimateFramePoseFromBuffers(None, sc.poses_init[k], depth, normals, color)
    assert (it_g, conv_g) == (it_w, conv_w)
    assert np.max(np.abs(got - want)) < 1e-6
    assert ba._lib.bba_keyframe_count(ba._h) == K
    # the backend is unchanged: the keyframe form gives the same answer again, BA still runs
    again, _, _ = ba.EstimateFramePose(None, sc.poses_init[k], k)
    assert np.max(np.abs(again - want)) < 1e-6
    assert ba.BundleAdjustment(None, False, False, False, True, True, 1, 1).iterations_done == 1
    # no free keyframe slot: a loud error, not a silent reallocation
    full = DirectBA.from_scene(sc, max_keyframes=K)
    from badslam_b200._lib import BadBAError
    with pytest.raises(BadBAError):
        full.EstimateFramePoseFromBuffers(None, sc.poses_init[k], depth, normals, color)


def test_calibration_files_round_trip_through_the_backend(mods, tiny_scene, tmp_path):
    """SaveCalibration / LoadCalibration (io.cc:570-700) on the real backend state."""
    S, DirectBA, O, R = mods
    from badslam_b200 import calibration_io as IO
    from badslam_b200.direct_ba import PinholeCamera4f
    sc = tiny_scene
    src, dst = DirectBA.from_scene(sc), DirectBA.from_scene(sc)
    src.SetDepthCamera(PinholeCamera4f(sc.cfg.width, sc.cfg.height, np.asarray(sc.depth_K) * np.float32(1.01)))
    src.SetA(0.0275)
    cf = (1e-3 * np.random.default_rng(1).random(src.cfactor_buffer().shape)).astype(np.float32)
    src.SetCFactorBuffer(cf)
    base = str(tmp_path / "calib")
    assert IO.SaveCalibration(src, base) and IO.LoadCalibration(dst, base)
    assert np.allclose(dst.depth_camera().parameters, src.depth_camera().parameters, rtol=1e-5)
    assert np.allclose(dst.color_camera().parameters, src.color_camera().parameters, rtol=1e-5)
    assert abs(dst.a() - 0.0275) < 1e-7 and np.allclose(dst.cfactor_buffer(), cf, rtol=1e-7)
