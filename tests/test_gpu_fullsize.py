"""GPU parity at the sizes bench.py measures (BASELINE.json configs 2 and 3): the sm_100a path through the C ABI against the
reference's own CUDA kernels (recorded runs, tests/golden/reference) on the same seeded scene -- the tile sizes (TILE = 1024 at 3 M surfels), the
8-keyframe work groups of the pose kernel and the 13 keyframe groups of the geometry kernels only exist at these sizes.

Tolerances (BASELINE.json north_star): 1e-4 relative on normal-equation coefficients / residual sums, 1e-5 m / 1e-5 rad on
poses (+ the reference's own run-to-run noise: its float atomics are unordered); counts are integers and must match.
"""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

REL = 1e-4
POSE_T, POSE_R = 1e-5, 1e-5


def rel(a, b):
    a, b = np.asarray(a, np.float64), np.asarray(b, np.float64)
    return float(np.max(np.abs(a - b)) / (np.max(np.abs(b)) + 1e-30))


@pytest.fixture(scope="module")
def mods():
    from badslam_b200 import scene as S
    from badslam_b200.direct_ba import DirectBA
    from oracle import cpu_oracle, ref_cuda
    return S, DirectBA, cpu_oracle, ref_cuda


def check_pose_coefficients(S, ba, ref, sc, keyframes):
    for k in keyframes:
        pc = ba.AccumulatePoseEstimationCoeffs(k, sc.poses_init[k])
        H, b, cnt, cost = ref.pose_coeffs(k, sc.poses_init[k])
        assert pc.n_assoc + pc.n_photo == cnt, (k, pc.n_assoc, pc.n_photo, cnt)
        assert pc.n_pair == sc.num_surfels and pc.n_pair >= pc.n_inimg >= pc.n_depthok >= pc.n_assoc >= pc.n_photo > 0
        assert rel(pc.H[:], H) < REL and rel(pc.b[:], b) < REL, (k, rel(pc.H[:], H), rel(pc.b[:], b))
        assert abs(pc.cost_depth + pc.cost_desc1 - cost) < REL * cost, (k, pc.cost_depth + pc.cost_desc1, cost)


def check_one_ba_iteration(S, ba, ref, ref2, sc):
    """One outer iteration of the alternation (activation, normals, position / descriptor, pose of every keyframe) from the
    same state on both sides; ref2 = a second run of the reference = its own noise floor."""
    from oracle import ref_cuda as R
    K = sc.cfg.num_keyframes
    # no end-of-scheme maintenance on either side (it would delete surfels first: direct_ba_alternating.cc:313-319 runs
    # PerformBASchemeEndTasks at the start of a call with increase_ba_iteration_count = false once the counter has moved)
    ba.SetLastBAIterationCount(ba.ba_iteration_count())
    ro = ba.BundleAdjustment(None, False, False, False, True, True, 1, 1, increase_ba_iteration_count=False)
    rr = ref.bundle_adjust(True, True, 1, 1, count_residuals=2, end_tasks=False)
    ref2.bundle_adjust(True, True, 1, 1, count_residuals=False, end_tasks=False)
    # residual counts at the pose step's starting state: depth residuals and descriptor pairs separately
    assert ro.depth_residual_count == rr.n_depth_count
    assert ro.depth_residual_count + ro.descriptor_residual_count // 2 == rr.n_count
    assert abs(ro.pose_iterations_total - rr.pose_iterations_total) <= max(2, K // 50)   # (1e-6 threshold, see test_gpu_parity)
    assert abs(ro.cost - rr.cost) < 5 * REL * rr.cost
    noise = max(max(S.pose_error(ref.pose(k), ref2.pose(k))) for k in range(K))
    worst = 0.0
    for k in range(K):
        dt, dr = S.pose_error(ba.keyframes()[k].global_T_frame(), ref.pose(k))
        worst = max(worst, dt, dr)
        assert dt < POSE_T + 2 * noise and dr < POSE_R + 2 * noise, (k, dt, dr, noise)
    assert np.array_equal(ba.GetKeyframeStates()[1], ref.activation())
    # activation flags: identical; surfel rows after the geometry step: positions to 2e-6 m, packed normals identical,
    # descriptors to 2e-3 of their +-180 range (tests/test_gpu_parity.py::test_activation_and_geometry at small size)
    assert R.identical(ba.GetActiveHost(), ref.active())
    a, b_ = R.same_sample(ba.GetSurfelsHost(), ref.surfels())
    d = np.abs(a[:3] - b_[:3])
    assert d.max() < 1e-5 and (d > 2e-6).mean() < 1e-5, (d.max(), (d > 2e-6).mean())   # (2e-6 on every one of the 30 k surfels of `small`)
    assert (a[3].view(np.uint32) != b_[3].view(np.uint32)).sum() == 0
    assert np.max(np.abs(a[6:8] - b_[6:8])) < 2e-3
    print(f"{sc.cfg.name}: worst pose difference to the reference {worst:.2e} (reference run-to-run {noise:.2e}), "
          f"{ro.depth_residual_count + ro.descriptor_residual_count} residuals, GN iterations {ro.pose_iterations_total} / {rr.pose_iterations_total}")


def test_cfg2_every_keyframe_and_one_ba_iteration(mods):
    S, DirectBA, O, R = mods
    sc = S.make_scene(S.config_by_name("cfg2"))
    ba, ref, ref2 = DirectBA.from_scene(sc), R.reference(sc), R.reference(sc)
    check_pose_coefficients(S, ba, ref, sc, range(sc.cfg.num_keyframes))
    check_one_ba_iteration(S, ba, ref, ref2, sc)


def test_cfg3_spread_keyframes_and_one_ba_iteration(mods):
    """The benchmarked workload itself: 200 keyframes x 3 M surfels.  Keyframes 0, 7, 8, 63, 100, 129, 150, 191, 192, 199 sit in
    different 8-keyframe work groups of the pose kernel (first / last slot of a group, first / middle / last group)."""
    S, DirectBA, O, R = mods
    sc = S.make_scene(S.config_by_name("cfg3"))
    ba, ref = DirectBA.from_scene(sc), R.reference(sc)
    check_pose_coefficients(S, ba, ref, sc, (0, 7, 8, 63, 100, 129, 150, 191, 192, 199))
    ref2 = R.reference(sc)
    check_one_ba_iteration(S, ba, ref, ref2, sc)


# BASELINE.json configs 4 and 5 (500 keyframes / 4 M surfels with intrinsics + depth deformation; 1280x720, 400 keyframes /
# 8 M surfels).  Scene generation alone takes minutes, so these two only run when BADBA_BIG_CONFIGS=1 (tools/r2_big_configs.sh;
# the logs of the hardware runs are under profiles/bench/).  The spot check is the one of the benchmarked configuration:
# association counts, H, b and cost of four keyframes from different work groups against the reference's own kernels.
import os

big = pytest.mark.skipif(not os.environ.get("BADBA_BIG_CONFIGS"), reason="set BADBA_BIG_CONFIGS=1 (minutes of scene generation)")


@big
@pytest.mark.parametrize("name", ["cfg4", "cfg5"])
def test_big_config_spot_check(mods, name):
    import torch
    S, DirectBA, O, R = mods
    sc = S.make_scene(S.config_by_name(name))
    K = sc.cfg.num_keyframes
    ba, ref = DirectBA.from_scene(sc), R.reference(sc)
    check_pose_coefficients(S, ba, ref, sc, (0, K // 3 + 1, 2 * K // 3 + 2, K - 1))
    if name == "cfg4":
        # one intrinsics + depth-deformation step (the cfg4 flags) on both sides from the same state
        ba.OptimizeIntrinsics(True, True)
        ref.optimize_intrinsics(True, True)
        di, ci, a = ba._intrinsics()
        rdi, rci, ra = ref.intrinsics()
        # tolerances of tests/test_gpu_parity.py::test_intrinsics_step_three_way
        assert np.all(np.abs(di - rdi) < REL * np.abs(rdi) + 1e-3) and np.all(np.abs(ci - rci) < REL * np.abs(rci) + 1e-3), (di, rdi, ci, rci)
        assert abs(a - ra) < 1e-5, (a, ra)
        cf0, cf1 = R.same_sample(ba.cfactor_buffer(), ref.cfactor())
        assert np.abs(cf0 - cf1).max() < 1e-4
        # ... and two iterations of the cfg4 alternation itself (activation, geometry, poses, intrinsics + depth deformation)
        # from that state; tolerances of tests/test_gpu_parity.py::test_bundle_adjustment_with_intrinsics without the
        # second reference run (its noise floor is not measured here: 5x the fixed part instead)
        ba.SetLastBAIterationCount(ba.ba_iteration_count())
        ro = ba.BundleAdjustment(None, True, True, False, True, True, 2, 2, increase_ba_iteration_count=False)
        rr = ref.bundle_adjust(True, True, 2, 2, optimize_depth_intrinsics=True, optimize_color_intrinsics=True, count_residuals=False,
                               end_tasks=False)
        assert ro.iterations_done == rr.iterations_done == 2
        di, ci, a = ba._intrinsics()
        rdi, rci, ra = ref.intrinsics()
        assert np.abs(di - rdi).max() < 2.5e-2 and np.abs(ci - rci).max() < 2.5e-2, (di, rdi, ci, rci)
        assert abs(a - ra) < 0.1, (a, ra)
        worst = max(max(S.pose_error(ba.keyframes()[k].global_T_frame(), ref.pose(k))) for k in range(K))
        assert worst < 1e-3, worst
        print(f"cfg4 after 2 BA iterations with intrinsics: a {a:.5f} / reference {ra:.5f}, fx {di[0]:.4f} / {rdi[0]:.4f}, "
              f"worst pose difference {worst:.2e}")
    free, total = torch.cuda.mem_get_info()
    print(f"{name}: device memory in use with product + reference resident {(total - free) / 2**30:.2f} GiB")
