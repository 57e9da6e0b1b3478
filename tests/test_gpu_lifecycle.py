"""GPU parity of the end-of-BA surfel maintenance (PerformBASchemeEndTasks, direct_ba.cc:566-653): the sm_100a path through the
C ABI against the reference's own kernels (oracle/_ref) and the CPU oracle.  Deletion decisions, the compaction
permutation and the radii are integer / exact-value work: the bar is bit-exact."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def mods():
    import torch
    assert torch.cuda.is_available()
    from badslam_b200 import scene as S
    from badslam_b200.direct_ba import DirectBA
    from oracle import cpu_oracle, ref_cuda
    return S, DirectBA, cpu_oracle, ref_cuda


def perturb(sc):
    from badslam_b200.scene import displace_surfels
    return displace_surfels(sc)[0]


@pytest.mark.parametrize("name", ["tiny", "small", "cfg2"])
def test_end_tasks_three_way(mods, name):
    S, DirectBA, O, R = mods
    sc = perturb(S.make_scene(S.config_by_name(name)))
    n = sc.num_surfels
    ba, ref = DirectBA.from_scene(sc), R.reference(sc)
    d0, n0 = ba.PerformBASchemeEndTasks()
    d1 = ref.end_tasks()
    assert d0 == d1 > 0 and n0 == ref.surfels_size() == n - d0 == ba.surfels_size()
    a, b = ba.GetSurfelsHost(), ref.surfels()
    assert a.shape == R.shape_of(b) == (8, n0)
    assert R.identical(a, b)                                              # same survivors, same slots, same radii
    assert not np.any(a[0].view(np.uint32) == 0x7fffffff)
    if name != "cfg2":
        orc = O.Oracle(sc)
        assert orc.end_tasks() == d0 and orc.n == n0
        assert np.array_equal(orc.surfels[:8, :n0].view(np.uint32), a.view(np.uint32))
    # idempotent
    assert ba.PerformBASchemeEndTasks() == (0, n0)
    assert np.array_equal(ba.GetSurfelsHost().view(np.uint32), a.view(np.uint32))


def test_bundle_adjustment_end_task_schedule(mods):
    """increase_ba_iteration_count = true: end tasks after the iterations; false: before them, once per counter value
    (direct_ba_alternating.cc:313-319,725-735)."""
    S, DirectBA, O, R = mods
    sc = perturb(S.make_scene(S.config_by_name("small")))
    n = sc.num_surfels
    ba, ref = DirectBA.from_scene(sc), R.reference(sc)
    ro = ba.BundleAdjustment(None, False, False, False, True, True, 2, 2)
    rr = ref.bundle_adjust(True, True, 2, 2)
    assert ro.surfels_deleted == rr.surfels_deleted > 0 and ro.surfels_size == rr.surfels_size == n - ro.surfels_deleted
    assert ba.ba_iteration_count() == 1
    a, b = R.same_sample(ba.GetSurfelsHost(), ref.surfels())
    assert a.shape == b.shape
    # same survivors in the same slots (the two BA iterations before differ by fp32 round-off: a packed normal or a radius
    # decision may flip for a handful of surfels)
    assert (a[3].view(np.uint32) != b[3].view(np.uint32)).mean() < 1e-3 and (a[4] != b[4]).mean() < 1e-3
    assert np.array_equal(a[5].view(np.uint32), b[5].view(np.uint32))
    assert np.abs(a[:3] - b[:3]).mean() < 1e-6 and np.abs(a[:3] - b[:3]).max() < 1e-3   # (displaced surfels that survive are ill-constrained)
    # increase_ba_iteration_count = false: counters 1 != -1 -> end tasks first (nothing left to delete), then not again
    r2 = ba.BundleAdjustment(None, False, False, False, True, True, 1, 1, increase_ba_iteration_count=False)
    assert r2.surfels_deleted == 0 and ba.last_ba_iteration_count() == 1 and ba.ba_iteration_count() == 1
    ba2 = DirectBA.from_scene(sc)      # a fresh handle (counters 0 != -1) runs the end tasks before its first iteration
    r3 = ba2.BundleAdjustment(None, False, False, False, True, True, 1, 1, increase_ba_iteration_count=False)
    assert r3.surfels_deleted > 0 and ba2.surfels_size() == n - r3.surfels_deleted and ba2.last_ba_iteration_count() == 0


def test_end_tasks_against_golden_fixture(mods):
    """The CUDA path against tests/golden/tiny_end_tasks.npz (outputs of the reference's kernels)."""
    import os
    S, DirectBA, O, R = mods
    g = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "tiny_end_tasks.npz"))
    sc = perturb(S.make_scene(S.config_by_name("tiny")))
    ba = DirectBA.from_scene(sc)
    deleted, size = ba.PerformBASchemeEndTasks()
    assert deleted == int(g["deleted"]) and size == int(g["surfels_size"])
    assert np.array_equal(ba.GetSurfelsHost().view(np.uint32), g["rows"].view(np.uint32))


def _half_map(S, name):
    """The scene with only the first half of its surfels (so that many sparse cells of every keyframe are unsupported) and
    the true poses (new surfels land on the surfaces)."""
    import copy
    sc = copy.copy(S.make_scene(S.config_by_name(name)))
    sc.poses_init = sc.poses_true.copy()
    sc.num_surfels = sc.num_surfels // 2
    # room for the new surfels (capacity = row pitch of the surfel buffer; the reference creates nothing when it is exceeded)
    cells = sc.cfactor.size * sc.cfg.num_keyframes
    sc.surfels = np.pad(sc.surfels, ((0, 0), (0, (cells + 127) // 128 * 128)))
    return sc


@pytest.mark.parametrize("name,filt", [("cfg1", False), ("cfg1", True), ("tiny", True), ("small", True)])
def test_create_surfels_for_keyframe_three_way(mods, name, filt):
    """DirectBA::CreateSurfelsForKeyframe (direct_ba.cc:340-405).  sparse cell size 1 (cfg1): the seed pixel of a cell is unique, so
    the result equals the reference's; larger cells: the reference seeds a random valid pixel of the cell (atomicCAS), this
    library and the oracle the first one in raster order -> same number of cells seeded, compared in distribution."""
    S, DirectBA, O, R = mods
    sc = _half_map(S, name)
    n0 = sc.num_surfels
    ba, ref, orc = DirectBA.from_scene(sc), R.reference(sc), O.Oracle(sc)
    # The reference's outcome for cell size > 1 depends on an atomicCAS race (kernel_create_surfels.cu:68): two more independent
    # runs give its own spread.  Measured on B200 with five runs (profiles/r2/lifecycle_spread.log): the reference scatters by
    # 0.1 - 1 % per keyframe, while a fixed tie-break rule is a DIFFERENT sample of the race, systematically: this backend's hashed
    # order creates +0.1 ... +3.5 % (13 % for the last keyframe of the smallest scene) more surfels than the reference's mean --
    # 4 to 13 of the reference's standard deviations.  So the reference's spread cannot be the bound; the bound is the measured
    # offset with a margin, and the spread is printed next to it.
    more = [R.reference(sc) for _ in range(2)] if sc.cfg.cell > 1 else []
    K = sc.cfg.num_keyframes
    for k in range(K):
        c0 = ba.CreateSurfelsForKeyframe(None, filt, k)
        c1 = ref.create_surfels_for_keyframe(k, filt)
        c2 = orc.create_surfels_for_keyframe(k, filt)
        assert c0 == c2, (k, c0, c2)                                   # deterministic definition: exact
        if sc.cfg.cell == 1:
            assert c0 == c1, (k, c0, c1)
        else:
            runs = [c1] + [r.create_surfels_for_keyframe(k, filt) for r in more]
            mean = float(np.mean(runs))
            print(name, filt, "keyframe", k, "created: ours", c0, "| reference runs", runs, f"relative offset {(c0 - mean) / mean:+.3f}")
            assert max(runs) - min(runs) <= max(20, 0.06 * mean), (k, runs)          # the reference's own scatter (measured: <= 3 % range over five runs)
            assert abs(c0 - mean) <= max(40, 0.16 * mean), (k, c0, runs)            # (different seed pixels: different coverage / filter outcome)
        assert ba.surfels_size() == orc.n
    n1 = ba.surfels_size()
    assert n1 > n0
    a, c = ba.GetSurfelsHost(), orc.surfels[:8, :orc.n]
    # vs the oracle: same pixels, same order; fp32 contraction differs (fast-math FMA vs plain C)
    assert np.abs(a[:3] - c[:3]).max() < 2e-6
    assert (a[3].view(np.uint32) != c[3].view(np.uint32)).mean() < 1e-3
    assert np.array_equal(a[4], c[4]) and np.array_equal(a[5].view(np.uint32), c[5].view(np.uint32))
    # descriptors: the tangent sample points differ by fast-math round-off, which can move a sample across a 1/256 step of the
    # bilinear weights (one step of one 8-bit level = 0.7 descriptor units)
    assert np.abs(a[6:8] - c[6:8]).mean() < 2e-3 and np.abs(a[6:8] - c[6:8]).max() < 1.0
    if sc.cfg.cell == 1:
        b = ref.surfels()
        assert R.shape_of(b) == a.shape
        a, b = R.same_sample(a, b)
        assert np.abs(a[:3] - b[:3]).max() < 2e-6 and (a[3].view(np.uint32) != b[3].view(np.uint32)).mean() < 1e-3
        assert np.array_equal(a[4], b[4]) and np.array_equal(a[5].view(np.uint32), b[5].view(np.uint32))
        assert np.abs(a[6:8] - b[6:8]).mean() < 2e-3 and np.abs(a[6:8] - b[6:8]).max() < 1.0
    # every new surfel is associated with the keyframe that created it: creating again adds (almost) nothing
    again = sum(ba.CreateSurfelsForKeyframe(None, filt, k) for k in range(K))
    assert again <= 0.02 * (n1 - n0) + 2


@pytest.mark.parametrize("name", ["tiny", "small"])
def test_merge_surfels_three_way(mods, name):
    """DetermineSupportingSurfelsAndMergeSurfelsCUDA on IDENTICAL surfels: surfels created by different keyframes for the same
    surface are merged.  Exact vs the oracle (fixed arrival order); the reference's first-come order marks a different but
    similarly sized set."""
    import copy
    S, DirectBA, O, R = mods
    sc = _half_map(S, name)
    K = sc.cfg.num_keyframes
    seed = DirectBA.from_scene(sc)
    for k in range(K):   # unfiltered creation from every keyframe: plenty of near-duplicates
        seed.CreateSurfelsForKeyframe(None, False, k)
    rows = seed.GetSurfelsHost()
    sc2 = copy.copy(sc)
    sc2.surfels = sc.surfels.copy()
    sc2.num_surfels = rows.shape[1]
    sc2.surfels[:8, :sc2.num_surfels] = rows
    ba, ref, ref2, orc = DirectBA.from_scene(sc2), R.reference(sc2), R.reference(sc2), O.Oracle(sc2)
    total = [0, 0, 0]
    total_ref2 = 0
    for k in range(K):
        d0, d1, d2 = ba.MergeSurfelsForKeyframe(k), ref.merge_surfels_for_keyframe(k), orc.merge_surfels_for_keyframe(k)
        total_ref2 += ref2.merge_surfels_for_keyframe(k)
        assert d0 == d2, (k, d0, d2)
        total = [total[0] + d0, total[1] + d1, total[2] + d2]
    print("merged (ours, reference, second reference run, oracle):", total[0], total[1], total_ref2, total[2], "of", sc2.num_surfels)
    # measured with five reference runs (profiles/r2/lifecycle_spread.log): the reference scatters by 0.3 - 0.7 %, this backend's
    # fixed order merges 0.9 % / 4.3 % fewer surfels than its mean (tiny / small)
    assert abs(total[1] - total_ref2) <= max(10, 0.05 * total[1]), (total[1], total_ref2)
    assert total[0] > 0 and abs(total[0] - total[1]) <= max(5, 0.08 * total[1]), total
    a, c = ba.GetSurfelsHost(), orc.surfels[:8, :orc.n]
    assert np.array_equal(a[0].view(np.uint32) == 0x7fffffff, c[0].view(np.uint32) == 0x7fffffff)   # the same surfels are marked
    n_a = ba.CompactSurfels(total[0], True)
    assert n_a == orc.compact_surfels() == a.shape[1] - total[0]
    a, c = ba.GetSurfelsHost(), orc.surfels[:8, :orc.n]
    assert np.array_equal(a.view(np.uint32), c.view(np.uint32)) and not np.any(a[0].view(np.uint32) == 0x7fffffff)
    assert ref.compact_surfels(total[1], True) == R.shape_of(ref.surfels())[1]


def test_bundle_adjustment_with_surfel_updates(mods):
    """do_surfel_updates = true: creation for newly active keyframes, merge + compaction in the loop, final merge + deletion
    at the end (direct_ba_alternating.cc:399-430,489-541, direct_ba.cc:577-622), against the oracle."""
    S, DirectBA, O, R = mods
    sc = _half_map(S, "small")
    sc.poses_init = S.make_scene(S.config_by_name("small")).poses_init      # perturbed poses: BA has work to do
    ba, orc = DirectBA.from_scene(sc), O.Oracle(sc)
    ro = ba.BundleAdjustment(None, False, False, True, True, True, 2, 2)
    rc = orc.bundle_adjust(True, True, 2, 2, do_surfel_updates=True)
    assert ro.surfels_created == rc.surfels_created > 0
    assert abs(ro.surfels_merged - rc.surfels_merged) <= max(2, 0.01 * rc.surfels_merged)
    assert abs(ro.surfels_size - orc.n) <= max(2, 0.005 * orc.n) and ro.surfels_size == ba.surfels_size()
    pa = ba.GetKeyframeStates()[0]
    for k in range(sc.cfg.num_keyframes):
        dt, dr = S.pose_error(pa[k], orc.poses[k])
        assert dt < 1e-4 and dr < 1e-4, (k, dt, dr)
    assert not np.any(ba.GetSurfelsHost()[0].view(np.uint32) == 0x7fffffff)
    # a second BA iteration block (the counter increased): the keyframes that are still active create surfels again, but only
    # where the end tasks deleted badly observed ones
    r2 = ba.BundleAdjustment(None, False, False, True, True, True, 1, 1)
    assert r2.surfels_created < ro.surfels_created and ba.ba_iteration_count() == 2
