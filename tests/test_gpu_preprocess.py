"""GPU parity of the fused keyframe preprocessing (bba_preprocess_frame; SURVEY.md 8(f3)): the sm_100a kernel through the C ABI
against the reference's own five kernels (oracle/_ref: cuda_depth_processing.cu, cuda_image_processing.cu) and the CPU oracle.

What can be demanded: the reference is built with -use_fast_math, so its bilateral filter is a chain of MUFU.RCP / MUFU.EX2
approximations whose float result is TRUNCATED to a raw depth unit.  The product kernel compiles the same expressions with the
same flags (same SASS arithmetic), so it is expected to agree with the reference bit for bit; the tests allow a difference of one
raw unit / one s8 normal step / two half ulps on a small fraction of the pixels, and demand identical validity masks and luma.
The IEEE oracle crosses a truncation boundary on more pixels; wherever the filtered depth of a pixel and its 4-neighbours
agrees, normals and radii must agree as well."""
import numpy as np
import pytest

pytestmark = [pytest.mark.gpu]


@pytest.fixture(scope="module")
def mods():
    import torch
    assert torch.cuda.is_available()
    from badslam_b200 import scene as S
    from badslam_b200.direct_ba import DirectBA
    from oracle import cpu_oracle, ref_cuda
    return S, DirectBA, cpu_oracle, ref_cuda


def run_cuda(ba, raw, rgb, **kw):
    import torch
    d_raw = torch.from_numpy(raw.view(np.int16)).cuda()
    d_rgb = None if rgb is None else torch.from_numpy(np.ascontiguousarray(rgb)).cuda()
    depth, normals, radius, rgba, mn, mx = ba.PreprocessFrame(d_raw, d_rgb, **kw)
    torch.cuda.synchronize()
    host = lambda t: t.view(torch.int16).cpu().numpy().view(np.uint16)
    return host(depth), host(normals), host(radius), None if rgba is None else rgba.cpu().numpy(), mn, mx


def s8_pair(n16):
    return (n16 & 0xff).astype(np.int8).astype(np.int32), (n16 >> 8).astype(np.int8).astype(np.int32)


def compare(got, want, rtf, depth_fraction, other_fraction, what, min_agree=0.5):
    from oracle.ref_cuda import identical, same_sample
    gd, gn, gr, gc, gmin, gmax = got
    wd, wn, wr, wc, wmin, wmax = want
    if wc is not None:
        assert identical(gc, wc), f"{what}: rgba / luma"
    assert np.all(gn[0] == 0) and np.all(gn[:, 0] == 0)
    any_valid = np.any((gd & 0x8000) == 0)
    (gd, wd), (gn, wn), (gr, wr) = same_sample(gd, wd), same_sample(gn, wn), same_sample(gr, wr)   # (a window of a recorded image)
    valid = (wd & 0x8000) == 0
    assert np.array_equal((gd & 0x8000) == 0, valid), f"{what}: different pixels dropped"
    assert np.all(gd[~valid] == 65535)
    dd = np.abs(gd[valid].astype(np.int32) - wd[valid].astype(np.int32))
    assert dd.size == 0 or (dd.max() <= 1 and np.mean(dd != 0) <= depth_fraction), (what, dd.max(), np.mean(dd != 0))
    # pixels whose own filtered depth and whose 4 neighbours' agree (and are valid in the output of both)
    same = valid & (gd == wd)
    nb = same.copy()
    nb[1:] &= same[:-1]; nb[:-1] &= same[1:]; nb[:, 1:] &= same[:, :-1]; nb[:, :-1] &= same[:, 1:]
    if valid.any():
        assert nb.sum() >= min_agree * valid.sum() or valid.sum() < 64, what
    ax, ay = s8_pair(gn[nb])
    bx, by = s8_pair(wn[nb])
    if ax.size:
        assert max(np.abs(ax - bx).max(), np.abs(ay - by).max()) <= 1, what
        assert np.mean((ax != bx) | (ay != by)) <= other_fraction, (what, np.mean((ax != bx) | (ay != by)))
        ra, rb = gr[nb].view(np.float16).astype(np.float64), wr[nb].view(np.float16).astype(np.float64)
        # radius^2 is stored as an IEEE half: close surfaces give SUBNORMAL halves (pixel spacing 1.7 mm at 0.2 m: r^2 = 3e-6 =
        # 50 units of 2^-24), where one rounding step is 2 % of the value -- the tolerance is two half ulps, normal or subnormal
        assert np.all(np.abs(ra - rb) <= np.maximum(2.0 ** -9 * rb, 2.0 ** -23)), (what, np.abs(ra - rb).max())
        assert np.mean(ra != rb) <= other_fraction, (what, np.mean(ra != rb))
    if any_valid:
        assert abs(gmin - wmin) <= 1.5 * rtf and abs(gmax - wmax) <= 1.5 * rtf, what
    else:
        assert gmin == wmin == float("inf") and gmax == wmax == 0.0, what
    return float(np.mean(dd != 0)) if dd.size else 0.0


@pytest.mark.parametrize("name,kf", [("small", 0), ("small", 1), ("cfg2", 3)])
def test_preprocess_frame_three_way(mods, name, kf):
    S, DirectBA, O, R = mods
    sc = S.make_scene(S.config_by_name(name))
    # a depth deformation for the normals stage (a, cfactor as after an intrinsics optimisation)
    rng = np.random.default_rng(5)
    sc.depth_a = 0.02
    sc.cfactor = (2e-3 * rng.random(sc.cfactor.shape)).astype(np.float32)
    raw, rgb = S.raw_frame(sc, kf)
    raw[100:103, :] = 0
    ba, ref = DirectBA.from_scene(sc), R.reference(sc)
    got = run_cuda(ba, raw, rgb)
    want_ref = ref.preprocess_frame(raw, rgb)
    rtf = sc.cfg.raw_to_float_depth
    f_ref = compare(got, want_ref, rtf, 1e-3, 1e-2, "cuda vs reference kernels")
    valid = (got[0] & 0x8000) == 0
    assert 0.3 < valid.mean() < 1.0
    if name == "small":
        want_orc = O.Oracle(sc).preprocess_frame(raw, rgb)
        f_orc = compare(got, want_orc, rtf, 3e-2, 2e-2, "cuda vs oracle")
        print(f"{name}/{kf}: depth differs from the reference kernels on {f_ref:.2e}, from the IEEE oracle on {f_orc:.2e} of the pixels")
    # the launch count: 2 (min/max init + fused kernel) against the reference's 5
    n0 = ba.kernel_launch_count()
    run_cuda(ba, raw, rgb)
    assert ba.kernel_launch_count() - n0 == 2


@pytest.mark.parametrize("opts", [dict(bilateral_filter_sigma_xy=1.0, bilateral_filter_radius_factor=1.0),
                                  dict(bilateral_filter_sigma_xy=0.2),                       # radius 0
                                  dict(bilateral_filter_sigma_xy=3.0, bilateral_filter_sigma_inv_depth=0.02, max_depth=2.5),
                                  dict(bilateral_filter_sigma_xy=8.0, bilateral_filter_radius_factor=2.0)])   # radius 16
def test_filter_parameters(mods, opts):
    S, DirectBA, O, R = mods
    sc = S.make_scene(S.config_by_name("small"))
    raw, rgb = S.raw_frame(sc, 2)
    ba, ref = DirectBA.from_scene(sc), R.reference(sc)
    got = run_cuda(ba, raw, rgb, **opts)
    kw = dict(sigma_xy=opts.get("bilateral_filter_sigma_xy", 1.5), sigma_inv_depth=opts.get("bilateral_filter_sigma_inv_depth", 0.005),
              radius_factor=opts.get("bilateral_filter_radius_factor", 2.0), max_depth=opts.get("max_depth", 3.0))
    compare(got, ref.preprocess_frame(raw, rgb, **kw), sc.cfg.raw_to_float_depth, 1e-3, 1e-2, f"cuda vs reference kernels {opts}")
    if kw["radius_factor"] * kw["sigma_xy"] + 0.5 < 1:
        # radius 0: the filter returns rcp(rcp(c)) truncated -- c or c - 1 depending on the last bit of the arithmetic, which only
        # an implementation with the reference's instruction sequence reproduces; the IEEE oracle agrees up to that unit
        compare(got, O.Oracle(sc).preprocess_frame(raw, rgb, **kw), sc.cfg.raw_to_float_depth, 1.0, 3e-2, f"cuda vs oracle {opts}", 0.0)
    else:
        compare(got, O.Oracle(sc).preprocess_frame(raw, rgb, **kw), sc.cfg.raw_to_float_depth, 5e-2, 3e-2, f"cuda vs oracle {opts}")


@pytest.mark.parametrize("size", [(70, 45), (33, 31), (8, 5), (641, 479)])   # smaller ones: CPU suite (tile program on the host)
def test_ragged_and_tiny_images(mods, size):
    S, DirectBA, O, R = mods
    w, h = size
    sc = S.blank_scene(w, h)
    raw, rgb = S.random_raw_frame(w, h, seed=w * 100 + h)
    ba, ref = DirectBA.from_scene(sc), R.reference(sc)
    got = run_cuda(ba, raw, rgb)
    compare(got, ref.preprocess_frame(raw, rgb), sc.cfg.raw_to_float_depth, 2e-3, 2e-2, f"cuda vs reference kernels {size}")
    compare(got, O.Oracle(sc).preprocess_frame(raw, rgb), sc.cfg.raw_to_float_depth, 5e-2, 3e-2, f"cuda vs oracle {size}")


def test_product_reproduces_the_reference_golden_fixture_bit_for_bit(mods):
    """tests/golden/tiny_preprocess.npz holds the reference kernels' outputs (tools/make_golden.py --preprocess-only).  On the B200
    the product agreed with the reference's -use_fast_math kernels bit for bit on every case measured (same SASS arithmetic),
    so the fixture is demanded exactly: depth, normals, radii, luma, min / max depth."""
    import os
    S, DirectBA, O, R = mods
    g = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "tiny_preprocess.npz"))
    sc = S.make_scene(S.config_by_name("tiny"))
    sc.depth_a = 0.02
    sc.cfactor = (2e-3 * np.random.default_rng(5).random(sc.cfactor.shape)).astype(np.float32)
    raw, rgb = S.raw_frame(sc, int(g["kf"]))
    assert int(raw.astype(np.uint64).sum()) == int(g["raw_checksum"])
    d, n, r, c, mn, mx = run_cuda(DirectBA.from_scene(sc), raw, rgb)
    valid = (g["depth"] & 0x8000) == 0
    assert np.array_equal(d, g["depth"])
    assert np.array_equal(n[valid], g["normals"][valid]) and np.array_equal(r[valid], g["radius"][valid])
    assert np.array_equal(c[..., 3], g["luma"])
    assert mn == float(g["min_depth"]) and mx == float(g["max_depth"])


def test_edge_cases_and_errors(mods):
    import torch
    S, DirectBA, O, R = mods
    from badslam_b200._lib import BadBAError
    w, h = 96, 64
    sc = S.blank_scene(w, h)
    ba = DirectBA.from_scene(sc)
    raw, rgb = S.random_raw_frame(w, h, seed=4)
    # an empty frame: everything unknown, min / max at their initial values
    d, n, r, c, mn, mx = run_cuda(ba, np.zeros((h, w), np.uint16), rgb)
    assert np.all(d == 65535) and np.all(n == 0) and np.all(r == 0) and mn == float("inf") and mx == 0.0
    # depth only (no colour image)
    got = run_cuda(ba, raw, None)
    want = O.Oracle(sc).preprocess_frame(raw, None)
    compare(got, want, sc.cfg.raw_to_float_depth, 5e-2, 3e-2, "depth only")
    # pitched inputs / outputs: a window of a wider allocation
    wide = torch.zeros((h, w + 24), dtype=torch.int16, device="cuda")
    wide[:, :w] = torch.from_numpy(raw.view(np.int16)).cuda()
    d2 = ba.PreprocessFrame(wide[:, :w], None)
    torch.cuda.synchronize()
    assert np.array_equal(d2[0].view(torch.int16).cpu().numpy().view(np.uint16), got[0])
    # without min / max the call does not synchronise and still fills the images
    d3 = ba.PreprocessFrame(torch.from_numpy(raw.view(np.int16)).cuda(), None, want_min_max=False)
    torch.cuda.synchronize()
    assert np.array_equal(d3[0].view(torch.int16).cpu().numpy().view(np.uint16), got[0])
    # loud failures
    with pytest.raises(BadBAError):
        ba.PreprocessFrame(torch.from_numpy(raw.view(np.int16)).cuda(), None, bilateral_filter_sigma_xy=20.0)   # radius 40 > 16
    with pytest.raises(BadBAError):
        ba.PreprocessFrame(torch.from_numpy(raw.view(np.int16)).cuda(), None, max_depth=0.0)


def test_keyframes_from_raw_frames_feed_bundle_adjustment(mods):
    """Raw frames -> PreprocessFrame -> AddKeyframe -> surfel creation -> BA: the path BadSlam::ProcessFrame /
    CreateKeyframe / RunBundleAdjustment takes (bad_slam.cc:640-1010), end to end on the device."""
    import torch
    S, DirectBA, O, R = mods
    sc = S.make_scene(S.config_by_name("small"))
    cfg = sc.cfg
    from badslam_b200.direct_ba import PinholeCamera4f
    cam = PinholeCamera4f(cfg.width, cfg.height, sc.depth_K)
    cap = 1 << 18
    ba = DirectBA(cap, cfg.raw_to_float_depth, cfg.baseline_fx, cfg.cell, color_camera_initial_estimate=cam,
                  depth_camera_initial_estimate=cam, max_keyframes=cfg.num_keyframes)
    surf = torch.zeros((17, cap), dtype=torch.float32, device="cuda")
    ba.SetSurfels(surf, 0)
    created = 0
    for k in range(cfg.num_keyframes):
        raw, rgb = S.raw_frame(sc, k, noise_raw=1.0)
        kf = ba.CreateKeyframeFromFrame(k, torch.from_numpy(raw.view(np.int16)).cuda(), torch.from_numpy(rgb).cuda(),
                                        sc.poses_init[k], max_depth=6.0)
        assert 0 < kf.min_depth < kf.max_depth <= 6.0
        created += ba.CreateSurfelsForKeyframe(None, True, kf.id)
    assert created > 1000 and ba.surfels_size() == created
    r = ba.BundleAdjustment(None, False, False, False, True, True, 3, 3)
    assert r.iterations_done == 3 and r.depth_residual_count > 0.5 * created
    poses = ba.GetKeyframeStates()[0]
    assert np.all(np.isfinite(poses))

    def rel(P, k):   # BA fixes relative poses (gauge freedom): keyframes 1..K-1 relative to keyframe 0
        return S.se3_mul(S.se3_inverse(P[0]), P[k])
    e_init = max(S.pose_error(rel(sc.poses_init, k), rel(sc.poses_true, k))[0] for k in range(1, cfg.num_keyframes))
    e_ba = max(S.pose_error(rel(poses, k), rel(sc.poses_true, k))[0] for k in range(1, cfg.num_keyframes))
    print(f"relative pose error: {e_init:.2e} m before, {e_ba:.2e} m after 3 BA iterations on preprocessed raw frames")
    assert e_ba < 1.5 * e_init + 1e-3      # noisy, filtered depth: BA must at least not diverge
