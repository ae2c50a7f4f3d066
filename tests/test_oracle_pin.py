"""Pins the plain-C oracle (oracle/t360_oracle.c) before anything is allowed to trust it.

The reference has no tests or golden vectors of its own (SURVEY.md 4), so the pins are
(a) tests/golden/golden.json -- outputs of THE REFERENCE ITSELF run in the build container
    (oracle/_ref = unmodified reference sources + oracle/shim, driving cv2 4.13.0; generator
    tests/golden/make_golden.py) -- checked without needing /root/reference at run time;
(b) further runs of the reference recorded in the same file ("reference_runs": other seeds, planes and contexts),
    and live comparison with cv2.
"""
import numpy as np
import pytest

from oracle import c_oracle as co
from oracle import ref_harness as rh
from tests.golden.cases import FULL, SMALL, plan_record, plane_dims

cv2 = pytest.importorskip("cv2")


def _ctx(case):
    return rh.default_context(**case["ov"])


def test_context_abi_size():
    import ctypes
    assert ctypes.sizeof(rh.FrameTransformContext) == 112
    assert rh.FrameTransformContext.interpolation_alg.offset == 28
    assert rh.FrameTransformContext.kernel_adjust_factor.offset == 108


def test_noise_generator_matches_numpy_and_survey():
    a = co.noise_plane(1920, 960)
    assert a[0, :8].tolist() == [0, 81, 48, 133, 36, 204, 92, 24]  # SURVEY.md 8(d)
    assert rh.sha16(a) == "ff168fc9d025a214"  # SURVEY.md Appendix D
    assert np.array_equal(a, rh.noise_plane(1920, 960))
    assert np.array_equal(co.noise_plane(333, 77, plane=2, frame=5), rh.noise_plane(333, 77, plane=2, frame=5))


@pytest.mark.parametrize("name", sorted(SMALL))
def test_oracle_vs_golden(name, golden):
    """C oracle end to end (map -> plan -> low-pass -> remap) == the reference's recorded outputs."""
    case = SMALL[name]
    ctx = _ctx(case)
    barrel = ctx.output_layout in (rh.LAYOUT_BARREL, rh.LAYOUT_BARREL_SPLIT)
    for plane in (0, 1):
        g = golden["small"][name]["planes"][str(plane)]
        iw, ih, ow, oh, idx = plane_dims(case, plane)
        assert g["dims"] == [iw, ih, ow, oh, idx]
        plan = co.OraclePlan(ctx, iw, ih, ow, oh)
        assert co.fnv1a64(plan.map) == g["map_fnv"], "geometry differs from the reference"
        assert plan.nsegs == g["nsegs"]
        if plan.nsegs:
            lst = co.plan_as_list(plan.segs, plan.nsegs, plan.taps)
            rects = np.array([s[:4] for s in lst], np.int32)
            taps = np.concatenate([np.concatenate([s[4], s[5]]) for s in lst])
            assert co.fnv1a64(rects) == g["rects_fnv"], "low-pass tile table differs from the reference"
            assert co.fnv1a64(taps) == g["taps_fnv"], "low-pass kernels differ from the reference"
        src = co.noise_plane(iw, ih, plane=plane, frame=0)
        assert rh.sha16(src) == g["src_sha"]
        out = co.transform_plane(ctx, plan, src, ow, oh, map_index=idx, prefill=7 if barrel else 0)
        assert out[0, :8].tolist() == g["out_head"]
        assert int(out.sum(dtype=np.int64)) == g["out_sum"]
        assert rh.sha16(out) == g["out_sha"], "pixels differ from the reference"


@pytest.mark.slow
@pytest.mark.parametrize("name", ["cfg2", "cfg3"])
def test_oracle_vs_golden_full_size(name, golden):
    case = FULL[name]
    ctx = _ctx(case)
    g = golden["full"][name]["planes"]["0"]
    iw, ih, ow, oh, idx = plane_dims(case, 0)
    plan = co.OraclePlan(ctx, iw, ih, ow, oh)
    assert co.fnv1a64(plan.map) == g["map_fnv"]
    out = co.transform_plane(ctx, plan, co.noise_plane(iw, ih), ow, oh)
    assert rh.sha16(out) == g["out_sha"]


@pytest.mark.parametrize("interp", [rh.NEAREST, rh.LINEAR, rh.CUBIC, rh.LANCZOS4])
def test_remap_arithmetic_vs_cv2(interp):
    """SURVEY.md Appendix A: bit-exact against cv2.remap, BORDER_WRAP, coordinates spilling over every edge."""
    rng = np.random.default_rng(1234 + interp)
    src = rng.integers(0, 256, (97, 131), dtype=np.uint8)
    m = np.empty((300, 400, 2), np.float32)
    m[..., 0] = rng.uniform(-9, 131 + 9, (300, 400))
    m[..., 1] = rng.uniform(-9, 97 + 9, (300, 400))
    m[:50, :, 0] = np.round(m[:50, :, 0] * 2) / 2  # exact .5 ties exercise round-half-even
    m[:50, :, 1] = np.round(m[:50, :, 1] * 64) / 64
    want = cv2.remap(src, m, None, interp, borderMode=cv2.BORDER_WRAP)
    got = co.remap_u8(src, m, interp, 3)
    assert np.array_equal(got, want)


@pytest.mark.parametrize("border", [cv2.BORDER_WRAP, cv2.BORDER_TRANSPARENT])
@pytest.mark.parametrize("interp", [rh.NEAREST, rh.LINEAR, rh.CUBIC, rh.LANCZOS4])
def test_remap_of_nan_and_out_of_range_coordinates_vs_cv2(interp, border):
    """Maps can hold NaN (off-centre + is_horizontal_offset divides by zero at the poles, ref:1203-1206) and values far
    outside the int range: cv2 rounds them to INT_MIN (cvtss2si) before saturating to 16 bits.  Bit-exact."""
    rng = np.random.default_rng(5 + interp)
    src = rng.integers(0, 256, (97, 131), dtype=np.uint8)
    m = np.empty((64, 96, 2), np.float32)
    m[..., 0] = rng.uniform(-9, 140, (64, 96))
    m[..., 1] = rng.uniform(-9, 106, (64, 96))
    specials = [np.nan, np.inf, -np.inf, 1e12, -1e12, 3e9, -3e9, 2147483648.0, -2147483648.0, 7e7, -7e7, 1e6, -1e6, 40000.5, -40000.5]
    k = 0
    for yy in range(0, 64, 4):
        for xx in range(0, 96, 3):
            v = specials[k % len(specials)]
            k += 1
            if k % 3 == 0:
                m[yy, xx, 0] = v
            elif k % 3 == 1:
                m[yy, xx, 1] = v
            else:
                m[yy, xx] = v
    if border == cv2.BORDER_TRANSPARENT:
        want = np.full((64, 96), 77, np.uint8)
        cv2.remap(src, m, None, interp, dst=want, borderMode=border)
        got = np.full((64, 96), 77, np.uint8)
        co.remap_u8(src, m, interp, 5, dst=got)
    else:
        want = cv2.remap(src, m, None, interp, borderMode=border)
        got = co.remap_u8(src, m, interp, 3)
    assert np.array_equal(got, want)


@pytest.mark.parametrize("interp", [rh.NEAREST, rh.LINEAR, rh.CUBIC, rh.LANCZOS4])
def test_remap_transparent_vs_cv2(interp):
    rng = np.random.default_rng(99 + interp)
    src = rng.integers(0, 256, (64, 80), dtype=np.uint8)
    m = np.empty((120, 150, 2), np.float32)
    m[..., 0] = rng.uniform(-6, 86, (120, 150))
    m[..., 1] = rng.uniform(-6, 70, (120, 150))
    m[10:20, 10:30] = (-1.0, 0.0)  # the reference's "no mapping" marker (cpp:1305-1306)
    want = np.full((120, 150), 128, np.uint8)
    cv2.remap(src, m, None, interp, dst=want, borderMode=cv2.BORDER_TRANSPARENT)
    got = co.remap_u8(src, m, interp, 5, dst=np.full((120, 150), 128, np.uint8))
    assert np.array_equal(got, want)


def test_bilinear_transparent_edge_rule_vs_cv2():
    """Pixels whose anchor is on the last row / column under BORDER_TRANSPARENT (renormalised blend, round half up)."""
    rng = np.random.default_rng(5)
    H, W = 40, 50
    src = rng.integers(0, 256, (H, W), dtype=np.uint8)
    m = np.zeros((3, 4000, 2), np.float32)
    m[0, :, 0] = W - 1 + rng.uniform(0, 0.99, 4000); m[0, :, 1] = rng.uniform(-0.4, H - 0.01, 4000)
    m[1, :, 0] = rng.uniform(-0.4, W - 0.01, 4000); m[1, :, 1] = H - 1 + rng.uniform(0, 0.99, 4000)
    m[2, :, 0] = W - 1 + rng.uniform(0, 0.99, 4000); m[2, :, 1] = H - 1 + rng.uniform(0, 0.99, 4000)
    want = np.full((3, 4000), 77, np.uint8)
    cv2.remap(src, m, None, cv2.INTER_LINEAR, dst=want, borderMode=cv2.BORDER_TRANSPARENT)
    got = co.remap_u8(src, m, rh.LINEAR, 5, dst=np.full((3, 4000), 77, np.uint8))
    assert np.array_equal(got, want)


@pytest.mark.parametrize("dims", [(64, 48, 32, 24), (96, 60, 32, 20), (96, 60, 48, 20), (64, 48, 32, 48), (128, 64, 32, 16),
                                  (65, 49, 32, 24), (96, 72, 64, 48), (100, 60, 40, 24), (75, 50, 50, 20), (64, 48, 48, 48),
                                  (97, 31, 13, 7), (1152, 1024, 768, 512)])
def test_area_resize_vs_cv2(dims):
    """cv::resize(INTER_AREA) shrinking, the call at reference cpp:770-776: integer ratios (2x2 and general) and
    fractional ratios, bit-exact."""
    sw, sh, dw, dh = dims
    src = np.random.default_rng(sw * 7 + dh).integers(0, 256, (sh, sw), dtype=np.uint8)
    assert np.array_equal(co.resize_area(src, dw, dh), cv2.resize(src, (dw, dh), interpolation=cv2.INTER_AREA))


def test_area_resize_enlarging_vs_cv2():
    """cv::resize(INTER_AREA) with at least one enlarging axis (the reference reaches it with *_scale_factor < 1): OpenCV
    falls back to its 8-bit fixed-point bilinear kernel with "area mode" coefficients.  300 random size pairs (shrinking,
    enlarging, mixed, tiny), bit-exact."""
    rng = np.random.default_rng(3)
    for _ in range(300):
        sw, sh = int(rng.integers(2, 200)), int(rng.integers(2, 150))
        dw, dh = int(rng.integers(max(1, sw // 3), sw * 3 + 2)), int(rng.integers(max(1, sh // 3), sh * 3 + 2))
        src = rng.integers(0, 256, (sh, sw), dtype=np.uint8)
        assert np.array_equal(co.resize_area(src, dw, dh), cv2.resize(src, (dw, dh), interpolation=cv2.INTER_AREA)), (sw, sh, dw, dh)


# width/height_scale_factor < 1 end to end: (context overrides, (in_w, in_h, out_w, out_h))
SCALE_BELOW_ONE = ((dict(width_scale_factor=0.5, height_scale_factor=0.5, interpolation_alg=2), (320, 160, 96, 64)),
                   (dict(width_scale_factor=0.75, height_scale_factor=1.0, interpolation_alg=1, enable_low_pass_filter=0), (256, 128, 96, 64)),
                   (dict(width_scale_factor=2.0, height_scale_factor=0.6, interpolation_alg=4, output_layout=rh.LAYOUT_EAC_32), (300, 150, 60, 50)),
                   (dict(width_scale_factor=0.9, height_scale_factor=0.8, interpolation_alg=0, output_layout=rh.LAYOUT_BARREL), (256, 128, 100, 40)))


def _prefill(ctx):
    return 9 if ctx.output_layout in (rh.LAYOUT_BARREL, rh.LAYOUT_BARREL_SPLIT) else 0


def test_scale_factors_below_one_end_to_end_vs_live_reference(golden):
    """width/height_scale_factor < 1: render at the smaller map size, then INTER_AREA *up* (ref:755-777); against the
    reference's own outputs for the same planes (golden.json "reference_runs", make_golden.py)."""
    runs = golden["reference_runs"]["scale_below_one"]
    assert len(runs) == len(SCALE_BELOW_ONE)
    for (ov, dims), want in zip(SCALE_BELOW_ONE, runs):
        ctx = rh.default_context(**ov)
        iw, ih, ow, oh = dims
        for idx in (0, 1):
            plan = co.OraclePlan(ctx, iw, ih, ow, oh)
            src = co.noise_plane(iw, ih, plane=idx, frame=5)
            got = co.transform_plane(ctx, plan, src, ow, oh, map_index=idx, prefill=_prefill(ctx))
            assert rh.sha16(got) == want[idx], (ov, idx)


def test_itab_sums():
    for interp in (rh.LINEAR, rh.CUBIC, rh.LANCZOS4):
        t = co.build_itab(interp)
        assert (t.reshape(1024, -1).astype(np.int32).sum(1) == 32768).all()


@pytest.mark.parametrize("sx,sy", [(0.75, 0.75), (1.2, 0.75), (7.2, 0.75), (2.3, 1.6), (14.9, 3.1)])
def test_sepfilter_arithmetic_vs_cv2(sx, sy):
    """The FMA model of cv2 4.13's optimized sepFilter2D (see t360_oracle.c): bit-exact on whole planes."""
    src = co.noise_plane(1024, 384, plane=1, frame=3)

    def gauss(sigma):
        half = int(np.float32(sigma) * 2)
        u = np.arange(-half, half + 1)
        v = np.exp(-(u * u).astype(np.float32) * np.float32(0.5 / (np.float32(sigma) * np.float32(sigma)))).astype(np.float32)
        return (v / v.sum(dtype=np.float32)).astype(np.float32)

    kx, ky = gauss(sx), gauss(sy)
    want = cv2.sepFilter2D(src, -1, kx.reshape(1, -1), ky.reshape(1, -1), borderType=cv2.BORDER_REPLICATE)
    got = co.sepfilter_roi(src, 0, 0, 1024, 384, kx, ky, np.zeros_like(src))
    assert np.array_equal(got, want)
    # a tile in the middle of the plane must equal the same window of the whole-plane result (non-isolated ROI)
    tile = co.sepfilter_roi(src, 300, 100, 240, 128, kx, ky, np.zeros_like(src))
    assert np.array_equal(tile[100:228, 300:540], want[100:228, 300:540])


LIVE_CASES = ["lp_tiles", "eac_tb_lanczos", "offcenter_adjust", "cube_to_equirect", "barrel"]


@pytest.mark.parametrize("name", LIVE_CASES)
def test_oracle_vs_live_reference(name, golden):
    """Same comparison as the golden test but with another frame seed and planes 0 and 2, down to the tile table and the
    taps, against the reference's own run of them (golden.json "reference_runs", make_golden.py)."""
    case = SMALL[name]
    ctx = _ctx(case)
    runs = golden["reference_runs"]["live_cases"][name]
    for plane in (0, 2):
        iw, ih, ow, oh, idx = plane_dims(case, plane)
        plan = co.OraclePlan(ctx, iw, ih, ow, oh)
        mine = co.plan_as_list(plan.segs, plan.nsegs, plan.taps) if plan.nsegs else []
        assert plan_record(plan.map, mine) == runs[str(plane)]["plan"], f"plane {plane}: plan differs from the reference"
        src = co.noise_plane(iw, ih, plane=plane, frame=17)
        got = co.transform_plane(ctx, plan, src, ow, oh, map_index=idx, prefill=_prefill(ctx))
        assert rh.sha16(got) == runs[str(plane)]["out_sha"], f"plane {plane}: pixels differ from the reference"


def _e2e_sweep_cases(seed):
    """(overrides, (in_w, in_h, out_w, out_h), plan index) of the end-to-end sweep.  Side-by-side stereo outputs of odd
    render width are left out: there the reference reads an uninitialised face basis (DESIGN.md 7)."""
    from tests.test_host_plan import _random_context
    rng = np.random.default_rng(1000 + seed)
    for _ in range(25):
        ov = _random_context(rng)
        iw, ih = int(rng.integers(64, 300)) * 2, int(rng.integers(32, 150)) * 2
        ow, oh = int(rng.integers(24, 120)) * 2 + int(rng.random() < 0.25), int(rng.integers(16, 90)) * 2 + int(rng.random() < 0.25)
        idx = int(rng.integers(0, 2))
        sw, _ = co.scaled_dims(rh.default_context(**ov), ow, oh)
        if ov["input_stereo_format"] != rh.STEREO_FORMAT_MONO and ov["output_stereo_format"] == rh.STEREO_FORMAT_LR and sw % 2 == 1:
            continue
        yield ov, (iw, ih, ow, oh), idx


@pytest.mark.parametrize("seed", [11, 12])
def test_random_end_to_end_sweep_against_the_live_reference(seed, golden):
    """Random contexts over the whole option space, end to end: the C restatement must produce the bytes the reference's
    own object code + cv2 produced for them (golden.json "reference_runs", make_golden.py).  (1300 cases of this sweep,
    offline, found the NaN-coordinate rule pinned above.)"""
    cases = list(_e2e_sweep_cases(seed))
    runs = golden["reference_runs"]["e2e_sweep"][str(seed)]
    assert len(runs) == len(cases)
    compared = 0
    for (ov, (iw, ih, ow, oh), idx), want in zip(cases, runs):
        if want is None:  # the reference refused the plan or the frame
            continue
        ctx = rh.default_context(**ov)
        plan = co.OraclePlan(ctx, iw, ih, ow, oh)
        src = co.noise_plane(iw, ih, plane=idx, frame=seed)
        try:
            got = co.transform_plane(ctx, plan, src, ow, oh, map_index=idx, prefill=_prefill(ctx))
        except RuntimeError:  # scale factors < 1 are not restated (INTER_AREA enlarging)
            continue
        assert rh.sha16(got) == want, f"pixels differ for {ov} {(iw, ih, ow, oh)} plan {idx}"
        compared += 1
    assert compared >= 15
