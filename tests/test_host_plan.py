"""Host-side logic of the product, no GPU: the planner inside libTransform360.so must reproduce the
reference's plan bit for bit (map floats, fixed-point samples, tile table, Gaussian taps, weight tables),
and the library must export the drop-in ABI."""
import ctypes
import re
import subprocess
from pathlib import Path

import numpy as np
import pytest

import transform360_b200 as t360
from oracle import c_oracle as co
from oracle import ref_harness as rh
from tests.golden.cases import FULL, SMALL, plan_record, plane_dims
from transform360_b200 import build as t360_build

ROOT = Path(__file__).resolve().parents[1]


@pytest.fixture(scope="module", autouse=True)
def _built():
    t360_build.build()


def _ctxs(case):
    return t360.make_context(**case["ov"]), rh.default_context(**case["ov"])


def test_library_exports_declared_abi():
    """Every symbol include/*.h declares is exported, with C linkage; nothing else of ours leaks."""
    from transform360_b200.handler import EXPORTED_SYMBOLS, LIB_PATH
    out = subprocess.run(["nm", "-D", "--defined-only", str(LIB_PATH)], capture_output=True, text=True, check=True).stdout
    exported = {line.split()[-1] for line in out.splitlines() if " T " in line}
    declared = set()
    for h in ["include/Transform360/VideoFrameTransformHandler.h", "include/transform360_b200.h"]:
        declared |= set(re.findall(r"\b(VideoFrameTransform_\w+|T360B200_\w+)\s*\(", (ROOT / h).read_text()))
    assert declared == set(EXPORTED_SYMBOLS)
    assert declared <= exported
    assert not any(s.startswith("_ZN4t360") for s in exported), "internal C++ symbols must stay hidden"
    lib = t360.load()
    for s in EXPORTED_SYMBOLS:
        assert getattr(lib, s)


def test_context_layout_matches_reference_header(tmp_path):
    assert ctypes.sizeof(t360.FrameTransformContext) == 112
    assert t360.FrameTransformContext.interpolation_alg.offset == 28
    assert t360.FrameTransformContext.kernel_adjust_factor.offset == 108
    src = (ROOT / "include/Transform360/VideoFrameTransformHelper.h").read_text()
    for name, val in [("LAYOUT_CUBEMAP_32", 0), ("LAYOUT_CUBEMAP_23_OFFCENTER", 1), ("LAYOUT_FLAT_FIXED", 2),
                      ("LAYOUT_EQUIRECT", 3), ("LAYOUT_BARREL", 4), ("LAYOUT_BARREL_SPLIT", 5), ("LAYOUT_EAC_32", 6),
                      ("LAYOUT_N", 7), ("STEREO_FORMAT_TB", 0), ("STEREO_FORMAT_LR", 1), ("STEREO_FORMAT_MONO", 2),
                      ("STEREO_FORMAT_GUESS", 3), ("NEAREST", 0), ("LINEAR", 1), ("CUBIC", 2), ("LANCZOS4", 4)]:
        assert re.search(rf"\b{name} = {val}\b", src), name
    # a C compiler sees the same struct
    prog = '#include "Transform360/VideoFrameTransformHandler.h"\n#include <stddef.h>\n#include <stdio.h>\n' \
           'int main(void){printf("%zu %zu %zu", sizeof(FrameTransformContext), offsetof(FrameTransformContext, interpolation_alg),' \
           ' offsetof(FrameTransformContext, kernel_adjust_factor));return 0;}'
    exe = tmp_path / "t360_abi_probe"
    subprocess.run(["gcc", "-std=c11", "-x", "c", "-", "-I", str(ROOT / "include"), "-o", str(exe)], input=prog, text=True, check=True)
    assert subprocess.run([str(exe)], capture_output=True, text=True).stdout == "112 28 108"


@pytest.mark.parametrize("name", sorted(SMALL))
def test_plan_matches_oracle_and_golden(name, golden):
    case = SMALL[name]
    ctx, octx = _ctxs(case)
    for plane in (0, 1):
        iw, ih, ow, oh, idx = plane_dims(case, plane)
        hp = t360.HostPlan(ctx, iw, ih, ow, oh)
        g = golden["small"][name]["planes"][str(plane)]
        m = hp.map
        assert co.fnv1a64(m) == g["map_fnv"], "planner geometry differs from the reference"
        om = co.generate_map(octx, iw, ih, ow, oh)
        assert np.array_equal(m.view(np.uint32), om.view(np.uint32))
        segs = hp.segments()
        assert len(segs) == g["nsegs"]
        if segs:
            rects = np.array([s[:4] for s in segs], np.int32)
            taps = np.concatenate([np.concatenate([s[4], s[5]]) for s in segs])
            assert co.fnv1a64(rects) == g["rects_fnv"]
            assert co.fnv1a64(taps) == g["taps_fnv"]
        hp.close()


def test_samples_follow_opencv_fixed_point():
    """word0/word1 of the sampling plan == cv::remap's conversion of the float map (Appendix A)."""
    for name in ("cube_cubic", "cube_nearest", "cube_lanczos", "cube_linear"):
        case = SMALL[name]
        ctx, _ = _ctxs(case)
        iw, ih, ow, oh, _ = plane_dims(case, 0)
        hp = t360.HostPlan(ctx, iw, ih, ow, oh)
        m, s, k = hp.map, hp.samples, hp.kernel_size
        if k == 1:
            sx = np.clip(np.rint(m[..., 0]).astype(np.int64), -32768, 32767)
            sy = np.clip(np.rint(m[..., 1]).astype(np.int64), -32768, 32767)
            assert np.array_equal(s[..., 0], sx) and np.array_equal(s[..., 1], sy * 1024)
        else:
            X = np.rint(m[..., 0] * np.float32(32)).astype(np.int64)
            Y = np.rint(m[..., 1] * np.float32(32)).astype(np.int64)
            assert np.array_equal(s[..., 0], np.clip(X >> 5, -32768, 32767) - (k // 2 - 1))
            assert np.array_equal(s[..., 1] >> 10, np.clip(Y >> 5, -32768, 32767) - (k // 2 - 1))
            assert np.array_equal(s[..., 1] & 1023, (Y & 31) * 32 + (X & 31))
        hp.close()


@pytest.mark.parametrize("interp", [t360.LINEAR, t360.CUBIC, t360.LANCZOS4])
def test_weight_tables_match_oracle(interp):
    assert np.array_equal(t360.remap_table(interp), co.build_itab(interp))


def test_invalid_parameters_fail_cleanly():
    ctx = t360.make_context()
    with pytest.raises(ValueError):
        t360.HostPlan(ctx, 0, 100, 10, 10)
    ctx = t360.make_context(output_layout=t360.handler.LAYOUT_N)
    with pytest.raises(ValueError):
        t360.HostPlan(ctx, 64, 32, 24, 16)
    # handle creation never needs a GPU; generateMapForPlane needs one and must fail loudly, not fall back
    h = t360.VideoFrameTransform(t360.make_context())
    if t360.device_count() == 0:
        assert h.generateMapForPlane(64, 32, 24, 16, 0) is False
        src = np.zeros((32, 64), np.uint8)
        with pytest.raises(RuntimeError):
            h.transform_plane(src, 24, 16, 0)
    h.close()


@pytest.mark.slow
@pytest.mark.parametrize("name", ["cfg2", "cfg4"])
def test_full_size_plan_matches_golden(name, golden):
    case = FULL[name]
    ctx, _ = _ctxs(case)
    iw, ih, ow, oh, _ = plane_dims(case, 0)
    hp = t360.HostPlan(ctx, iw, ih, ow, oh)
    assert co.fnv1a64(hp.map) == golden["full"][name]["planes"]["0"]["map_fnv"]
    hp.close()


ODD_PARAMETERS = dict(fixed_yaw=123.4, fixed_pitch=-67.8, fixed_roll=179.0, fixed_cube_offcenter_x=0.2, fixed_cube_offcenter_y=-0.15,
                      fixed_cube_offcenter_z=-0.4, num_vertical_segments=12, num_horizontal_segments=7, expand_coef=1.05,
                      kernel_height_scale_factor=1.7, kernel_adjust_factor=1.3, output_layout=t360.LAYOUT_EAC_32)


def test_plan_matches_live_reference_with_odd_parameters(golden):
    """Map, tile table and taps of a 700x350 -> 300x200 plan against the reference's own (golden.json "reference_runs")."""
    hp = t360.HostPlan(t360.make_context(**ODD_PARAMETERS), 700, 350, 300, 200)
    assert plan_record(hp.map, hp.segments()) == golden["reference_runs"]["odd_parameters"]
    hp.close()


def _random_context(rng):
    ov = {}
    ov["input_layout"] = int(rng.choice([3, 3, 3, 0, 6]))  # equirect mostly; cubemap_32 and eac_32 inputs too
    ov["output_layout"] = int(rng.choice([0, 1, 2, 3, 4, 5, 6]))
    st = int(rng.choice([2, 2, 0, 1]))
    ov["input_stereo_format"] = st
    ov["output_stereo_format"] = int(rng.choice([st, 2])) if st != 2 else 2
    ov["vflip"] = int(rng.integers(0, 2))
    ov["input_expand_coef"] = float(rng.choice([1.0, 1.01, 1.03]))
    ov["expand_coef"] = float(rng.choice([1.0, 1.01, 1.05]))
    ov["interpolation_alg"] = int(rng.choice([0, 1, 2, 4]))
    if rng.random() < 0.2:
        ov["width_scale_factor"] = float(rng.choice([1.5, 2.0, 3.0]))
        ov["height_scale_factor"] = float(rng.choice([1.0, 1.25, 2.0]))
    if rng.random() < 0.6:
        ov["fixed_yaw"], ov["fixed_pitch"], ov["fixed_roll"] = (float(rng.uniform(-180, 180)), float(rng.uniform(-90, 90)),
                                                                  float(rng.uniform(-180, 180)))
    ov["fixed_hfov"], ov["fixed_vfov"] = float(rng.uniform(60, 150)), float(rng.uniform(50, 120))
    if rng.random() < 0.4:
        ov["fixed_cube_offcenter_x"] = float(rng.uniform(-0.3, 0.3))
        ov["fixed_cube_offcenter_y"] = float(rng.uniform(-0.3, 0.3))
        ov["fixed_cube_offcenter_z"] = float(rng.uniform(-0.6, 0.3))
        ov["is_horizontal_offset"] = int(rng.integers(0, 2))
    ov["enable_low_pass_filter"] = int(rng.random() < 0.6)
    ov["kernel_height_scale_factor"] = float(rng.uniform(0.5, 3))
    ov["min_kernel_half_height"] = float(rng.uniform(0.5, 2))
    ov["max_kernel_half_height"] = float(rng.choice([3.0, 10000.0]))
    ov["num_vertical_segments"] = int(rng.integers(1, 20))
    ov["num_horizontal_segments"] = int(rng.integers(1, 9))
    ov["adjust_kernel"] = int(rng.integers(0, 2))
    ov["kernel_adjust_factor"] = float(rng.uniform(0.5, 2))
    return ov


def _plan_sweep_cases(seed):
    """(overrides, (in_w, in_h, out_w, out_h)) of the random parameter sweep."""
    rng = np.random.default_rng(seed)
    for _ in range(50):
        ov = _random_context(rng)
        iw, ih = int(rng.integers(64, 400)) * 2, int(rng.integers(32, 200)) * 2
        ow, oh = int(rng.integers(24, 160)) * 2, int(rng.integers(16, 120)) * 2
        yield ov, (iw, ih, ow, oh)


@pytest.mark.parametrize("seed", [1, 2, 3])
def test_random_parameter_sweep_against_the_compiled_reference(seed, golden):
    """Random contexts over the whole option space (layouts both ways, stereo, rotation, off-centre, scale factors,
    low-pass parameters, odd sizes): the planner's float map, tile table and taps must equal, bit for bit, what the
    reference's own object code produced (golden.json "reference_runs", make_golden.py) -- and fail where it failed.  One
    documented exception: the centre column of a side-by-side stereo output of odd render width, where the reference reads
    an uninitialised face basis (DESIGN.md 7); there the planner must equal the C oracle instead.  (1200 cases of this
    sweep found the out-of-range face index and the negative-sigma refusal fixed alongside this test.)"""
    cases = list(_plan_sweep_cases(seed))
    runs = golden["reference_runs"]["plan_sweep"][str(seed)]
    assert len(runs) == len(cases)
    compared = 0
    for (ov, dims), want in zip(cases, runs):
        try:
            hp = t360.HostPlan(t360.make_context(**ov), *dims)
        except ValueError:
            hp = None
        assert (want is not None) == (hp is not None), f"status differs for {ov} {dims}"
        if hp is None:
            continue
        got = plan_record(hp.map, hp.segments(), centre_column=True)
        if got["map"] != want["map"]:
            mw = got["shape"][1]
            lr_centre = ov["input_stereo_format"] != 2 and ov["output_stereo_format"] == 1 and mw % 2 == 1
            assert lr_centre and got["map_but_centre"] == want["map_but_centre"], f"map differs for {ov} {dims}"
            oracle_map = co.generate_map(rh.default_context(**ov), *dims)
            assert np.array_equal(hp.map.view(np.uint32), oracle_map.view(np.uint32)), "planner != C oracle on the centre column"
            got["map"] = want["map"]
        assert got == want, f"plan differs for {ov} {dims}"
        compared += 1
        hp.close()
    assert compared >= 40


NON_POSITIVE_HORIZONTAL_SEGMENTS = [(0, 1), (-2, 1), (0, 0), (-3, 0)]


def _non_positive_overrides(nh, adjust):
    return dict(interpolation_alg=2, enable_low_pass_filter=1, num_vertical_segments=5, num_horizontal_segments=nh, adjust_kernel=adjust)


@pytest.mark.parametrize("nh,adjust", NON_POSITIVE_HORIZONTAL_SEGMENTS)
def test_non_positive_horizontal_segment_counts_follow_the_reference(nh, adjust, golden):
    """Not an error in the reference: with adjust_kernel its tile loop does not run (no tiles: the low-pass output stays
    zero), without adjust_kernel the value is ignored (cpp:224-235).  Against the reference's plan (golden.json)."""
    hp = t360.HostPlan(t360.make_context(**_non_positive_overrides(nh, adjust)), 320, 160, 96, 64)
    segs = hp.segments()
    assert len(segs) == (0 if adjust else 5)
    assert plan_record(hp.map, segs) == golden["reference_runs"]["non_positive_horizontal_segments"][f"{nh},{adjust}"]
    hp.close()
