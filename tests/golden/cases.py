"""Named parity cases shared by the golden-vector generator and the tests.

Each case: context overrides on top of the reference filter defaults
(vf_transform360.c:407-987), luma input dims, luma output dims.  yuv420p is assumed
(chroma = ceil(dim / 2), vf_transform360.c:87-97), plan index 0 = luma, 1 = chroma.
"""
import numpy as np

L_CUBE32, L_CUBE23, L_FLAT, L_EQUIRECT, L_BARREL, L_BARREL_SPLIT, L_EAC = 0, 1, 2, 3, 4, 5, 6
S_TB, S_LR, S_MONO = 0, 1, 2
I_NEAREST, I_LINEAR, I_CUBIC, I_LANCZOS4 = 0, 1, 2, 4

# BASELINE.json configs at full size (GPU tests / bench); cfg1 is also a CPU plumbing case.
FULL = {
    "cfg1": dict(ov=dict(interpolation_alg=I_NEAREST, enable_low_pass_filter=0), inp=(1920, 960), out=(768, 512)),
    "cfg2": dict(ov=dict(interpolation_alg=I_CUBIC, enable_low_pass_filter=0), inp=(7680, 3840), out=(3840, 2560)),
    "cfg3": dict(ov=dict(interpolation_alg=I_CUBIC, enable_low_pass_filter=1, num_horizontal_segments=32,
                         num_vertical_segments=15, adjust_kernel=1), inp=(7680, 3840), out=(3840, 2560)),
    "cfg4": dict(ov=dict(input_stereo_format=S_TB, output_stereo_format=S_TB, output_layout=L_EAC,
                         interpolation_alg=I_LANCZOS4, enable_low_pass_filter=1, num_horizontal_segments=32,
                         num_vertical_segments=15, adjust_kernel=1), inp=(7680, 7680), out=(3840, 5120)),
}

# Small cases: every interpolator, low-pass on/off, stereo, EAC, rotation, off-centre, inverse direction.
SMALL = {
    "cfg1": FULL["cfg1"],
    "cube_nearest": dict(ov=dict(interpolation_alg=I_NEAREST, enable_low_pass_filter=0), inp=(512, 256), out=(192, 128)),
    "cube_linear": dict(ov=dict(interpolation_alg=I_LINEAR, enable_low_pass_filter=0), inp=(512, 256), out=(192, 128)),
    "cube_cubic": dict(ov=dict(interpolation_alg=I_CUBIC, enable_low_pass_filter=0), inp=(512, 256), out=(192, 128)),
    "cube_lanczos": dict(ov=dict(interpolation_alg=I_LANCZOS4, enable_low_pass_filter=0), inp=(512, 256), out=(192, 128)),
    "cube_cubic_odd": dict(ov=dict(interpolation_alg=I_CUBIC, enable_low_pass_filter=0), inp=(509, 251), out=(189, 126)),
    "lp_default": dict(ov=dict(interpolation_alg=I_CUBIC), inp=(640, 320), out=(240, 160)),
    "lp_tiles": dict(ov=dict(interpolation_alg=I_CUBIC, num_horizontal_segments=8, num_vertical_segments=15),
                     inp=(960, 480), out=(240, 160)),
    "lp_even_segments": dict(ov=dict(interpolation_alg=I_LINEAR, num_vertical_segments=6, adjust_kernel=0,
                                     kernel_height_scale_factor=2.5), inp=(640, 320), out=(96, 64)),
    "lp_big_kernels": dict(ov=dict(interpolation_alg=I_CUBIC, num_vertical_segments=41, num_horizontal_segments=3,
                                   min_kernel_half_height=2.0), inp=(800, 400), out=(96, 64)),
    "eac_tb_lanczos": dict(ov=dict(input_stereo_format=S_TB, output_stereo_format=S_TB, output_layout=L_EAC,
                                   interpolation_alg=I_LANCZOS4, num_horizontal_segments=4, num_vertical_segments=7),
                           inp=(512, 512), out=(192, 256)),
    "eac_mono_cubic": dict(ov=dict(output_layout=L_EAC, interpolation_alg=I_CUBIC, enable_low_pass_filter=0),
                           inp=(640, 320), out=(240, 160)),
    "tb_vflip": dict(ov=dict(input_stereo_format=S_TB, output_stereo_format=S_TB, vflip=1,
                             interpolation_alg=I_LINEAR, enable_low_pass_filter=0), inp=(256, 256), out=(96, 128)),
    "lr_stereo": dict(ov=dict(input_stereo_format=S_LR, output_stereo_format=S_LR, interpolation_alg=I_CUBIC,
                              num_vertical_segments=5, num_horizontal_segments=2), inp=(1024, 256), out=(384, 128)),
    "rotated": dict(ov=dict(fixed_yaw=33.0, fixed_pitch=-12.5, fixed_roll=7.0, interpolation_alg=I_CUBIC,
                            enable_low_pass_filter=0), inp=(512, 256), out=(192, 128)),
    "offcenter_adjust": dict(ov=dict(fixed_cube_offcenter_z=-0.3, fixed_cube_offcenter_x=0.1, interpolation_alg=I_CUBIC,
                                     num_horizontal_segments=6, num_vertical_segments=9), inp=(600, 300), out=(192, 128)),
    "offcenter_horizontal": dict(ov=dict(fixed_cube_offcenter_z=-0.3, is_horizontal_offset=1, fixed_yaw=10.0,
                                         interpolation_alg=I_LINEAR, enable_low_pass_filter=0),
                                 inp=(512, 256), out=(192, 128)),
    "cube_to_equirect": dict(ov=dict(input_layout=L_CUBE32, output_layout=L_EQUIRECT, interpolation_alg=I_CUBIC,
                                     enable_low_pass_filter=0), inp=(384, 256), out=(512, 256)),
    "equirect_to_equirect_rot": dict(ov=dict(output_layout=L_EQUIRECT, fixed_yaw=40.0, fixed_pitch=20.0,
                                             interpolation_alg=I_LANCZOS4, enable_low_pass_filter=0),
                                     inp=(512, 256), out=(256, 128)),
    "cube23_offcenter": dict(ov=dict(output_layout=L_CUBE23, fixed_cube_offcenter_z=-0.5, interpolation_alg=I_CUBIC,
                                     enable_low_pass_filter=0), inp=(512, 256), out=(128, 192)),
    "flat_fixed": dict(ov=dict(output_layout=L_FLAT, fixed_yaw=100.0, fixed_pitch=50.0, interpolation_alg=I_CUBIC,
                               enable_low_pass_filter=0), inp=(512, 256), out=(160, 120)),
    "scaled_2x2": dict(ov=dict(width_scale_factor=2.0, height_scale_factor=2.0, interpolation_alg=I_CUBIC,
                               enable_low_pass_filter=0), inp=(512, 256), out=(96, 64)),
    "scaled_fractional_lp": dict(ov=dict(width_scale_factor=1.5, height_scale_factor=1.25, interpolation_alg=I_LINEAR,
                                         num_vertical_segments=7, num_horizontal_segments=2), inp=(640, 320), out=(96, 64)),
    "scaled_3x1": dict(ov=dict(width_scale_factor=3.0, height_scale_factor=1.0, interpolation_alg=I_LANCZOS4,
                               enable_low_pass_filter=0), inp=(512, 256), out=(96, 64)),
    # scale factors below 1: cv::resize(INTER_AREA) ENLARGES (its bilinear variant, ref:770-776)
    "scaled_half": dict(ov=dict(width_scale_factor=0.5, height_scale_factor=0.5, interpolation_alg=I_CUBIC,
                                enable_low_pass_filter=0), inp=(512, 256), out=(192, 128)),
    "scaled_075_lp": dict(ov=dict(width_scale_factor=0.75, height_scale_factor=0.75, interpolation_alg=I_LINEAR,
                                  num_vertical_segments=7, num_horizontal_segments=2), inp=(640, 320), out=(192, 128)),
    "scaled_mixed": dict(ov=dict(width_scale_factor=0.5, height_scale_factor=2.0, interpolation_alg=I_LANCZOS4,
                                 enable_low_pass_filter=0), inp=(512, 256), out=(190, 126)),
    "barrel": dict(ov=dict(output_layout=L_BARREL, interpolation_alg=I_CUBIC, enable_low_pass_filter=0),
                   inp=(512, 256), out=(250, 100)),
    "barrel_split_linear": dict(ov=dict(output_layout=L_BARREL_SPLIT, interpolation_alg=I_LINEAR,
                                        enable_low_pass_filter=0), inp=(512, 256), out=(180, 120)),
}


def plan_record(m, segments, centre_column=False):
    """A plan as golden.json records it: hashes of the float map bit for bit, of the low-pass tile table (rectangle and
    kernel lengths per tile) and of the taps.  segments: [(left, top, width, height, kx, ky)] in the reference's order.
    centre_column also records the map without its centre column (side-by-side stereo outputs of odd width, DESIGN.md 7)."""
    from oracle.ref_harness import sha16
    bits = np.ascontiguousarray(m).view(np.uint32)
    rects = np.array([(*s[:4], len(s[4]), len(s[5])) for s in segments], np.int32).reshape(-1, 6)
    taps = np.concatenate([np.concatenate([s[4], s[5]]) for s in segments]) if segments else np.zeros(0, np.float32)
    rec = {"shape": list(m.shape[:2]), "map": sha16(bits), "tiles": sha16(rects), "taps": sha16(taps.astype(np.float32))}
    if centre_column:
        rec["map_but_centre"] = sha16(np.delete(bits, m.shape[1] // 2, axis=1))
    return rec


def chroma(dim):
    return ((dim[0] + 1) >> 1, (dim[1] + 1) >> 1)


def plane_dims(case, plane):
    """(in_w, in_h, out_w, out_h, plan_index) of image plane 0/1/2 for a case (vf_transform360.c:368-381)."""
    inp, out = case["inp"], case["out"]
    if plane == 0:
        return inp[0], inp[1], out[0], out[1], 0
    ci, co = chroma(inp), chroma(out)
    return ci[0], ci[1], co[0], co[1], 1
