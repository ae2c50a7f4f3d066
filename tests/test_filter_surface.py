"""Filter-level drop-in: the reference's UNMODIFIED ffmpeg filter source (Transform360/vf_transform360.c), compiled
against the libavfilter stand-in oracle/ffshim and driven by oracle/ff_driver.c, linked with
  * the reference library (oracle/_ref/libt360ref.so + cv2)            -> variant "ref"
  * the product          (transform360_b200/lib/libTransform360.so)    -> variant "b200".
Same filter object code, same option strings; only libTransform360 differs.  Both variants are built from the reference's
filter source (make -C oracle ref), so the tests that use them skip where that source is absent.  The product's own
CUDA-frame filter is checked against the sizes and frames the reference filter gave, recorded in tests/golden/golden.json."""
import numpy as np
import pytest

from oracle import c_oracle as co
from oracle import ff_harness as ff
from oracle import ref_harness as rh

needs_filters = pytest.mark.skipif(not (ff.available("ref") and ff.available("b200")), reason="oracle/_ref filter objects not built")


def yuv_noise_frame(w, h):
    return [co.noise_plane(w, h, 0, 3), co.noise_plane((w + 1) // 2, (h + 1) // 2, 1, 3), co.noise_plane((w + 1) // 2, (h + 1) // 2, 2, 3)]


@needs_filters
def test_option_table_and_config_output_through_the_product_headers():
    """No GPU needed: defaults, named constants, ranges and the output-size rules of config_output (vf:167-304)."""
    f = ff.Filter("b200", "cube_edge_length=70", 512, 256)  # rounded down to a multiple of 16 (vf:213) -> 3*64 x 2*64
    assert (f.out_w, f.out_h) == (192, 128)
    f = ff.Filter("b200", "input_stereo_format=TB:cube_edge_length=100", 512, 512)  # TB output doubles the height (vf:293)
    assert (f.out_w, f.out_h) == (288, 384)
    f = ff.Filter("b200", "max_cube_edge_length=1000", 7680, 3840)  # edge = in_w / 4 capped, multiple of 16 (vf:198-213)
    assert (f.out_w, f.out_h) == (2976, 1984)
    f = ff.Filter("b200", "output_layout=eac_32:w=300:h=200", 512, 256)  # non-cubemap layouts take w/h (vf:224-291)
    assert (f.out_w, f.out_h) == (300, 200)
    f = ff.Filter("b200", "output_layout=cubemap_23_offcenter:cube_edge_length=64", 512, 256)
    assert (f.out_w, f.out_h) == (128, 192)
    for bad in ("interpolation_alg=bogus", "num_vertical_segments=1", "nonexistent=1"):
        with pytest.raises(ValueError):
            ff.Filter("b200", bad, 512, 256)
    # the two builds agree on every size decision
    for args, dims in (("cube_edge_length=333", (1920, 960)), ("input_stereo_format=LR:cube_edge_length=96", (2048, 256))):
        a, b = ff.Filter("ref", args, *dims), ff.Filter("b200", args, *dims)
        assert (a.out_w, a.out_h) == (b.out_w, b.out_h)


@needs_filters
@pytest.mark.gpu
@pytest.mark.parametrize("args,dims", [
    ("cube_edge_length=64:interpolation_alg=cubic:enable_low_pass_filter=0", (512, 256)),
    ("cube_edge_length=80:num_vertical_segments=15:num_horizontal_segments=8", (960, 480)),                    # filter defaults: cubic + low-pass
    ("input_stereo_format=TB:output_layout=eac_32:w=192:h=128:interpolation_alg=lanczos4:num_vertical_segments=7", (512, 512)),
    ("cube_edge_length=64:yaw=33:pitch=-12.5:roll=7:interpolation_alg=linear:enable_low_pass_filter=0", (512, 256)),
    ("cube_edge_length=48:width_scale_factor=2:height_scale_factor=2:enable_low_pass_filter=0", (512, 256)),
    ("input_layout=cubemap_32:output_layout=equirect:w=512:h=256:enable_low_pass_filter=0", (384, 256)),
])
def test_unmodified_reference_filter_gives_identical_frames_with_either_library(args, dims):
    import torch
    if not torch.cuda.is_available():
        pytest.fail("needs the B200 box")
    w, h = dims
    planes = yuv_noise_frame(w, h)
    ref, b200 = ff.Filter("ref", args, w, h), ff.Filter("b200", args, w, h)
    assert (ref.out_w, ref.out_h) == (b200.out_w, b200.out_h)
    for frame in range(2):  # the first frame also runs generate_map (vf:346-352)
        want, got = ref.filter(planes), b200.filter(planes)
        for p in range(3):
            assert np.array_equal(got[p], want[p]), f"plane {p} of frame {frame} differs ({args})"
    ref.close()
    b200.close()


# ---- the product's own CUDA-frame filter (transform360_b200/filter/vf_transform360_cuda.c) ----------------------------
needs_cuda_filter = pytest.mark.skipif(not ff.available("cuda"), reason="oracle/_ref/libvf_t360_cuda.so not built")

SIZE_CASES = [("cube_edge_length=70", (512, 256)), ("input_stereo_format=TB:cube_edge_length=100", (512, 512)),
              ("max_cube_edge_length=1000", (7680, 3840)), ("output_layout=eac_32:w=300:h=200", (512, 256)),
              ("output_layout=cubemap_23_offcenter:cube_edge_length=64", (512, 256)), ("cube_edge_length=333", (1920, 960)),
              ("input_stereo_format=LR:cube_edge_length=96", (2048, 256)), ("output_layout=EAC_32:cube_edge_length=64", (640, 320)),
              ("input_stereo_format=lr:output_stereo_format=mono:output_layout=barrel:w=250:h=100", (1024, 128))]


def size_key(args, dims):
    return f"{args} {dims[0]}x{dims[1]}"


@needs_cuda_filter
def test_cuda_filter_option_table_and_output_size_without_a_device(golden):
    """transform360_cuda takes the reference filter's option strings (vf:407-987) and decides the same output size
    (vf:167-304) as the reference filter did (golden.json "reference_runs"); graph configuration needs no GPU (the
    sampling plans wait for the first frame, like vf:346-352)."""
    sizes = golden["reference_runs"]["filter_sizes"]
    for args, dims in SIZE_CASES:
        f = ff.CudaFilter(args, *dims, device=False)
        assert [f.out_w, f.out_h] == sizes[size_key(args, dims)], args
        f.close()
    assert (ff.CudaFilter("output_layout=eac_32:size=300x200", 512, 256, device=False).out_w) == 300  # honoured here (see the file header)
    for bad in ("interpolation_alg=bogus", "num_vertical_segments=1", "nonexistent=1", "yaw=400", "output_layout=eac_32:w=300",
                "output_layout=eac_32:w=300:h=200:size=30x20", "output_layout=equirect"):
        with pytest.raises(ValueError):
            ff.CudaFilter(bad, 512, 256, device=False)
    with pytest.raises(ValueError):  # planar 8-bit only
        ff.CudaFilter("cube_edge_length=64", 512, 256, sw_format=ff.AV_PIX_FMT_NV12, device=False)


@needs_cuda_filter
def test_cuda_filter_defaults_are_the_reference_filters():
    """Every option the reference filter's table has exists here with the same default: an empty argument string leaves
    both private contexts describing the same transform (checked through the sizes and, on the GPU, the pixels)."""
    import re
    from pathlib import Path
    src = (Path(__file__).resolve().parents[1] / "transform360_b200" / "filter" / "vf_transform360_cuda.c").read_text()
    names = set(re.findall(r'(?:TEXT|INT|REAL)\("([a-z_0-9]+)"', src))
    expected = {"w", "width", "h", "height", "size", "s", "is_horizontal_offset", "cube_edge_length", "max_cube_edge_length", "max_output_h",
                "max_output_w", "input_stereo_format", "output_stereo_format", "input_layout", "output_layout", "vflip", "input_expand_coef",
                "expand_coef", "yaw", "pitch", "roll", "hfov", "vfov", "cube_offcenter_x", "cube_offcenter_y", "cube_offcenter_z",
                "interpolation_alg", "width_scale_factor", "height_scale_factor", "enable_low_pass_filter", "enable_multi_threading",
                "num_vertical_segments", "num_horizontal_segments", "kernel_height_scale_factor", "min_kernel_half_height",
                "max_kernel_half_height", "adjust_kernel", "kernel_adjust_factor"}
    assert expected <= names and names - expected == {"sync"}


CUDA_FRAME_CASES = [
    ("cube_edge_length=64:interpolation_alg=cubic:enable_low_pass_filter=0", (512, 256), ""),
    ("cube_edge_length=80:num_vertical_segments=15:num_horizontal_segments=8", (960, 480), ""),
    ("input_stereo_format=TB:output_layout=eac_32:w=192:h=128:interpolation_alg=lanczos4:num_vertical_segments=7", (512, 512), ":sync=0"),
    ("cube_edge_length=64:yaw=33:pitch=-12.5:roll=7:interpolation_alg=linear:enable_low_pass_filter=0", (512, 256), ""),
    ("cube_edge_length=48:width_scale_factor=2:height_scale_factor=2:enable_low_pass_filter=0", (512, 256), ":sync=0"),
    ("input_layout=cubemap_32:output_layout=equirect:w=512:h=256:enable_low_pass_filter=0", (384, 256), ""),
    ("output_layout=barrel:w=320:h=128:interpolation_alg=cubic", (640, 320), ""),
]


@needs_cuda_filter
@pytest.mark.gpu
@pytest.mark.parametrize("args,dims,extra", CUDA_FRAME_CASES)
def test_cuda_frame_filter_matches_the_reference_filter(args, dims, extra, golden):
    """Device planes in, device planes out, whole frame per call on the device context's stream; the frames are those the
    reference's software filter (reference object code + cv2) gave for the same option string (golden.json
    "reference_runs", make_golden.py)."""
    import torch
    if not torch.cuda.is_available():
        pytest.fail("needs the B200 box")
    w, h = dims
    planes = yuv_noise_frame(w, h)
    want = golden["reference_runs"]["filter_frames"][args]
    stream = torch.cuda.Stream()
    gpu = ff.CudaFilter(args + extra, w, h, stream=stream)
    assert [gpu.out_w, gpu.out_h] == want["size"]
    # decoder surfaces are pitched: 256-byte rows with the plane in the first columns
    dev = []
    for p in planes:
        pitch = (p.shape[1] + 255) // 256 * 256
        store = torch.zeros((p.shape[0], pitch), dtype=torch.uint8, device="cuda")
        store[:, :p.shape[1]] = torch.from_numpy(p).cuda()
        dev.append(store[:, :p.shape[1]])
    torch.cuda.synchronize()
    for frame in range(3):
        got = gpu.filter(dev, out_pitch_pad=48)
        stream.synchronize()
        for p in range(3):
            assert list(got[p].shape) == want["shapes"][p]
            assert rh.sha16(got[p].cpu().numpy()) == want["planes"][p], f"plane {p} of frame {frame} differs ({args})"
            assert bool((gpu.last_store[p][:, got[p].shape[1]:] == 0xA5).all()), "wrote beyond the plane's width"
    gpu.close()


@needs_cuda_filter
@pytest.mark.gpu
def test_cuda_frame_filter_gray8_and_refusals(golden):
    import torch
    if not torch.cuda.is_available():
        pytest.fail("needs the B200 box")
    w, h = 512, 256
    y = co.noise_plane(w, h, 0, 5)
    gpu = ff.CudaFilter("cube_edge_length=64:interpolation_alg=cubic:enable_low_pass_filter=0", w, h, sw_format=ff.AV_PIX_FMT_GRAY8)
    got = gpu.filter([torch.from_numpy(y).cuda()])
    torch.cuda.synchronize()
    want = golden["reference_runs"]["gray8"]  # the reference's transform of the same plane at the same output size
    assert [gpu.out_w, gpu.out_h] == want["size"]
    assert rh.sha16(got[0].cpu().numpy()) == want["out_sha"]
    # a frame pool that has nothing to hand out: ENOMEM surfaces, nothing crashes
    rc = gpu.L.t360f_filter_cuda(gpu.h, (ff.C.c_void_p * 1)(got[0].data_ptr()), (ff.C.c_int * 1)(w), (ff.C.c_void_p * 1)(None), (ff.C.c_int * 1)(0))
    assert rc == -12
    gpu.close()
