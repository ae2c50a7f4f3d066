#!/usr/bin/env python
"""Generates tests/golden/golden.json from THE REFERENCE ITSELF, run in this container:
``oracle/_ref/libt360ref.so`` (unmodified /root/reference sources + oracle/shim) driving cv2 4.13.0.

    python tests/golden/make_golden.py            # small cases (+ cfg1), reference_runs
    python tests/golden/make_golden.py --full     # also cfg2/cfg3/cfg4 luma known answers

Needs the reference's sources (to build oracle/_ref: make -C oracle ref) and cv2; the output is committed so that the
tests do not.  Input planes are the integer-hash ``noise`` generator of SURVEY.md 8(d); plane p of a case uses
noise(w, h, plane=p, frame=0).  "reference_runs" holds what further tests compare with: the reference run on the inputs
those tests define (other seeds, planes, random contexts, the ffmpeg filter), plans as cases.plan_record hashes and
pixels as sha16.
"""
import argparse
import json
import sys
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parents[2]
sys.path.insert(0, str(ROOT))

from oracle import ref_harness as rh  # noqa: E402
from tests.golden.cases import FULL, SMALL, plan_record, plane_dims  # noqa: E402


def run_case(name, case, planes=(0, 1)):
    ctx = rh.default_context(**case["ov"])
    ref = rh.RefTransform(ctx)
    rec = {"planes": {}}
    for plane in planes:
        iw, ih, ow, oh, idx = plane_dims(case, plane)
        assert ref.generate_map(iw, ih, ow, oh, idx)
        m = ref.map(idx)
        segs = ref.segments(idx)
        taps = np.concatenate([np.concatenate([s[4], s[5]]) for s in segs]) if segs else np.zeros(0, np.float32)
        rects = np.array([s[:4] for s in segs], np.int32) if segs else np.zeros((0, 4), np.int32)
        src = rh.noise_plane(iw, ih, plane=plane, frame=0)
        barrel = ctx.output_layout in (rh.LAYOUT_BARREL, rh.LAYOUT_BARREL_SPLIT)
        out = ref.transform_plane(src, ow, oh, idx, image_plane=plane, prefill=0 if not barrel else 7)
        rec["planes"][str(plane)] = {
            "dims": [iw, ih, ow, oh, idx],
            "map_fnv": rh.fnv1a64(m),
            "map_corners": [float(m[0, 0, 0]), float(m[0, 0, 1]), float(m[-1, -1, 0]), float(m[-1, -1, 1])],
            "nsegs": len(segs),
            "rects_fnv": rh.fnv1a64(rects),
            "taps_fnv": rh.fnv1a64(taps),
            "ntaps": int(taps.size),
            "src_sha": rh.sha16(src),
            "out_sha": rh.sha16(out),
            "out_sum": int(out.sum(dtype=np.int64)),
            "out_head": [int(v) for v in out[0, :8]],
        }
        print(name, plane, rec["planes"][str(plane)]["out_sha"], rec["planes"][str(plane)]["out_sum"], flush=True)
    ref.close()
    return rec


def ref_plan(ref, idx, centre_column=False):
    return plan_record(ref.map(idx), ref.segments(idx), centre_column)


def reference_runs():
    from oracle import ff_harness as ff
    from tests import test_filter_surface as tf
    from tests import test_host_plan as th
    from tests import test_oracle_pin as to
    runs = {}

    runs["scale_below_one"] = []
    for ov, (iw, ih, ow, oh) in to.SCALE_BELOW_ONE:
        ctx = rh.default_context(**ov)
        ref = rh.RefTransform(ctx)
        shas = []
        for idx in (0, 1):
            assert ref.generate_map(iw, ih, ow, oh, idx)
            src = rh.noise_plane(iw, ih, plane=idx, frame=5)
            shas.append(rh.sha16(ref.transform_plane(src, ow, oh, idx, image_plane=idx, prefill=to._prefill(ctx))))
        runs["scale_below_one"].append(shas)
        ref.close()

    runs["live_cases"] = {}
    for name in to.LIVE_CASES:
        case = SMALL[name]
        ctx = rh.default_context(**case["ov"])
        ref = rh.RefTransform(ctx)
        rec = {}
        for plane in (0, 2):
            iw, ih, ow, oh, idx = plane_dims(case, plane)
            assert ref.generate_map(iw, ih, ow, oh, idx)
            src = rh.noise_plane(iw, ih, plane=plane, frame=17)
            out = ref.transform_plane(src, ow, oh, idx, image_plane=plane, prefill=to._prefill(ctx))
            rec[str(plane)] = {"plan": ref_plan(ref, idx), "out_sha": rh.sha16(out)}
        runs["live_cases"][name] = rec
        ref.close()

    runs["e2e_sweep"] = {}
    for seed in (11, 12):
        recs = []
        for ov, (iw, ih, ow, oh), idx in to._e2e_sweep_cases(seed):
            ctx = rh.default_context(**ov)
            ref = rh.RefTransform(ctx)
            want = None  # the reference refused the plan or the frame
            if ref.generate_map(iw, ih, ow, oh, idx):
                src = rh.noise_plane(iw, ih, plane=idx, frame=seed)
                try:
                    want = rh.sha16(ref.transform_plane(src, ow, oh, idx, image_plane=idx, prefill=to._prefill(ctx)))
                except RuntimeError:
                    pass
            recs.append(want)
            ref.close()
        runs["e2e_sweep"][str(seed)] = recs

    ref = rh.RefTransform(rh.default_context(**th.ODD_PARAMETERS))
    assert ref.generate_map(700, 350, 300, 200, 0)
    runs["odd_parameters"] = ref_plan(ref, 0)
    ref.close()

    runs["plan_sweep"] = {}
    for seed in (1, 2, 3):
        recs = []
        for ov, dims in th._plan_sweep_cases(seed):
            ref = rh.RefTransform(rh.default_context(**ov))
            recs.append(ref_plan(ref, 0, centre_column=True) if ref.generate_map(*dims, 0) else None)
            ref.close()
        runs["plan_sweep"][str(seed)] = recs

    runs["non_positive_horizontal_segments"] = {}
    for nh, adjust in th.NON_POSITIVE_HORIZONTAL_SEGMENTS:
        ref = rh.RefTransform(rh.default_context(**th._non_positive_overrides(nh, adjust)))
        assert ref.generate_map(320, 160, 96, 64, 0)
        runs["non_positive_horizontal_segments"][f"{nh},{adjust}"] = ref_plan(ref, 0)
        ref.close()

    # the reference's ffmpeg filter (variant "ref": its unmodified filter source around the reference library)
    runs["filter_sizes"] = {}
    for args, dims in tf.SIZE_CASES:
        f = ff.Filter("ref", args, *dims)
        runs["filter_sizes"][tf.size_key(args, dims)] = [f.out_w, f.out_h]
        f.close()
    runs["filter_frames"] = {}
    for args, (w, h), _ in tf.CUDA_FRAME_CASES:
        f = ff.Filter("ref", args, w, h)
        outs = f.filter(tf.yuv_noise_frame(w, h))
        runs["filter_frames"][args] = {"size": [f.out_w, f.out_h], "shapes": [list(o.shape) for o in outs],
                                       "planes": [rh.sha16(o) for o in outs]}
        f.close()
    # test_cuda_frame_filter_gray8_and_refusals: the luma plane of its filter arguments, through the reference library
    w, h = 512, 256
    f = ff.Filter("ref", "cube_edge_length=64:interpolation_alg=cubic:enable_low_pass_filter=0", w, h)
    ow, oh = f.out_w, f.out_h
    f.close()
    ref = rh.RefTransform(rh.default_context(interpolation_alg=2, enable_low_pass_filter=0))
    assert ref.generate_map(w, h, ow, oh, 0)
    runs["gray8"] = {"size": [ow, oh], "out_sha": rh.sha16(ref.transform_plane(rh.noise_plane(w, h, 0, 5), ow, oh, 0))}
    ref.close()
    return runs


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--full", action="store_true")
    args = ap.parse_args()
    path = Path(__file__).with_name("golden.json")
    gold = json.loads(path.read_text()) if path.exists() else {}
    gold.setdefault("_meta", {})
    import cv2
    import platform
    gold["_meta"] = {"cv2": cv2.__version__, "glibc": platform.libc_ver()[1], "generator": "tests/golden/make_golden.py",
                     "note": "hashes depend on host libm (sinf/cosf/expf/atan2f/asinf) -- regenerate if the image changes"}
    gold.setdefault("small", {})
    for name, case in SMALL.items():
        gold["small"][name] = run_case(name, case)
    gold["reference_runs"] = reference_runs()
    if args.full:
        gold.setdefault("full", {})
        for name in ("cfg2", "cfg3", "cfg4"):
            gold["full"][name] = run_case(name, FULL[name], planes=(0,))
    path.write_text(json.dumps(gold, indent=1, sort_keys=True) + "\n")


if __name__ == "__main__":
    main()
