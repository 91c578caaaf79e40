"""The libjxl-side integration, compiled: oracle/build_ref.py builds a third variant of the reference ("gpu")
from build-time patched copies of lib/jxl/dec_frame.cc / dec_group.cc (integration/patch_libjxl.py) whose hooks
call integration/libjxl_gpu_backend.h -> include/jxl_b200.h.  These tests drive it through the PUBLIC
JxlDecoder API (JxlDecoderSetParallelRunner + JxlDecoderSetImageOutBuffer, oracle/ref_harness.cc:
ref_decode_linear_f32 / ref_decode_native), i.e. exactly what djxl does.

  * without a CUDA device the patched decoder must behave like the stock one (CPU path, same bytes);
  * with the SIMT-emulated product library preloaded (tests/emu) the whole hand-off runs on the CPU:
    eligibility, pinned group-major storage, kDontDraw entropy decode, row-wise submit, frame_finish;
  * on a GPU (-m gpu) the same through the real library, pixels within the conformance tolerance.
"""
import os
import subprocess
import sys
from pathlib import Path

import numpy as np
import pytest

import jxl_workload as wl
from oracle import build_ref

ROOT = Path(__file__).resolve().parents[1]
HAVE_REF_TREE = build_ref.reference_present()

# peak error of linear RGB in [0,1] against the stock CPU decoder (ISO 18181-3 tooling default is 1e-3,
# tools/conformance/tooling_test.sh:49-50; the reference's fast-vs-simple pipeline bound is 2e-4)
TOL_PEAK = 2e-5


def need_gpu_variant():
    from oracle import ref
    if not ref.available("gpu"):
        if HAVE_REF_TREE:
            pytest.fail("oracle/_ref/libjxl_ref_harness_gpu.so missing although the reference is present: "
                        "run `python oracle/build_ref.py` (after building libjxl_b200.so)")
        pytest.skip("integrated reference variant not built (no reference source tree)")
    return ref


CHILD = r"""
import ctypes, os, sys, json
import numpy as np
sys.path.insert(0, {root!r})
mode = sys.argv[1]
if mode == "emu":
    from tests.emu import build_emu
    ctypes.CDLL(str(build_emu.build()), mode=ctypes.RTLD_GLOBAL)   # jxlgpu_* resolve to the emulated library
import jxl_workload as wl
from oracle import ref
res = {{}}
for case in {cases!r}:
    w, h, dist, epf, fmt = case[:5]
    rs = case[5] if len(case) > 5 else -1          # frame_header.upsampling (JXL_ENC_FRAME_SETTING_RESAMPLING)
    img = wl.synth_image(w, h, seed=w + h)
    if fmt == "jpeg":      # a 4:4:4 JPEG recompressed losslessly: YCbCr frame, the application gets 8-bit pixels
        import io
        from PIL import Image
        b = io.BytesIO()
        Image.fromarray(img).save(b, format="JPEG", quality=int(dist), subsampling=0)
        data = ref.encode_jpeg(b.getvalue(), 4)
        fmt = "u8"
    else:
        data = ref.encode_rgb8(img, dist, 7, -1, epf, 4, resampling=rs)
    ref.use_variant("default")
    dec = (lambda: ref.decode_linear_f32(data, 4)) if fmt == "f32" else (lambda: ref.decode_native(data, (h, w, 3), np.uint8, 4))
    want = dec()
    ref.use_variant("gpu")
    before = ref.gpu_frames_taken()
    got = dec()
    taken = ref.gpu_frames_taken() - before
    d = np.abs(got.astype(np.float64) - want.astype(np.float64))
    res[f"{{w}}x{{h}}-d{{dist}}-epf{{epf}}-{{case[4]}}-{{fmt}}" + (f"-rs{{rs}}" if rs > 0 else "")] = dict(taken=int(taken), peak=float(d.max()), differing=float((d != 0).mean()))
print("RESULT " + json.dumps(res))
"""


def run_child(mode, cases, sparse=True):
    code = CHILD.format(root=str(ROOT), cases=cases)
    env = dict(os.environ, JXLB_GPU_SPARSE="1" if sparse else "0")
    r = subprocess.run([sys.executable, "-c", code, mode], capture_output=True, text=True, timeout=1500, cwd=str(ROOT),
                       env=env)
    assert r.returncode == 0, r.stderr[-4000:]
    import json
    line = [l for l in r.stdout.splitlines() if l.startswith("RESULT ")][-1]
    return json.loads(line[7:])


def test_patch_anchors_match_the_reference(tmp_path):
    """integration/patch_libjxl.py applies cleanly (every anchor exactly once) to the reference as it is."""
    if not HAVE_REF_TREE:
        pytest.skip("no reference source tree")
    subprocess.check_call([sys.executable, str(ROOT / "integration" / "patch_libjxl.py"), str(build_ref.REF), str(tmp_path)])
    for name in ("dec_frame.cc", "dec_group.cc"):
        assert "jxlb_integration::" in (tmp_path / "lib" / "jxl" / name).read_text()


def test_patched_decoder_without_device_is_the_stock_decoder():
    import torch
    if torch.cuda.is_available():
        pytest.skip("a device is present: covered by the gpu test")
    ref = need_gpu_variant()
    img = wl.synth_image(520, 300, seed=9)
    data = ref.encode_rgb8(img, 1.0, 7, -1, -1, 4)
    try:
        ref.use_variant("default")
        want = ref.decode_linear_f32(data, 4)
        ref.use_variant("gpu")
        got = ref.decode_linear_f32(data, 4)
        assert ref.gpu_frames_taken() == 0          # no device: the hooks said "not mine"
    finally:
        ref.use_variant("default")
    assert np.array_equal(got, want)


@pytest.mark.timeout(1800)
@pytest.mark.parametrize("sparse", [True, False], ids=["sparse-lists", "dense-blocks"])
def test_patched_decoder_through_the_emulated_library(sparse):
    """.jxl bytes -> public JxlDecoder API -> patched FrameDecoder -> C ABI -> (emulated) kernels -> the
    application's buffer; compared with the stock decoder's pixels."""
    need_gpu_variant()
    import torch
    if torch.cuda.is_available():
        pytest.skip("a device is present: covered by the gpu test")
    cases = [(300, 200, 1.0, -1, "f32"), (520, 264, 2.0, 2, "f32"), (300, 200, 1.0, -1, "u8"),
             (600, 300, 1.0, -1, "f32", 2),               # an upsampled frame (resampling 2)
             (300, 200, 1.0, -1, "f32", 1 + (32 << 16)),  # photon noise ISO 3200 (frame flag kNoise)
             (300, 200, 90, -1, "jpeg")]                  # JPEG-origin frame (YCbCr colour transform), quality 90
    res = run_child("emu", cases if sparse else cases[1:3] + cases[4:5], sparse)
    for k, v in res.items():
        assert v["taken"] == 1, (k, v)               # the frame really went through the backend
        if "-u8" in k:                         # the application's default: 8-bit sRGB, dithered
            assert v["peak"] <= 1 and v["differing"] < 1e-3, (k, v)
        else:
            assert v["peak"] <= TOL_PEAK, (k, v)


@pytest.mark.timeout(1800)
def test_progressive_frames_accumulate_in_the_dense_blocks():
    """A frame with several AC passes (JXL_ENC_FRAME_SETTING_PROGRESSIVE_AC; lib/jxl/dec_group.cc:219,335-338 adds
    every pass into the stored coefficients) goes to the backend too: the passes accumulate in the pinned dense
    blocks (zero-filled before a group's first pass only), the group is handed over after its last pass; the
    sparse lists (each position once) are not used for such frames."""
    need_gpu_variant()
    import torch
    mode = "gpu" if torch.cuda.is_available() else "emu"
    for sparse in (True, False):       # JXLB_GPU_SPARSE=1 must fall back to dense for this frame by itself
        res = run_child(mode, [(300, 200, 1.0, -1, "f32", 1 + 256), (520, 264, 2.0, 2, "f32", 1 + 256)], sparse)
        for k, v in res.items():
            assert v["taken"] == 1 and v["peak"] <= TOL_PEAK, (k, v)


@pytest.mark.gpu
@pytest.mark.timeout(1800)
@pytest.mark.parametrize("sparse", [True, False], ids=["sparse-lists", "dense-blocks"])
def test_patched_decoder_on_the_gpu(sparse):
    """sparse: the patched entropy decoder (lib/jxl/dec_group.cc:515-534) appends non-zero coefficients to
    per-thread lists that go to jxlgpu_submit_groups_sparse; dense: pinned [group][3][65536] blocks."""
    need_gpu_variant()
    res = run_child("gpu", [(1000, 700, 1.0, -1, "f32"), (2048, 1100, 2.0, 2, "f32"), (777, 333, 0.5, 0, "f32"),
                            (1500, 900, 4.0, 3, "f32"), (1000, 700, 1.0, -1, "u8"),
                            (1400, 900, 1.0, -1, "f32", 2), (2200, 1100, 1.0, -1, "u8", 4),   # upsampled frames
                            (1000, 700, 1.0, -1, "f32", 1 + (32 << 16)), (1400, 900, 1.0, -1, "f32", 2 + (64 << 16)),   # noise
                            (1000, 700, 85, -1, "jpeg")],   # JPEG-origin
                           sparse)
    for k, v in res.items():
        assert v["taken"] == 1, (k, v)
        if "-u8" in k:
            assert v["peak"] <= 1 and v["differing"] < 1e-3, (k, v)
        else:
            assert v["peak"] <= TOL_PEAK, (k, v)
