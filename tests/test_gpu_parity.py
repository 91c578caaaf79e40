"""-m gpu: the CUDA path, called through the C ABI (include/jxl_b200.h), against the oracle and
the committed reference goldens.  Bar: bit-exact vs oracle/jxl_oracle.c in exact-reciprocal mode
(float work whose operation order is pinned); vs the reference pixels the stated tolerance
(the reference's AdjustQuantBias uses a 12-bit rcpps: quantizer-inl.h:62-64)."""
import numpy as np
import pytest

import jxl_workload as wl
from libjxl_b200 import abi, pipeline, sharding
from tests import support

pytestmark = [pytest.mark.gpu, pytest.mark.usefixtures("built")]


@pytest.fixture(scope="module", params=["two-kernel", "fused"])
def pipe(request):
    """Both device paths: plan -> IDCT kernels -> strip filter (default) and the fused decode kernel
    (JXLGPU_FUSED=1, read when the context is created)."""
    import os
    old = os.environ.get("JXLGPU_FUSED")
    os.environ["JXLGPU_FUSED"] = "1" if request.param == "fused" else "0"
    try:
        p = pipeline.TransformPipeline(device=0, num_host_threads=4)
        yield p
        p.close()
    finally:
        if old is None:
            os.environ.pop("JXLGPU_FUSED", None)
        else:
            os.environ["JXLGPU_FUSED"] = old


def oracle(desc, coeffs):
    from oracle import cpu
    return cpu.render_frame(desc, coeffs, rcp_mode=0)


def assert_same(got, want, what=""):
    assert got.shape == want.shape and got.dtype == want.dtype
    if got.dtype != np.float32:   # packed output formats: compare the stored code values
        if got.dtype == np.float16:
            got, want = got.view(np.uint16), want.view(np.uint16)
        if not np.array_equal(got, want):
            d = np.abs(got.astype(np.int64) - want.astype(np.int64))
            idx = np.unravel_index(np.argmax(d), d.shape)
            raise AssertionError(f"{what}: max code diff {d.max()} at {idx} ({got[idx]} vs {want[idx]}), "
                                 f"{int((d > 0).sum())} of {d.size} differ")
        return
    if not np.array_equal(got, want):
        d = np.abs(got - want)
        idx = np.unravel_index(np.argmax(d), d.shape)
        raise AssertionError(f"{what}: max|diff| {d.max():.3e} at {idx} ({got[idx]} vs {want[idx]}), "
                             f"{int((d > 0).sum())} of {d.size} differ, {support.ulp_diff(got, want)} ulp")


@pytest.mark.parametrize("w,h,ac_type", [(520, 264, abi.AC_INT16), (2048, 1032, abi.AC_INT16),
                                          (777, 523, abi.AC_INT32)])
def test_all_strategies_bit_exact(pipe, w, h, ac_type):
    desc, coeffs = wl.synthetic_frame(w, h, seed=w + h, ac_type=ac_type)
    if w >= 2048:
        assert len(wl.strategy_histogram(desc.ac_strategy)) == 27
    assert_same(pipe.decode_frame(desc, coeffs), oracle(desc, coeffs), "full chain")


@pytest.mark.parametrize("mask", [0, 1, 2, 4, 8, 16, 1 | 4, 1 | 4 | 8, 1 | 2 | 4 | 8, 31])
def test_stage_taps_bit_exact(pipe, mask):
    desc, coeffs = wl.synthetic_frame(600, 300, seed=mask)
    desc.stage_mask = abi.STAGE_EXPLICIT | mask
    desc.out_format = abi.OUT_PLANAR_F32
    assert_same(pipe.decode_frame(desc, coeffs), oracle(desc, coeffs), f"mask {mask}")


@pytest.mark.parametrize("gab", [0, 1])
@pytest.mark.parametrize("epf_iters", [0, 1, 2, 3])
@pytest.mark.parametrize("w,h", [(1000, 700), (261, 1031)])
def test_production_stage_chains(pipe, gab, epf_iters, w, h):
    """The eight stage chains PreparePipeline can build (dec_cache.cc:151-170) run through the
    row-streaming strip kernel; sizes chosen so that strips have left/right edge handling, several
    strips and several vertical segments."""
    desc, coeffs = wl.synthetic_frame(w, h, seed=gab * 10 + epf_iters, gab=gab, epf_iters=epf_iters)
    assert_same(pipe.decode_frame(desc, coeffs), oracle(desc, coeffs), f"gab={gab} epf={epf_iters}")


@pytest.mark.parametrize("strategy", range(27))
def test_single_strategy_frames(pipe, strategy):
    """One strategy at a time (plus 8x8 filler where it does not tile): isolates each transform."""
    desc, coeffs = wl.synthetic_frame(512, 256, seed=100 + strategy, strategies=f"{strategy},0", gab=0,
                                      epf_iters=0)
    desc.stage_mask = abi.STAGE_EXPLICIT | 0
    desc.out_format = abi.OUT_PLANAR_F32
    assert wl.strategy_histogram(desc.ac_strategy).get(abi.STRATEGY_NAMES[strategy], 0) > 0
    assert_same(pipe.decode_frame(desc, coeffs), oracle(desc, coeffs), abi.STRATEGY_NAMES[strategy])


@pytest.mark.parametrize("w,h", [(1, 1), (5, 3), (8, 8), (9, 17), (255, 257), (256, 256), (264, 72), (31, 700)])
def test_ragged_and_tiny_sizes(pipe, w, h):
    """Mirror padding about the true image size (image_ops.h:184-196), partial blocks/groups."""
    desc, coeffs = wl.synthetic_frame(w, h, seed=w * 1000 + h)
    assert_same(pipe.decode_frame(desc, coeffs), oracle(desc, coeffs), f"{w}x{h}")


def test_zero_coefficients_and_extremes(pipe):
    desc, coeffs = wl.synthetic_frame(300, 200, seed=4)
    coeffs[:] = 0
    assert_same(pipe.decode_frame(desc, coeffs), oracle(desc, coeffs), "all-zero AC")
    coeffs[:, :, ::97] = 32767
    coeffs[:, :, 1::89] = -32768
    assert_same(pipe.decode_frame(desc, coeffs), oracle(desc, coeffs), "int16 extremes")


def test_int32_large_magnitudes(pipe):
    """int32 coefficients far beyond int16 (the Newton reciprocal in the dequantiser must stay
    correctly rounded for every magnitude, DESIGN.md §2)."""
    desc, coeffs = wl.synthetic_frame(300, 200, seed=8, ac_type=abi.AC_INT32)
    rng = np.random.default_rng(0)
    big = rng.integers(-(1 << 30), 1 << 30, coeffs.shape, dtype=np.int64).astype(np.int32)
    mask = rng.random(coeffs.shape) < 0.02
    coeffs = np.where(mask, big, coeffs).astype(np.int32)
    desc.stage_mask = abi.STAGE_EXPLICIT | 0      # post-IDCT XYB: keeps the huge values finite
    desc.out_format = abi.OUT_PLANAR_F32
    got = pipe.decode_frame(desc, coeffs)
    assert np.isfinite(got).all()
    assert_same(got, oracle(desc, coeffs), "int32 large magnitudes")


def test_golden_frame_against_reference_pixels(pipe):
    """Real bitstream (tests/golden/frame_small.npz): coefficients as the reference's entropy
    decoder produced them; pixels vs the reference decoder. Tolerances in absolute units."""
    desc, coeffs, g = support.golden_desc()
    got = pipe.decode_frame(desc, coeffs)
    assert_same(got, oracle(desc, coeffs), "golden frame vs oracle")
    peak = float(np.abs(got - g.decoded_default).max())
    rmse = float(np.sqrt(np.mean((got - g.decoded_default) ** 2)))
    assert peak <= 5e-5 and rmse <= 5e-6, (peak, rmse)   # conformance tooling default is 1e-3 / 1e-3
    for tap, mask in support.TAP_MASKS.items():
        desc.stage_mask = abi.STAGE_EXPLICIT | mask
        desc.out_format = abi.OUT_PLANAR_F32
        got = pipe.decode_frame(desc, coeffs)
        assert np.abs(got - g.taps[tap]).max() <= 2e-5, tap


PACKED = [abi.OUT_RGB_U8, abi.OUT_RGBA_U8, abi.OUT_RGB_U16, abi.OUT_RGB_F16]


@pytest.mark.parametrize("srgb", [0, abi.STAGE_SRGB])
@pytest.mark.parametrize("fmt", [abi.OUT_RGB_F32, abi.OUT_PLANAR_F32] + PACKED)
def test_output_stages_bit_exact(pipe, fmt, srgb):
    """sRGB transfer function (FromLinearStage<OpRgb>) and WriteToOutput packing fused into the
    filter kernel's store: identical bytes to the oracle, strip kernel (derived chain) and generic
    tile kernel (a chain outside the production set), odd width so rows are not 4-byte multiples."""
    if fmt in (abi.OUT_RGB_F32, abi.OUT_PLANAR_F32) and not srgb:
        pytest.skip("covered by the tests above")
    desc, coeffs = wl.synthetic_frame(773, 530, seed=fmt * 2 + (1 if srgb else 0))
    desc.out_format = fmt
    desc.stage_mask = srgb
    assert_same(pipe.decode_frame(desc, coeffs), oracle(desc, coeffs), "strip kernel")
    desc.stage_mask = abi.STAGE_EXPLICIT | abi.STAGE_GAB | abi.STAGE_EPF2 | abi.STAGE_XYB | srgb
    assert_same(pipe.decode_frame(desc, coeffs), oracle(desc, coeffs), "tile kernel")


@pytest.mark.parametrize("case", ["srgb_f32", "srgb_u8", "srgb_rgba8", "srgb_u16", "srgb_f16", "linear_u8",
                                  "linear_f16"])
def test_golden_frame_packed_outputs(pipe, case):
    """Real bitstream, the reference's own FromLinear + WriteToOutput bytes (tests/golden/
    outputs_small.npz): at most one code value off where the reference's 12-bit rcpps moved a sample
    across a rounding boundary; bit-exact against the oracle."""
    from tests.test_oracle_golden import OUTPUT_CASES
    fmt, mask = OUTPUT_CASES[case]
    desc, coeffs, _ = support.golden_desc(out_format=fmt, stage_mask=mask)
    got = pipe.decode_frame(desc, coeffs)
    assert_same(got, oracle(desc, coeffs), case)
    want = np.load(support.GOLDEN / "outputs_small.npz")[case]
    if got.dtype == np.float32:
        assert np.abs(got - want).max() <= 2e-5
        return
    if got.dtype == np.float16:
        got = got.view(np.uint16)
    d = np.abs(got.astype(np.int64) - want.astype(np.int64))
    if case.endswith("f16"):
        d = d[(got & 0x7fff) > 0x0400]
    assert d.max() <= 1 and (d != 0).mean() <= (2e-3 if got.dtype == np.uint8 else 5e-2)


def test_packed_output_streaming_and_bands(pipe):
    """8-bit sRGB output through the streaming path (rows copied back as they finish, shuffled
    submission) and rendered band by band: same bytes as the one-shot whole-frame call."""
    desc, coeffs = wl.synthetic_frame(901, 1300, seed=34)
    desc.out_format, desc.stage_mask = abi.OUT_RGB_U8, abi.STAGE_SRGB
    want = pipe.decode_frame(desc, coeffs)
    assert want.dtype == np.uint8 and want.shape == (1300, 901, 3)
    out = pipeline.pinned_array((desc.ysize, desc.xsize, 3), np.uint8)
    out[:] = 7
    order = np.random.default_rng(5).permutation(desc.num_groups)
    assert_same(pipe.decode_frame(desc, coeffs, out=out, order=order, stream_output=True), want, "streamed")
    rows = []
    for (y0, ny) in sharding.band_partition(desc.ysize_groups, 3):
        desc.band_y0_groups, desc.band_ny_groups = y0, ny
        pipe.set_device_coefficients(None)
        pipe.frame_begin(desc)
        for gidx in sharding.groups_needed(desc, y0, ny):
            pipe.submit_group(gidx, [coeffs[c, gidx] for c in range(3)])
        rows.append(pipe.frame_finish())
    desc.band_y0_groups = desc.band_ny_groups = 0
    assert_same(np.concatenate(rows, axis=0), want, "bands")


def test_band_sharded_equals_whole_frame(pipe):
    """Each band rendered separately (as a rank would, receiving only the groups it needs)
    concatenates to exactly the whole-frame result: sharding is invisible in the pixels."""
    desc, coeffs = wl.synthetic_frame(700, 1500, seed=21)     # 3 x 6 groups
    whole = pipe.decode_frame(desc, coeffs)
    for world in (2, 4):
        rows = []
        for (y0, ny) in sharding.band_partition(desc.ysize_groups, world):
            if ny == 0:
                continue
            desc.band_y0_groups, desc.band_ny_groups = y0, ny
            pipe.set_device_coefficients(None)
            pipe.frame_begin(desc)
            for gidx in sharding.groups_needed(desc, y0, ny):
                pipe.submit_group(gidx, [coeffs[c, gidx] for c in range(3)])
            rows.append(pipe.frame_finish())
        desc.band_y0_groups = desc.band_ny_groups = 0
        assert_same(np.concatenate(rows, axis=0), whole, f"world={world}")


def test_device_resident_entry_points(pipe):
    import torch
    desc, coeffs = wl.synthetic_frame(640, 520, seed=9)
    want = pipe.decode_frame(desc, coeffs)
    dev = torch.from_numpy(coeffs).cuda()
    out = torch.empty((desc.ysize, desc.xsize, 3), dtype=torch.float32, device="cuda")
    pipe.set_device_coefficients([dev[c].data_ptr() for c in range(3)])
    pipe.frame_begin(desc)
    before = pipe.launch_count()
    pipe.render_device(out.data_ptr(), desc.xsize * 12, torch.cuda.current_stream().cuda_stream)
    torch.cuda.synchronize()
    assert pipe.launch_count() - before == 6   # plan, idct_mid, idct_large rows + columns, idct8, filter
    assert_same(out.cpu().numpy(), want, "device-resident")
    pipe.set_device_coefficients(None)


def test_full_size_4096_against_oracle(pipe):
    """BASELINE config 2 size (4096x4096, all IDCT sizes + Gaborish + EPF): full compare, the
    oracle takes a few seconds with OpenMP."""
    desc, coeffs = wl.synthetic_frame(4096, 4096, seed=4096)
    got = pipe.decode_frame(desc, coeffs)
    assert np.isfinite(got).all()
    assert_same(got, oracle(desc, coeffs), "4096x4096")
    # determinism (work lists are filled with atomics; results must not depend on their order)
    assert_same(pipe.decode_frame(desc, coeffs), got, "second run")


def test_streaming_any_submission_order(pipe):
    """Groups may arrive in any order from the host's worker threads (FakeParallelRunner-style
    shuffle, render_pipeline_test.cc:254-255); rows are transformed / filtered / copied back as
    they complete. Result identical to the in-order run."""
    desc, coeffs = wl.synthetic_frame(900, 1300, seed=33)     # 4 x 6 groups
    want = pipe.decode_frame(desc, coeffs)
    rng = np.random.default_rng(123)
    for trial in range(3):
        order = rng.permutation(desc.num_groups)
        assert_same(pipe.decode_frame(desc, coeffs, order=order, stream_output=bool(trial % 2)), want,
                    f"shuffle {trial}")
    out = pipeline.pinned_array((desc.ysize, desc.xsize, 3), np.float32)
    out[:] = -1
    got = pipe.decode_frame(desc, coeffs, out=out, order=rng.permutation(desc.num_groups), stream_output=True)
    assert got is out
    assert_same(got, want, "pinned streamed output")


@pytest.mark.parametrize("ac_type", [abi.AC_INT16, abi.AC_INT32])
def test_sparse_submit_equals_dense(pipe, ac_type):
    """jxlgpu_submit_groups_sparse (non-zero lists + scatter kernel) produces the same pixels as the
    dense hand-off: all 27 strategies, ragged size, shuffled group order, streamed output; the int32
    frame carries values beyond 16 bits (the {pos, value} pair lists)."""
    desc, coeffs = wl.synthetic_frame(1100, 777, seed=77 + ac_type, ac_type=ac_type)
    if ac_type == abi.AC_INT32:
        coeffs = coeffs.copy()
        rng = np.random.default_rng(2)
        for c in range(3):
            g = rng.integers(0, desc.num_groups, 200)
            k = rng.integers(64, 4096, 200)
            coeffs[c, g, k] = rng.integers(-300000, 300000, 200)
        assert np.abs(coeffs).max() > 40000
    want = pipe.decode_frame(desc, coeffs)
    assert_same(pipe.decode_frame(desc, coeffs, sparse=True), want, "sparse, in order")
    order = np.random.default_rng(9).permutation(desc.num_groups).tolist()
    assert_same(pipe.decode_frame(desc, coeffs, sparse=True, order=order, stream_output=True), want, "sparse, shuffled")
    # a frame of zeros after a frame with content: the planes really are re-zeroed
    zeros = np.zeros_like(coeffs)
    assert_same(pipe.decode_frame(desc, zeros, sparse=True), pipe.decode_frame(desc, zeros), "all-zero frame")
    # mixing both hand-offs inside one frame
    pipe.set_device_coefficients(None)
    pipe.frame_begin(desc)
    xg = desc.xsize_groups
    keep = []
    for row in range(desc.ysize_groups):
        gs = list(range(row * xg, (row + 1) * xg))
        if row % 2:
            keep.append(pipe.make_sparse_batch(gs, coeffs, pinned=False))
            pipe.submit_sparse_batch(keep[-1])
        else:
            for g in gs:
                pipe.submit_group(g, [coeffs[c, g] for c in range(3)])
    assert_same(pipe.frame_finish(), want, "mixed")


def test_sparse_submit_errors(pipe):
    desc, coeffs = wl.synthetic_frame(300, 300, seed=1)          # int16 frame
    pipe.set_device_coefficients(None)
    pipe.frame_begin(desc)
    n, arr, buf, _ = pipe.make_sparse_batch([0], coeffs, pinned=False)
    arr[0].group_idx = 99
    with pytest.raises(pipeline.JxlGpuError):      # group index out of range
        pipe.submit_sparse_batch((n, arr))
    arr[0].group_idx = 0
    arr[0].n32[0] = 1
    arr[0].nz32[0] = buf.ctypes.data
    with pytest.raises(pipeline.JxlGpuError):      # wide values cannot go into int16 planes
        pipe.submit_sparse_batch((n, arr))
    arr[0].n32[0] = 0
    arr[0].n16[1] = 70000
    with pytest.raises(pipeline.JxlGpuError):      # more entries than the plane has coefficients
        pipe.submit_sparse_batch((n, arr))
    with pytest.raises(pipeline.JxlGpuError):      # the frame is still incomplete
        pipe.frame_finish()


def test_submit_errors(pipe):
    desc, coeffs = wl.synthetic_frame(300, 300, seed=1)
    pipe.set_device_coefficients(None)
    pipe.frame_begin(desc)
    with pytest.raises(pipeline.JxlGpuError):      # group index out of range
        pipe.submit_group(99, [coeffs[c, 0] for c in range(3)])
    with pytest.raises(pipeline.JxlGpuError):      # finishing with missing groups
        pipe.frame_finish()


@pytest.mark.parametrize("n,w,h", [(2, 1201, 531), (4, 600, 270), (8, 300, 130)])
@pytest.mark.parametrize("fmt,srgb", [(abi.OUT_RGB_F32, 0), (abi.OUT_RGB_U8, abi.STAGE_SRGB)])
def test_upsampling_bit_exact(pipe, n, w, h, fmt, srgb):
    """SURVEY.md §8f rank 4: UpsamplingStage (stage_upsampling.cc:51-271) 2x / 4x / 8x after the filters, fused with
    XYB -> RGB, transfer function and packing; the restatement it is compared with is pinned bit-exactly against
    the reference's own stage (tests/test_oracle_vs_reference.py::test_upsampling_stage_bit_exact)."""
    from tests.test_emulated_cuda import upsampled_frame
    desc, coeffs = upsampled_frame(n, w, h, seed=11 + n, fmt=fmt, srgb=srgb)
    assert_same(pipe.decode_frame(desc, coeffs), oracle(desc, coeffs), f"upsampling {n}x")


@pytest.mark.parametrize("rs", [2, 4, 8])
def test_upsampled_reference_frames(pipe, rs):
    """Frames the reference encoder made with resampling 2 / 4 / 8, entropy-decoded by the reference, rendered here,
    compared with the reference decoder's own pixels (tests/golden/vs_reference.npz.xz: the hand-off and the digest of
    the pixels of its -ffp-contract=off build, which the restatement in host-rcpss mode reproduces bit for bit)."""
    from oracle import cpu
    z = support.load_xz_npz(support.GOLDEN / "vs_reference.npz.xz")
    support.require_host_rcpss(z)
    d = support.load_dump(z, f"ups{rs}")
    desc = cpu.desc_from_dump(d)
    assert desc.upsampling == rs
    got = pipe.decode_frame(desc, d.coeffs)
    assert got.shape == (d.info.ysize_upsampled, d.info.xsize_upsampled, 3)
    assert_same(got, oracle(desc, d.coeffs), f"resampling {rs} vs oracle")
    desc.out_format = abi.OUT_PLANAR_F32
    want = cpu.render_frame(desc, d.coeffs, rcp_mode=1)
    assert support.digest(want) == z[f"ups{rs}.want"][0].tobytes()
    assert np.abs(got - np.moveaxis(want, 0, 2)).max() <= 2e-5       # vs the reference decoder (rcpps in AdjustQuantBias)


@pytest.mark.parametrize("n,w,h", [(1, 1201, 531), (2, 600, 270)])
@pytest.mark.parametrize("fmt,srgb", [(abi.OUT_RGB_F32, 0), (abi.OUT_RGB_U8, abi.STAGE_SRGB)])
def test_noise_bit_exact(pipe, n, w, h, fmt, srgb):
    """SURVEY.md §8f rank 4: noise generation + ConvolveNoise + AddNoise on the device (noise_gen_kernel, finish_px),
    alone and behind the upsampling; the restatement is pinned bit-exactly against the reference's stages
    (tests/test_oracle_vs_reference.py::test_noise_stages_bit_exact)."""
    from tests.test_emulated_cuda import NOISE_LUT, upsampled_frame
    if n > 1:
        desc, coeffs = upsampled_frame(n, w, h, seed=21 + n, fmt=fmt, srgb=srgb)
    else:
        desc, coeffs = wl.synthetic_frame(w, h, seed=21, epf_iters=1)
        desc.out_format, desc.stage_mask = fmt, srgb
    desc.noise, desc.noise_lut = 1, NOISE_LUT
    desc.visible_frame_index, desc.nonvisible_frame_index = 2, 5
    assert_same(pipe.decode_frame(desc, coeffs), oracle(desc, coeffs), f"noise, upsampling {n}")


@pytest.mark.parametrize("mode", ["ce", "sm", "kernel"])
def test_gather_mechanisms_on_one_device(mode, monkeypatch):
    """The multi-GPU gather (DESIGN.md §6) with the "peers" being three more buffers on this GPU: copy-engine copies
    per row chunk (default), peer_copy_kernel per row chunk (JXLGPU_GATHER=sm), replay inside the filter kernel
    (=kernel).  Every replica ends up identical to the local band, in an f32 and an 8-bit layout."""
    import torch
    if mode == "ce":
        monkeypatch.delenv("JXLGPU_GATHER", raising=False)
    else:
        monkeypatch.setenv("JXLGPU_GATHER", mode)
    p = pipeline.TransformPipeline(device=0, num_host_threads=1)
    try:
        for fmt, srgb, dt in ((abi.OUT_RGB_F32, 0, torch.float32), (abi.OUT_RGB_U8, abi.STAGE_SRGB, torch.uint8)):
            desc, coeffs = wl.synthetic_frame(1200, 1100, seed=40 + fmt, epf_iters=1)
            desc.out_format, desc.stage_mask = fmt, srgb
            want = oracle(desc, coeffs)
            dev = torch.from_numpy(coeffs).cuda()
            p.set_device_coefficients([dev[c].data_ptr() for c in range(3)])
            p.frame_begin(desc)
            bufs = [torch.zeros((desc.ysize, desc.xsize, 3), dtype=dt, device="cuda") for _ in range(4)]
            p.set_output_replicas([b.data_ptr() for b in bufs[1:]])
            try:
                p.render_device(bufs[0].data_ptr(), desc.out_row_bytes, torch.cuda.current_stream().cuda_stream)
                torch.cuda.synchronize()
            finally:
                p.set_output_replicas([])
                p.set_device_coefficients(None)
            for i, b in enumerate(bufs):
                assert_same(b.cpu().numpy(), want, f"{mode}: buffer {i}")
    finally:
        p.close()


@pytest.mark.parametrize("fmt", [abi.OUT_RGB_F32, abi.OUT_RGB_U8])
def test_ycbcr_colour_transform_bit_exact(pipe, fmt):
    """SURVEY.md §8f rank 4: JPEG-origin 4:4:4 frames -- kYCbCrStage (stage_ycbcr.cc:33-71) in the place of the opsin
    inverse; the restatement is pinned against the reference's stage and public decoder
    (tests/test_oracle_vs_reference.py::test_jpeg_origin_ycbcr_frames)."""
    desc, coeffs = wl.synthetic_frame(1201, 531, seed=31, gab=0, epf_iters=0, strategies="0")
    desc.color_transform, desc.out_format = 1, fmt
    assert_same(pipe.decode_frame(desc, coeffs), oracle(desc, coeffs), "ycbcr")


def test_jpeg_origin_frame_against_the_reference_decoder(pipe):
    """A 4:4:4 JPEG, recompressed by the reference encoder, entropy-decoded by the reference, rendered here: the 8-bit
    pixels are the reference decoder's (tests/golden/vs_reference.npz.xz: the hand-off and the digest of the public
    decoder's pixels, which the restatement in host-rcpss mode reproduces bit for bit)."""
    from oracle import cpu
    from tests.test_oracle_vs_reference import JPEG_CASES
    w, h, q = JPEG_CASES[0]
    z = support.load_xz_npz(support.GOLDEN / "vs_reference.npz.xz")
    support.require_host_rcpss(z)
    d = support.load_dump(z, f"jpeg{w}x{h}_{q}")
    desc = cpu.desc_from_dump(d)
    assert desc.color_transform == 1
    desc.out_format = abi.OUT_RGB_U8
    want = cpu.render_frame(desc, d.coeffs, rcp_mode=1)
    assert support.digest(want) == z[f"jpeg{w}x{h}_{q}.want"][1].tobytes()
    got = pipe.decode_frame(desc, d.coeffs)
    diff = np.abs(got.astype(np.int16) - want.astype(np.int16))
    assert diff.max() <= 1 and (diff != 0).mean() < 1e-3      # (rcpps in AdjustQuantBias may cross a rounding boundary)
