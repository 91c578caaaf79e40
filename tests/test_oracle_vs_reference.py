"""Pins oracle/jxl_oracle.c against the UNMODIFIED reference.  The reference's outputs (strict build =
-ffp-contract=off, so bit-exact is expected) and the coefficient hand-offs of the frames it encoded are stored
in tests/golden/vs_reference.npz.xz (tests/golden/make_vs_reference.py); the tests that drive the reference's own
decoder through the integration headers need oracle/_ref, compiled by oracle/build_ref.py, and skip without it."""
import numpy as np
import pytest

import jxl_workload as wl
from libjxl_b200 import abi
from tests import support

pytestmark = pytest.mark.usefixtures("built")

# The golden data stores every frame's coefficients, so the frames are small; each still spans more than one
# 256x256 group (the reference's decoder does not hand single-group frames to the hot path).
STAGE_FRAMES = [
    dict(w=261, h=85, distance=1.0, gaborish=1, epf=3, kind="photo"),      # odd size, full chain
    dict(w=264, h=96, distance=1.0, gaborish=-1, epf=-1, kind="photo"),    # BASELINE config 1 settings (defaults: gab, epf 1)
    dict(w=264, h=48, distance=0.5, gaborish=0, epf=0, kind="photo"),      # no filters: dequant+IDCT+XYB only
    dict(w=264, h=136, distance=3.0, gaborish=1, epf=2, kind="smooth"),    # large transforms (up to 64x64)
]
OUTPUT_FRAME = (259, 61)
OUTPUT_STAGE_CASES = [(abi.OUT_RGB_F32, True), (abi.OUT_RGB_U8, True), (abi.OUT_RGBA_U8, True), (abi.OUT_RGB_U16, True),
                      (abi.OUT_RGB_F16, True), (abi.OUT_RGB_U8, False), (abi.OUT_RGB_F16, False)]
PUBLIC_CASES = [(abi.OUT_RGB_U8, np.uint8, 3), (abi.OUT_RGBA_U8, np.uint8, 4), (abi.OUT_RGB_U16, np.uint16, 3),
                (abi.OUT_RGB_F16, np.float16, 3), (abi.OUT_RGB_F32, np.float32, 3)]
DC_CASES = [(256, 256), (960, 540), (37, 21)]
UPSAMPLING_CASES = [(2, 600, 300), (4, 1100, 210), (8, 2100, 160)]
NOISE_CASES = [(1, 300, 150, 3200), (2, 600, 299, 6400), (1, 261, 130, 1600)]
JPEG_CASES = [(300, 150, 90), (261, 165, 75)]


@pytest.fixture(scope="module")
def golden():
    return support.load_xz_npz(support.GOLDEN / "vs_reference.npz.xz")


@pytest.fixture(scope="module")
def host_rcpss(golden):
    support.require_host_rcpss(golden)


def chain(info) -> int:
    return (1 if info.gab else 0) | (2 if info.epf_iters >= 3 else 0) | (4 if info.epf_iters >= 1 else 0) | \
        (8 if info.epf_iters >= 2 else 0)


def stage_masks(info) -> list[int]:
    """Every stage prefix of the frame's chain (and the chain with XYB) that test_frames_stage_by_stage renders."""
    frame_mask = chain(info)
    masks = [0, 16, frame_mask, frame_mask | 16]
    if info.epf_iters > 0:
        masks += [1, 1 | 4, 2 | 4 | 8]
    return masks


def same(got: np.ndarray, want_digest: np.ndarray) -> bool:
    return support.digest(got) == want_digest.tobytes()


@pytest.fixture(scope="module")
def refmod(ref_available):
    from oracle import build_ref
    if not ref_available:
        if build_ref.reference_present():
            pytest.fail("oracle/_ref is not built although the reference is present: the oracle (and the tables it "
                        "shares with the product, csrc/jxl_tables.h) would go unpinned -- run `python oracle/build_ref.py`")
        pytest.skip("oracle/_ref not built (no reference source tree)")
    from oracle import ref
    ref.use_variant("strict")
    yield ref
    ref.use_variant("default")


@pytest.mark.parametrize("strategy", range(27))
def test_all_strategies_bit_exact(strategy, golden):
    from oracle import cpu
    rng = np.random.default_rng(1000 + strategy)
    r, c = abi.COVERED_Y[strategy] * 8, abi.COVERED_X[strategy] * 8
    want = golden[f"strategy{strategy}"]
    for trial in range(2):
        co = (rng.laplace(0, 1.0, r * c) * (rng.random(r * c) < 0.3)).astype(np.float32)
        assert same(cpu.transform_to_pixels(strategy, co), want[trial]), trial
    dc = rng.normal(0, 1, (abi.COVERED_Y[strategy], abi.COVERED_X[strategy])).astype(np.float32)
    assert same(cpu.llf_from_dc(strategy, dc, np.zeros(r * c, np.float32)), want[2])


@pytest.mark.parametrize("cfg", range(len(STAGE_FRAMES)), ids=[f"cfg{k}" for k in range(len(STAGE_FRAMES))])
def test_frames_stage_by_stage(cfg, golden, host_rcpss):
    """Every stage prefix, hot path only, same coefficients: the reference's own
    DecodeGroupForRoundtrip + stages vs the C restatement. rcp_mode 1 (host rcpss, what the
    reference's AVX2 path executes) must be bit-exact; rcp_mode 0 (exact reciprocal = what the
    CUDA path computes) within 2e-5 absolute."""
    from oracle import cpu
    d = support.load_dump(golden, f"stage{cfg}")
    desc = cpu.desc_from_dump(d, out_format=abi.OUT_PLANAR_F32)
    masks = golden[f"stage{cfg}.masks"].tolist()
    assert masks == sorted(set(stage_masks(d.info)))
    for mask, want in zip(masks, golden[f"stage{cfg}.want"]):
        desc.stage_mask = abi.STAGE_EXPLICIT | mask
        got1 = cpu.render_frame(desc, d.coeffs, rcp_mode=1)
        assert same(got1, want), mask
        got0 = cpu.render_frame(desc, d.coeffs, rcp_mode=0)
        assert np.abs(got0 - got1).max() <= 2e-5, mask
    # and the full public-API decode of the default-flag build (compiler-made FMAs differ)
    desc.stage_mask = 0
    desc.out_format = abi.OUT_RGB_F32
    got = cpu.render_frame(desc, d.coeffs, rcp_mode=0)
    full = golden[f"stage{cfg}.full_sample"]
    assert np.abs(got.reshape(-1)[support.sample_index(got.size)] - full).max() <= 5e-5


def test_hot_path_render_equals_public_decode(refmod):
    """The transform-only CPU baseline (ref_frame_render) is the same computation the public
    decoder does after entropy decoding: identical pixels."""
    refmod.use_variant("default")
    try:
        img = wl.synth_image(520, 300, 5)
        data = refmod.encode_rgb8(img, 1.0, 7, -1, -1, 2)
        full = refmod.decode_linear_f32(data, 2)
        fr = refmod.Frame(data, 2)
        planar, secs = fr.render(-1, reps=2)
        assert np.array_equal(planar.transpose(1, 2, 0), full)
        assert len(secs) == 2 and all(s > 0 for s in secs)
        fr.close()
    finally:
        refmod.use_variant("strict")


@pytest.mark.parametrize("fmt,srgb", OUTPUT_STAGE_CASES)
def test_output_stages_bit_exact(fmt, srgb, golden, host_rcpss):
    """FromLinearStage<OpRgb> + WriteToOutputStage (dithered u8, RGBA, u16, binary16, f32) of the strict
    reference build vs the restatement, whole frame, host-rcpss mode: identical bytes."""
    from oracle import cpu
    d = support.load_dump(golden, "outputs")
    desc = cpu.desc_from_dump(d, out_format=fmt, stage_mask=abi.STAGE_SRGB if srgb else 0)
    got = cpu.render_frame(desc, d.coeffs, rcp_mode=1)
    assert got.shape == (*OUTPUT_FRAME[::-1], 4 if fmt == abi.OUT_RGBA_U8 else 3)
    assert same(got, golden[f"outputs.{fmt}_{int(srgb)}"][0])


@pytest.mark.parametrize("xs,ys", DC_CASES)
def test_dc_stage_bit_exact(xs, ys, golden):
    """DequantDC + AdaptiveDCSmoothing of the reference (both builds) vs the restatement."""
    from oracle import cpu
    q = support.dc_stage_input(xs, ys)
    for variant in ("strict", "default"):
        want = golden[f"dc_{variant}_{xs}x{ys}"]
        for k, mul in enumerate((1.0, 0.5)):
            assert same(cpu.dequant_dc(q, support.DC_FACTORS, mul, support.DC_CFL), want[k]), (variant, mul)
        dc = cpu.dequant_dc(q, support.DC_FACTORS, 1.0, support.DC_CFL)
        assert same(cpu.adaptive_dc_smoothing(dc, support.DC_FACTORS), want[2]), variant


@pytest.mark.parametrize("fmt,dtype,ch", PUBLIC_CASES)
def test_full_chain_equals_default_public_decode(fmt, dtype, ch, golden, host_rcpss):
    """The path with JXLGPU_STAGE_SRGB and a packed output format is, byte for byte, what the reference's
    PUBLIC decoder delivers by default for an sRGB image (what `djxl in.jxl out.png` writes): public API
    == hot path + FromLinear + WriteToOutput (reference stages, checked when the golden data is made)
    == the restatement (strict build)."""
    from oracle import cpu
    img = wl.synth_image(*OUTPUT_FRAME, 5)
    d = support.load_dump(golden, "outputs")
    desc = cpu.desc_from_dump(d, out_format=fmt, stage_mask=abi.STAGE_SRGB)
    restated = cpu.render_frame(desc, d.coeffs, rcp_mode=1)
    assert restated.dtype == dtype and restated.shape == (*OUTPUT_FRAME[::-1], ch)
    assert same(restated, golden[f"public.{fmt}"][0])
    # and it is a decode of the image that went in (8-bit sRGB in, d1.0): mean abs error < 2 %
    scale = {np.uint8: 255.0, np.uint16: 65535.0}.get(dtype, 1.0)
    assert np.abs(restated[..., :3].astype(np.float64) / scale - img / 255.0).mean() < 0.02


@pytest.mark.parametrize("distance", [1.0, 8.0])
def test_group_major_ac_image_is_a_drop_in(distance, refmod):
    """integration/pinned_ac_image.h (the storage class a libjxl host installs for a GPU frame) driven by
    the UNMODIFIED reference decoder through libjxl's abstract ACImage interface: same coefficients,
    same pixels, and the allocation is the [group][channel][65536] layout the C ABI takes as is."""
    img = wl.synth_image(600, 300, 21)
    data = refmod.encode_rgb8(img, distance, 7, -1, -1, 2)
    a = refmod.Frame(data, 2)
    b = refmod.Frame(data, 2, storage=1)
    da, db = a.dump(), b.dump()
    assert da.coeffs.dtype == db.coeffs.dtype and np.array_equal(da.coeffs, db.coeffs)
    assert np.array_equal(da.decoded, db.decoded)
    raw = b.raw_group_major_coeffs()
    assert raw.shape == (da.info.num_groups, 3, 65536)
    assert np.array_equal(raw.transpose(1, 0, 2), da.coeffs)
    assert np.count_nonzero(raw) > 0
    a.close()
    b.close()


@pytest.mark.parametrize("cfg", [dict(w=517, h=331, distance=1.0, gaborish=1, epf=3), dict(w=300, h=520, distance=0.5, gaborish=0, epf=0)])
def test_gpu_frame_binding_from_decoder_state(cfg, refmod):
    """integration/gpu_frame_binding.h -- the C++ a libjxl maintainer adds to fill jxlgpu_frame from
    PassesDecoderState -- applied to the unmodified reference's live decoder state: every scalar equals
    the description the tests build by hand, and the oracle rendered straight from the bound struct
    (zero-copy pointers + strides into libjxl's images) gives the reference's pixels."""
    import ctypes as C
    from oracle import cpu
    img = wl.synth_image(cfg["w"], cfg["h"], 31)
    data = refmod.encode_rgb8(img, cfg["distance"], 7, cfg["gaborish"], cfg["epf"], 2)
    fr = refmod.Frame(data, 2)
    d = fr.dump()
    bound = fr.bind_gpu_frame(abi.OUT_RGB_F32, 0)
    by_hand = cpu.desc_from_dump(d).to_struct()
    pointer_fields = {"ac_strategy", "raw_quant", "epf_sharpness", "ytox_map", "ytob_map", "dc", "dequant_table",
                      "quant_dc", "dc_group_mul"}
    stride_fields = {"ac_strategy_stride", "raw_quant_stride", "epf_sharpness_stride", "cmap_stride", "dc_stride"}
    for name, _ in abi.JxlGpuFrame._fields_:
        if name in pointer_fields or name in stride_fields:
            continue
        a, b = getattr(bound, name), getattr(by_hand, name)
        if hasattr(a, "__len__"):
            assert list(a) == list(b), name
        else:
            assert a == b, name
    assert bound.raw_quant_stride >= bound.xsize_blocks and bound.dc_stride >= bound.xsize_blocks
    # render with the oracle straight from the bound struct
    co = np.ascontiguousarray(d.coeffs)
    ptrs = (C.c_void_p * 3)(*[co.ctypes.data + c * co[0].nbytes for c in range(3)])
    out = np.zeros((d.info.ysize, d.info.xsize, 3), np.float32)
    assert cpu.lib().jxo_render_frame(C.byref(bound), ptrs, 1, out.ctypes.data) == 0
    want, _ = fr.render(-1)
    assert np.array_equal(out, want.transpose(1, 2, 0))
    fr.close()


@pytest.mark.parametrize("rs,w,h", UPSAMPLING_CASES)
def test_upsampling_stage_bit_exact(rs, w, h, golden, host_rcpss):
    """SURVEY.md §8f rank 4, UpsamplingStage (stage_upsampling.cc:51-271): frames encoded with resampling 2/4/8.
    The restatement (jxo_upsample_plane, after the filters and before XYB like PreparePipeline orders them) is
    bit-exact against the reference's own stage, whose output is the reference's public decode (checked when
    the golden data is made)."""
    from oracle import cpu
    d = support.load_dump(golden, f"ups{rs}")
    i = d.info
    assert i.upsampling == rs and (i.xsize_upsampled, i.ysize_upsampled) == (w, h)
    desc = cpu.desc_from_dump(d)
    assert desc.upsampling == rs and desc.out_xsize == w and desc.out_ysize == h
    desc.out_format = abi.OUT_PLANAR_F32
    want, want_xyb = golden[f"ups{rs}.want"]
    got = cpu.render_frame(desc, d.coeffs, rcp_mode=1)
    assert got.shape == (3, h, w) and same(got, want)
    desc.stage_mask = abi.STAGE_EXPLICIT | chain(i)          # the upsampled XYB planes themselves
    assert same(cpu.render_frame(desc, d.coeffs, rcp_mode=1), want_xyb)


@pytest.mark.parametrize("rs,w,h,iso", NOISE_CASES)
def test_noise_stages_bit_exact(rs, w, h, iso, golden, host_rcpss):
    """SURVEY.md §8f rank 4, noise: frames the reference encoder made with photon noise (frame flag kNoise).
    Random3Planes (dec_noise.cc:45-152) + ConvolveNoiseStage + AddNoiseStage (stage_noise.cc) restated in
    oracle/jxl_oracle.c: bit-exact against the reference's own stages, alone and behind the upsampling, whose
    output is the reference's public decode (checked when the golden data is made)."""
    from oracle import cpu
    d = support.load_dump(golden, f"noise{rs}_{w}x{h}_{iso}")
    i = d.info
    assert i.noise == 1 and max(i.noise_lut) > 1e-3 and i.upsampling == rs
    desc = cpu.desc_from_dump(d)
    assert desc.noise == 1 and (desc.visible_frame_index, desc.nonvisible_frame_index) == (1, 0)
    desc.out_format = abi.OUT_PLANAR_F32
    got = cpu.render_frame(desc, d.coeffs, rcp_mode=1)
    assert same(got, golden[f"noise{rs}_{w}x{h}_{iso}.want"][0])
    desc.noise = 0
    assert not np.array_equal(cpu.render_frame(desc, d.coeffs, rcp_mode=1), got)


def make_jpeg(w, h, quality, seed=5):
    """A baseline 4:4:4 JPEG of the seeded test image (Pillow)."""
    import io
    from PIL import Image
    b = io.BytesIO()
    Image.fromarray(wl.synth_image(w, h, seed)).save(b, format="JPEG", quality=quality, subsampling=0)
    return b.getvalue()


@pytest.mark.parametrize("w,h,q", JPEG_CASES)
def test_jpeg_origin_ycbcr_frames(w, h, q, golden, host_rcpss):
    """SURVEY.md §8f rank 4, YCbCr: a 4:4:4 JPEG recompressed by the reference encoder (JxlEncoderAddJPEGFrame) is a
    VarDCT frame with the YCbCr colour transform.  Dequantisation + IDCT are the XYB path's; the colour stage is
    kYCbCrStage (stage_ycbcr.cc:33-71).  Restatement bit-exact against the reference's stages, and its 8-bit output
    identical to the reference's PUBLIC decoder (no transfer function follows: the image is not XYB-encoded)."""
    from oracle import cpu
    d = support.load_dump(golden, f"jpeg{w}x{h}_{q}")
    i = d.info
    assert i.ycbcr == 1 and i.gab == 0 and i.epf_iters == 0
    desc = cpu.desc_from_dump(d)
    assert desc.color_transform == 1
    want, public = golden[f"jpeg{w}x{h}_{q}.want"]
    desc.out_format = abi.OUT_PLANAR_F32
    assert same(cpu.render_frame(desc, d.coeffs, rcp_mode=1), want)
    desc.out_format = abi.OUT_RGB_U8
    got = cpu.render_frame(desc, d.coeffs, rcp_mode=1)
    assert got.shape == (h, w, 3) and same(got, public)
