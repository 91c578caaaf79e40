"""The C restatement (oracle/jxl_oracle.c) against the committed golden vectors that
tests/golden/make_golden.py produced from the unmodified reference build."""
import numpy as np
import pytest

from libjxl_b200 import abi
from tests import support
from tests.golden.make_golden import transform_inputs

pytestmark = pytest.mark.usefixtures("built")


@pytest.fixture(scope="module")
def golden_transforms():
    return np.load(support.GOLDEN / "transforms.npz")


@pytest.mark.parametrize("strategy", range(27))
def test_transform_to_pixels_bit_exact(strategy, golden_transforms):
    from oracle import cpu
    coeffs, _ = transform_inputs(strategy)
    got = cpu.transform_to_pixels(strategy, coeffs)
    want = golden_transforms[f"px_{strategy}"]
    assert got.shape == want.shape
    assert np.array_equal(got, want), (abi.STRATEGY_NAMES[strategy], float(np.abs(got - want).max()))


@pytest.mark.parametrize("strategy", range(27))
def test_llf_from_dc_bit_exact(strategy, golden_transforms):
    from oracle import cpu
    _, dc = transform_inputs(strategy)
    n = 64 * abi.COVERED_X[strategy] * abi.COVERED_Y[strategy]
    got = cpu.llf_from_dc(strategy, dc, np.zeros(n, np.float32))
    want = np.zeros(n, np.float32)
    want[golden_transforms[f"llf_idx_{strategy}"]] = golden_transforms[f"llf_val_{strategy}"]
    assert np.array_equal(got, want)


def test_idct_dc_only_is_flat():
    """ac_strategy_test.cc:96-154 property: a DC-only block decodes to a constant."""
    from oracle import cpu
    for s in (0, 4, 5, 6, 7, 18, 21, 24):
        n = 64 * abi.COVERED_X[s] * abi.COVERED_Y[s]
        co = np.zeros(n, np.float32)
        co[0] = 1.25
        px = cpu.transform_to_pixels(s, co)
        assert np.allclose(px, 1.25, atol=1e-6)


def test_dct_idct_roundtrip():
    """dct_test.cc:217-249: ComputeScaledDCT then ComputeScaledIDCT is the identity."""
    from oracle import cpu
    rng = np.random.default_rng(5)
    for s in (0, 4, 5, 6, 7, 8, 9, 10, 11, 18, 19, 20):
        r, c = abi.COVERED_Y[s] * 8, abi.COVERED_X[s] * 8
        px = rng.normal(0, 1, (r, c)).astype(np.float32)
        co = cpu.scaled_dct(px)
        back = cpu.transform_to_pixels(s, co)
        assert np.abs(back - px).max() < 2e-5 * max(r, c)


def test_adjust_quant_bias():
    """quantizer-inl.h:35-67: 0 -> 0, +-1 -> +-biases[c], else q - biases[3]/q."""
    from oracle import cpu
    b = np.array([0.9453, 0.9299, 0.95, 0.145], np.float32)
    assert cpu.adjust_quant_bias(0, 0, b) == 0.0
    assert cpu.adjust_quant_bias(1, 1, b) == b[1]
    assert cpu.adjust_quant_bias(2, -1, b) == -b[2]
    for q in (2, -3, 17, -1000, 32767):
        want = np.float32(q) - np.float32(b[3] / np.float32(q))
        assert abs(cpu.adjust_quant_bias(0, q, b, 0) - want) <= 1e-6 * abs(q)
        # the rcpss flavour (reference's ApproximateReciprocal) stays within 12-bit accuracy
        assert abs(cpu.adjust_quant_bias(0, q, b, 1) - want) <= 0.145 * 4e-4 / abs(q) + 1e-6 * abs(q)


@pytest.mark.parametrize("tap", list(support.TAP_MASKS))
def test_frame_taps_against_reference(tap):
    """Whole small frame, stage by stage, against the reference's own DecodeGroupForRoundtrip +
    Gaborish/EPF/XYB stages (strict build). Exact-reciprocal mode: the only difference is the
    reference's 12-bit rcpps in AdjustQuantBias => tolerance, stated in absolute pixel units
    (XYB ~ [-1,1], linear RGB ~ [0,1])."""
    from oracle import cpu
    desc, coeffs, g = support.golden_desc(out_format=abi.OUT_PLANAR_F32)
    desc.stage_mask = abi.STAGE_EXPLICIT | support.TAP_MASKS[tap]
    got = cpu.render_frame(desc, coeffs, rcp_mode=0)
    want = g.taps[tap]
    assert got.shape == want.shape
    assert np.abs(got - want).max() <= 2e-5


def test_frame_full_decode_default_build():
    """Against what the public API of the default-flag reference build decodes (djxl
    --color_space=RGB_D65_SRG_Rel_Lin equivalent); conformance-style statistics."""
    from oracle import cpu
    desc, coeffs, g = support.golden_desc()
    got = cpu.render_frame(desc, coeffs, rcp_mode=0)
    want = g.decoded_default
    peak = float(np.abs(got - want).max())
    rmse = float(np.sqrt(np.mean((got - want) ** 2)))
    assert peak <= 5e-5 and rmse <= 5e-6, (peak, rmse)


def test_sigma_against_reference():
    from oracle import cpu
    desc, _, g = support.golden_desc()
    sg = cpu.compute_sigma(desc)[2:-2, 2:-2]
    assert np.array_equal(sg, g.sigma_interior)


OUTPUT_CASES = {"srgb_f32": (abi.OUT_RGB_F32, abi.STAGE_SRGB), "srgb_u8": (abi.OUT_RGB_U8, abi.STAGE_SRGB),
                "srgb_rgba8": (abi.OUT_RGBA_U8, abi.STAGE_SRGB), "srgb_u16": (abi.OUT_RGB_U16, abi.STAGE_SRGB),
                "srgb_f16": (abi.OUT_RGB_F16, abi.STAGE_SRGB), "linear_u8": (abi.OUT_RGB_U8, 0),
                "linear_f16": (abi.OUT_RGB_F16, 0)}


@pytest.mark.parametrize("case", list(OUTPUT_CASES))
def test_packed_outputs_against_reference(case):
    """sRGB transfer function + WriteToOutput packing (8-bit dither, 16-bit, binary16, RGBA) against
    the reference's own FromLinear/WriteToOutput stages.  Exact-reciprocal mode, so the 12-bit rcpps of
    the reference's AdjustQuantBias may move a value across a rounding boundary: at most one code
    value, on a small fraction of the samples (f32: absolute 2e-5).  tests/test_oracle_vs_reference.py
    holds the bit-exact version of this comparison (host-rcpss mode)."""
    from oracle import cpu
    fmt, mask = OUTPUT_CASES[case]
    desc, coeffs, _ = support.golden_desc(out_format=fmt, stage_mask=mask)
    got = cpu.render_frame(desc, coeffs, rcp_mode=0)
    want = np.load(support.GOLDEN / "outputs_small.npz")[case]
    if got.dtype == np.float32:
        assert np.abs(got - want).max() <= 2e-5
        return
    if got.dtype == np.float16:
        got = got.view(np.uint16)
        ok = (got & 0x7fff) > 0x0400          # leave binary16 subnormals (|v| < 6.1e-5) out of the ULP count
        d = np.abs(got.astype(np.int64) - want.astype(np.int64))[ok]
    else:
        d = np.abs(got.astype(np.int64) - want.astype(np.int64))
    assert got.shape == want.shape
    # one 16-bit code value (1.5e-5) is the size of the rcpps effect itself: more samples move
    frac = 2e-3 if got.dtype == np.uint8 else 5e-2
    assert d.max() <= 1 and (d != 0).mean() <= frac, (int(d.max()), float((d != 0).mean()))


def test_srgb_transfer_function_properties():
    """TF_SRGB::EncodedFromDisplay: 0 -> 0, odd symmetry, linear segment below 0.0031308, within the
    5e-7 the reference documents of the analytic curve (transfer_functions-inl.h:243)."""
    from oracle import cpu
    x = np.concatenate([np.linspace(0, 1, 2001), [0.0031308, 0.00313081, 2.0, 10.0]]).astype(np.float32)
    y = cpu.srgb_from_linear(x)
    xd = x.astype(np.float64)
    analytic = np.where(xd <= 0.0031308, 12.92 * xd, 1.055 * np.power(xd, 1 / 2.4) - 0.055)
    assert np.abs(y[:2003] - analytic[:2003]).max() <= 1e-6
    assert np.array_equal(cpu.srgb_from_linear(-x), -y)
    assert y[0] == 0.0 and np.all(np.diff(y[:2001]) >= 0)
    lin = x[x <= np.float32(0.0031308)]
    assert np.array_equal(cpu.srgb_from_linear(lin), lin * np.float32(12.92))


def test_binary16_demotion_matches_ieee():
    from oracle import cpu
    rng = np.random.default_rng(3)
    v = np.concatenate([rng.standard_normal(4000).astype(np.float32) * s for s in (1e-8, 1e-5, 1e-3, 1, 300, 7e4)] +
                       [np.array([0, -0.0, 65504, 65519.99, 65520, 1e10, -1e10, np.inf, -np.inf, 5.9604645e-8,
                                  2.9802322e-8, 2.9802326e-8, 6.1e-5, 6.0975552e-5], np.float32)])
    with np.errstate(over="ignore"):
        want = v.astype(np.float16).view(np.uint16)
    assert np.array_equal(cpu.f16_from_f32(v), want)


def test_make_unsigned_dither_and_rounding():
    """MakeUnsigned: round-half-even, clamp, and the dither indexed (x + 23c, y + 13c) mod 32."""
    from oracle import cpu
    assert cpu.make_unsigned(0.5, 16, 0, 0, 0) == 32768          # 32767.5 -> even
    assert cpu.make_unsigned(1.5 / 65535, 16, 5, 9, 1) == 2      # 1.5 -> 2
    assert cpu.make_unsigned(2.5 / 65535, 16, 5, 9, 1) == 2      # 2.5 -> 2
    assert cpu.make_unsigned(-3.0, 8, 1, 2, 0) == 0 and cpu.make_unsigned(7.0, 8, 1, 2, 0) == 255
    assert cpu.make_unsigned(float("nan"), 16, 0, 0, 0) == 0
    # periodicity and the channel offsets
    for (x, y, c) in ((0, 0, 0), (7, 30, 1), (31, 31, 2)):
        a = cpu.make_unsigned(0.5, 8, x, y, c)
        assert a == cpu.make_unsigned(0.5, 8, x + 32, y + 64, c)
        assert a == cpu.make_unsigned(0.5, 8, (x + 23 * c) % 32, (y + 13 * c) % 32, 0)


@pytest.mark.parametrize("xs,ys", support.DC_STAGE_CASES)
def test_dc_stage_against_reference(xs, ys):
    """DequantDC (4:4:4) and AdaptiveDCSmoothing -- the step in front of the path, restated for the
    next row of SURVEY §8f -- bit-exact against the reference's outputs (tests/golden/dc_stage.npz)."""
    from oracle import cpu
    z = np.load(support.GOLDEN / "dc_stage.npz")
    q = support.dc_stage_input(xs, ys)
    for mul in (1.0, 0.25):
        got = cpu.dequant_dc(q, support.DC_FACTORS, mul, support.DC_CFL)
        assert np.array_equal(got, z[f"dequant_{xs}x{ys}_mul{mul}"]), mul
    dc = z[f"dequant_{xs}x{ys}_mul1.0"]
    got = cpu.adaptive_dc_smoothing(dc, support.DC_FACTORS)
    want = z[f"smooth_{xs}x{ys}"]
    assert np.array_equal(got, want)
    if xs > 2 and ys > 2:
        # borders untouched; the smooth region changes, the busy quadrant mostly does not
        assert np.array_equal(got[:, 0], dc[:, 0]) and np.array_equal(got[:, :, -1], dc[:, :, -1])
        if xs >= 16:
            changed = got != dc
            assert changed[:, 1:ys // 2 - 1, 1:xs // 2 - 1].mean() > 0.5
            assert changed[:, ys // 2 + 1:-1, xs // 2 + 1:-1].mean() < 0.2
    else:
        assert np.array_equal(got, dc)


def test_render_frame_with_quantised_dc_matches_prepared_dc():
    """jxo_render_frame's optional DC stage (quant_dc given) == rendering with the DC planes that
    DequantDC + AdaptiveDCSmoothing produce, on a synthetic all-strategy frame with two DC groups."""
    import jxl_workload as wl
    from oracle import cpu
    desc, coeffs = wl.synthetic_frame(2100, 300, seed=5)
    yb, xb = desc.ysize_blocks, desc.xsize_blocks
    q = support.dc_stage_input(xb, yb)
    gm = np.array([[1.0, 0.5]], np.float32)
    dc = np.zeros((3, yb, xb), np.float32)
    for gx in range(2):
        sl = (slice(None), slice(None), slice(gx * 256, (gx + 1) * 256))
        dc[sl] = cpu.dequant_dc(q[sl], support.DC_FACTORS, float(gm[0, gx]), support.DC_CFL)
    desc.dc = cpu.adaptive_dc_smoothing(dc, support.DC_FACTORS)
    want = cpu.render_frame(desc, coeffs, rcp_mode=0)
    desc.dc = None
    desc.quant_dc, desc.dc_group_mul = q, gm
    desc.dc_factors, desc.dc_cfl_factors = support.DC_FACTORS, support.DC_CFL
    assert np.array_equal(cpu.render_frame(desc, coeffs, rcp_mode=0), want)
