#!/usr/bin/env python3
"""Regenerate tests/golden/vs_reference.npz.xz from the UNMODIFIED reference (oracle/_ref, built by
oracle/build_ref.py):

    python tests/golden/make_vs_reference.py

It holds what tests/test_oracle_vs_reference.py and the reference-frame tests of tests/test_gpu_parity.py
compare with, so that they run without the reference:
  * per frame `<case>.*`: the reference decoder's coefficient hand-off (side information, non-zero
    coefficients as a position bit mask + values; dequantisation matrices of unused strategies zeroed);
  * outputs that must match bit for bit as SHA-256 digests (tests/support.py:digest);
  * outputs compared within a tolerance as a fixed sample of their values (tests/support.py:sample_index);
  * `rcpss`: the digest of what this CPU's rcpss gives AdjustQuantBias (tests/support.py:rcpss_probe), since
    the outputs of the restatement in host-rcpss mode can only be compared on CPUs that agree with it.
Every reference-side identity the tests used to check at run time (hot path == public decode, noise changes
the pixels, ...) is asserted here instead.
"""
from __future__ import annotations

import io
import lzma
import sys
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parents[2]
sys.path.insert(0, str(ROOT))

import jxl_workload as wl  # noqa: E402
from libjxl_b200 import abi  # noqa: E402
from oracle import ref  # noqa: E402
from tests import support  # noqa: E402
from tests import test_oracle_vs_reference as T  # noqa: E402

HERE = Path(__file__).resolve().parent


def digests(*arrays) -> np.ndarray:
    return np.stack([np.frombuffer(support.digest(a), np.uint8) for a in arrays])


def main() -> int:
    fx: dict[str, np.ndarray] = {"rcpss": np.frombuffer(support.digest(support.rcpss_probe()), np.uint8)}
    ref.use_variant("strict")

    for s in range(27):
        rng = np.random.default_rng(1000 + s)
        r, c = abi.COVERED_Y[s] * 8, abi.COVERED_X[s] * 8
        px = []
        for _ in range(2):
            co = (rng.laplace(0, 1.0, r * c) * (rng.random(r * c) < 0.3)).astype(np.float32)
            px.append(ref.transform_to_pixels(s, co, r, c))
        dc = rng.normal(0, 1, (abi.COVERED_Y[s], abi.COVERED_X[s])).astype(np.float32)
        fx[f"strategy{s}"] = digests(*px, ref.llf_from_dc(s, dc, np.zeros(r * c, np.float32)))

    for k, cfg in enumerate(T.STAGE_FRAMES):
        img = wl.synth_image(cfg["w"], cfg["h"], 77, cfg["kind"])
        data = ref.encode_rgb8(img, cfg["distance"], 7, cfg["gaborish"], cfg["epf"], 2)
        fr = ref.Frame(data, 2)
        d = fr.dump()
        masks = sorted(set(T.stage_masks(d.info)))
        support.store_dump(fx, f"stage{k}", d)
        fx[f"stage{k}.masks"] = np.array(masks, np.int32)
        fx[f"stage{k}.want"] = digests(*[fr.render(m)[0] for m in masks])
        fr.close()
        ref.use_variant("default")
        full = ref.decode_linear_f32(data, 1)
        ref.use_variant("strict")
        fx[f"stage{k}.full_sample"] = full.reshape(-1)[support.sample_index(full.size)]

    img = wl.synth_image(*T.OUTPUT_FRAME, 5)
    data = ref.encode_rgb8(img, 1.0, 7, -1, -1, 2)
    fr = ref.Frame(data, 2)
    support.store_dump(fx, "outputs", fr.dump())
    for fmt, srgb in T.OUTPUT_STAGE_CASES:
        fx[f"outputs.{fmt}_{int(srgb)}"] = digests(fr.render_out(-33 if srgb else -1, fmt)[0])
    for fmt, dtype, ch in T.PUBLIC_CASES:
        public = ref.decode_native(data, (*T.OUTPUT_FRAME[::-1], ch), dtype, 2)
        hot, _ = fr.render_out(-33, fmt)
        assert support.digest(public) == support.digest(hot), fmt
        fx[f"public.{fmt}"] = digests(public)
    fr.close()

    for variant in ("strict", "default"):
        ref.use_variant(variant)
        for xs, ys in T.DC_CASES:
            q = support.dc_stage_input(xs, ys)
            dq = [ref.dequant_dc(q, support.DC_FACTORS, mul, support.DC_CFL) for mul in (1.0, 0.5)]
            fx[f"dc_{variant}_{xs}x{ys}"] = digests(*dq, ref.adaptive_dc_smoothing(dq[0], support.DC_FACTORS, 3))
    ref.use_variant("strict")

    for rs, w, h in T.UPSAMPLING_CASES:
        data = ref.encode_rgb8(wl.synth_image(w, h, seed=rs), 1.0, 7, -1, -1, 4, resampling=rs)
        fr = ref.Frame(data, 2)
        i = fr.info
        want, _ = fr.render(T.chain(i) | ref.STAGE_XYB | ref.STAGE_UPSAMPLING)
        want_xyb, _ = fr.render(T.chain(i) | ref.STAGE_UPSAMPLING)
        support.store_dump(fx, f"ups{rs}", fr.dump())
        fr.close()
        assert np.array_equal(np.moveaxis(want, 0, 2), ref.decode_linear_f32(data, 2))
        fx[f"ups{rs}.want"] = digests(want, want_xyb)

    for rs, w, h, iso in T.NOISE_CASES:
        data = ref.encode_rgb8(wl.synth_image(w, h, seed=rs + iso), 1.0, 7, -1, -1, 4, resampling=rs | ((iso // 100) << 16))
        fr = ref.Frame(data, 2)
        i = fr.info
        want, _ = fr.render(T.chain(i) | ref.STAGE_XYB | ref.STAGE_UPSAMPLING | ref.STAGE_NOISE)
        without, _ = fr.render(T.chain(i) | ref.STAGE_XYB | ref.STAGE_UPSAMPLING)
        assert not np.array_equal(without, want)
        support.store_dump(fx, f"noise{rs}_{w}x{h}_{iso}", fr.dump())
        fr.close()
        assert np.array_equal(np.moveaxis(want, 0, 2), ref.decode_linear_f32(data, 2))
        fx[f"noise{rs}_{w}x{h}_{iso}.want"] = digests(want)

    for w, h, q in T.JPEG_CASES:
        data = ref.encode_jpeg(T.make_jpeg(w, h, q), 4)
        fr = ref.Frame(data, 2)
        want, _ = fr.render(ref.STAGE_XYB)
        support.store_dump(fx, f"jpeg{w}x{h}_{q}", fr.dump())
        fr.close()
        fx[f"jpeg{w}x{h}_{q}.want"] = digests(want, ref.decode_native(data, (h, w, 3), np.uint8, 2))

    buf = io.BytesIO()
    np.savez(buf, **fx)
    (HERE / "vs_reference.npz.xz").write_bytes(lzma.compress(buf.getvalue(), preset=9 | lzma.PRESET_EXTREME))
    print("vs_reference.npz.xz", (HERE / "vs_reference.npz.xz").stat().st_size, "bytes")
    return 0


if __name__ == "__main__":
    sys.exit(main())
