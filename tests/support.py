"""Shared helpers for the test-suite."""
from __future__ import annotations

import hashlib
import io
import json
import lzma
from pathlib import Path

import numpy as np

from libjxl_b200 import abi

GOLDEN = Path(__file__).resolve().parent / "golden"


class _Info:
    pass


class GoldenDump:
    """tests/golden/frame_small.npz viewed like an oracle.ref.FrameDump."""

    def __init__(self):
        z = np.load(GOLDEN / "frame_small.npz")
        self.z = z
        self.info = _Info()
        for k in z.files:
            if k.startswith("info_"):
                v = z[k]
                setattr(self.info, k[5:], v.tolist() if v.ndim else v.item())
        self.ac_strategy, self.raw_quant, self.sharpness = z["ac_strategy"], z["raw_quant"], z["sharpness"]
        self.ytox, self.ytob, self.dc = z["ytox"], z["ytob"], z["dc"]
        self.dequant, self.dequant_offsets, self.coeffs = z["dequant"], z["dequant_offsets"], z["coeffs"]
        self.taps = {k[4:]: z[k] for k in z.files if k.startswith("tap_")}
        self.decoded_default = z["decoded_default"]
        self.sigma_interior = z["sigma_interior"]


DUMP_FIELDS = ("ac_strategy", "raw_quant", "sharpness", "ytox", "ytob", "dc", "dequant", "dequant_offsets")


def store_dump(fx: dict, case: str, d) -> None:
    """An oracle.ref.FrameDump as `<case>.*` entries of a golden .npz: side information, the info scalars, and
    the non-zero coefficients (a bit mask of their positions + their values).  Dequantisation matrices of strategies the
    frame does not use are zeroed (they are never read, and zeros compress)."""
    i = d.info
    info = {name: (list(v) if hasattr(v, "__len__") else v) for name, v in
            ((name, getattr(i, name)) for name, _ in type(i)._fields_)}
    # tables the decoder leaves unset in frames that do not use them
    if not i.noise:
        info["noise_lut"] = [0.0] * len(info["noise_lut"])
    if i.ycbcr:
        info["inverse_opsin_matrix"] = [0.0] * len(info["inverse_opsin_matrix"])
    fx[f"{case}.info"] = np.frombuffer(json.dumps(info).encode(), np.uint8)
    dq = d.dequant.copy()
    keep = np.zeros(dq.size, bool)
    for s in np.unique(d.ac_strategy[(d.ac_strategy & 1) == 1] >> 1):
        n = 64 * abi.COVERED_X[s] * abi.COVERED_Y[s]
        for c in range(3):
            keep[d.dequant_offsets[s, c]: d.dequant_offsets[s, c] + n] = True
    dq[~keep] = 0
    planes = {name: getattr(d, name) for name in DUMP_FIELDS}
    planes["dequant"] = dq
    planes["raw_quant"] = np.where(d.ac_strategy & 1, d.raw_quant, 0).astype(np.int32)   # defined on first blocks only
    for name, a in planes.items():
        fx[f"{case}.{name}"] = a
    flat = d.coeffs.reshape(-1)
    fx[f"{case}.coeff_shape"] = np.array(d.coeffs.shape, np.int64)
    fx[f"{case}.coeff_nonzero"] = np.packbits(flat != 0)
    fx[f"{case}.coeff_val"] = flat[flat != 0]


def load_dump(z, case: str):
    """What store_dump wrote, viewed like an oracle.ref.FrameDump (without the decoded pixels)."""
    d = _Info()
    d.info = _Info()
    for name, v in json.loads(z[f"{case}.info"].tobytes()).items():
        setattr(d.info, name, v)
    for name in DUMP_FIELDS:
        setattr(d, name, z[f"{case}.{name}"])
    val = z[f"{case}.coeff_val"]
    d.coeffs = np.zeros(tuple(z[f"{case}.coeff_shape"]), val.dtype)
    d.coeffs.reshape(-1)[np.unpackbits(z[f"{case}.coeff_nonzero"], count=d.coeffs.size).astype(bool)] = val
    return d


def load_xz_npz(path: Path):
    """A golden .npz stored whole under xz (the members share their dequantisation tables and headers)."""
    return np.load(io.BytesIO(lzma.decompress(path.read_bytes())))


def digest(a: np.ndarray) -> bytes:
    """SHA-256 of an array's dtype, shape and bytes: a stored reference output is compared bit for bit
    through it without being stored."""
    a = np.ascontiguousarray(a)
    h = hashlib.sha256(f"{a.dtype.str}{a.shape}".encode())
    h.update(a.tobytes())
    return h.digest()


def rcpss_probe() -> np.ndarray:
    """AdjustQuantBias in host-rcpss mode (oracle rcp_mode 1) over a spread of quantised values."""
    from oracle import cpu
    b = np.array([0.9453, 0.9299, 0.95, 0.145], np.float32)
    return np.array([cpu.adjust_quant_bias(0, int(q), b, 1) for q in range(-70000, 70001, 7)], np.float32)


def require_host_rcpss(z) -> None:
    """Outputs rendered in host-rcpss mode are compared bit for bit with digests made on another machine, and
    rcpss is not the same on every x86 CPU: skip where this host's rcpss differs from that machine's."""
    import pytest
    if digest(rcpss_probe()) != z["rcpss"].tobytes():
        pytest.skip("this CPU's rcpss differs from the one the golden digests were made with")


def sample_index(size: int, n: int = 512) -> np.ndarray:
    """The fixed positions (seed 0) at which a reference output compared within a tolerance is stored."""
    return np.sort(np.random.default_rng(0).choice(size, min(n, size), replace=False))


def golden_desc(**overrides) -> tuple[abi.FrameDesc, np.ndarray, GoldenDump]:
    from oracle import cpu as ocpu
    g = GoldenDump()
    return ocpu.desc_from_dump(g, **overrides), g.coeffs, g


def ulp_diff(a: np.ndarray, b: np.ndarray) -> int:
    """max distance in float32 ULPs (ordered-integer representation)."""
    ai = a.astype(np.float32).view(np.int32).astype(np.int64)
    bi = b.astype(np.float32).view(np.int32).astype(np.int64)
    ai = np.where(ai < 0, np.int64(-2147483648) - ai, ai)
    bi = np.where(bi < 0, np.int64(-2147483648) - bi, bi)
    return int(np.abs(ai - bi).max())


TAP_MASKS = {"idct": 0, "gab_epf012": 15, "full": 31}


DC_STAGE_CASES = [(37, 21), (64, 48), (3, 3), (2, 9)]
DC_FACTORS = (3.1 / 4096, 1.7 / 512, 0.9 / 256)
DC_CFL = (0.0117, 0.0, 0.935)


def dc_stage_input(xs: int, ys: int) -> np.ndarray:
    """Seeded quantised DC planes (X, Y, B): smooth gradients (adaptive smoothing engages) with one busy
    quadrant (it must switch itself off there)."""
    rng = np.random.default_rng(1000 * xs + ys)
    yy, xx = np.mgrid[0:ys, 0:xs]
    q = np.stack([np.round(20 * np.sin(xx / 17 + c) + 15 * np.cos(yy / 23 + c) + rng.random((ys, xs)) * 1.2)
                  for c in range(3)]).astype(np.int32)
    q[:, ys // 2:, xs // 2:] += rng.integers(-40, 40, (3, ys - ys // 2, xs - xs // 2))
    return q
