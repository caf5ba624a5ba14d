"""The hand-written device arithmetic of csrc/p2p_kernels.cuh over its whole input domain.

The projection kernels claim bit-exact agreement with the reference, and that claim rests on a few device primitives:
the range-check-free IEEE sqrt and division, NumPy's SVML arccos / arctan2 restated with the 128 seed coefficient
pairs, the magic-constant FMA that is cvRound(x * 32), and - in the minimax mode - acos_fast, atan2_fast and the
compensated pi - a of the mirrored pixel.  End-to-end tests only see the inputs a few views produce, and a one-ulp
coordinate error that does not move a 1/32-px bin leaves every pixel unchanged.  tests/device_math_probe.cu calls the
real __device__ functions; each test compares them with a reference from outside the function under test (the generic
CUDA intrinsics, NumPy's own arccos / arctan2, or the device's double-precision functions).
"""
import ctypes as C
import json
import subprocess
import tempfile
from pathlib import Path

import numpy as np
import pytest

from oracle import svml_model

ROOT = Path(__file__).resolve().parent.parent
PROBE_SRC = Path(__file__).resolve().parent / "device_math_probe.cu"
CSRC = ROOT / "360-to-planer-images_b200" / "csrc"

F32_ONE, F32_HALF_PI = 0x3F800000, 0x3FC90FDB   # bit patterns of 1.0f and f32(pi / 2)
F32_PI = np.float32(np.pi)
NEG = 0x80000000
# Accuracy of the minimax fits as measured by the tests below over their whole domains (every float in [-1, 1] for
# acos_fast; the four atan2 input sets for atan2_fast; every float in [-pi/2, pi/2] for mirror_phi_fast) on an
# NVIDIA B200, profiles/r4_device_math_accuracy.json.  Max error in ulps of the result's binade, against the device's
# double acos / atan2; the correctly rounded fraction is among the inputs whose rounding is decided.
ACOS_FAST_MAX_ULP, ACOS_FAST_CR_MIN = 1.07, 0.9979    # measured 1.0696, 0.99798
ATAN2_FAST_MAX_ULP, ATAN2_FAST_CR_MIN = 1.76, 0.6728   # measured 1.7582, 0.67284


# sha256 of np.arccos(z) + np.arctan2(z, w) on the seeded inputs of svml_model.host_numpy_uses_svml, as NumPy's SVML
# routines compute them.  Fixed here rather than asked of oracle/svml_model.py, which reads the same seed tables as the
# kernels: a changed table must make the tests below fail, not switch them to a reference built from that table.
SVML_OUTPUT_SHA256 = "cf3bf014c23406b0178c922e7d90920def40d2b7d07072c2bda0c75f63cb62e9"


def numpy_uses_svml() -> bool:
    import hashlib

    rng = np.random.default_rng(123)
    z = rng.uniform(-1, 1, 20000).astype(np.float32)
    w = rng.uniform(-1, 1, 20000).astype(np.float32)
    return hashlib.sha256(np.arccos(z).tobytes() + np.arctan2(z, w).tobytes()).hexdigest() == SVML_OUTPUT_SHA256


def _bits(x):
    return np.ascontiguousarray(x, np.float32).view(np.uint32)


def build_probe(out_dir: Path) -> Path:
    """Compile the probe with the library's own nvcc flags (no fast-math, no flush-to-zero) for sm_100a."""
    import __graft_entry__ as g

    b = g._load_build_module()
    so = Path(out_dir) / "device_math_probe.so"
    cmd = [b.find_nvcc(), *b.NVCC_FLAGS, "-I", str(CSRC), "-o", str(so), str(PROBE_SRC)]
    res = subprocess.run(cmd, capture_output=True, text=True)
    assert res.returncode == 0, "nvcc failed:\n" + " ".join(cmd) + "\n" + res.stdout + res.stderr
    return so


PROTOTYPES = {
    "probe_sqrt": [C.c_uint32, C.c_uint32, C.c_void_p],
    "probe_div": [C.c_uint32, C.c_uint32, C.c_int, C.c_int, C.c_int, C.c_uint32, C.c_void_p],
    "probe_round": [C.c_uint32, C.c_void_p],
    "probe_eval": [C.c_int, C.c_void_p, C.c_void_p, C.c_uint32, C.c_longlong, C.c_void_p],
    "probe_unit_pairs": [C.c_uint32, C.c_ulonglong, C.c_longlong, C.c_void_p, C.c_void_p],
    "probe_accuracy": [C.c_int, C.c_void_p, C.c_void_p, C.c_uint32, C.c_longlong, C.c_void_p],
}


def load_probe(so: Path) -> C.CDLL:
    lib = C.CDLL(str(so))
    for name, args in PROTOTYPES.items():
        fn = getattr(lib, name)
        fn.restype = C.c_int
        fn.argtypes = args
    return lib


def test_probe_builds_for_sm100a(tmp_path):
    """A broken probe shows up without a GPU: it compiles for sm_100a against the current header and exports every
    launcher the GPU tests call."""
    load_probe(build_probe(tmp_path))


# ------------------------------------------------------------------------------------------------------------------
# GPU
# ------------------------------------------------------------------------------------------------------------------
class Probe:
    def __init__(self, lib):
        import torch

        self.lib, self.torch = lib, torch
        self.dev = torch.device("cuda:0")

    def _run(self, name, *args):
        rc = getattr(self.lib, name)(*args)
        assert rc == 0, f"{name}: CUDA error {rc}"
        self.torch.cuda.synchronize()
        return rc

    def counters(self, n=8, init=None):
        t = self.torch.zeros(n, dtype=self.torch.int64, device=self.dev)
        if init:
            for i, v in init.items():
                t[i] = v
        return t

    def tensor(self, a):
        return self.torch.from_numpy(np.ascontiguousarray(a, np.float32)).to(self.dev)

    def eval(self, fn, a=None, b=None, base=0, n=None):
        n = int(a.numel() if a is not None else n)
        out = self.torch.empty(n, dtype=self.torch.float32, device=self.dev)
        self._run("probe_eval", fn, a.data_ptr() if a is not None else None,
                  b.data_ptr() if b is not None else None, base, n, out.data_ptr())
        return out

    def accuracy(self, fn, st, a=None, b=None, base=0, n=None):
        n = int(a.numel() if a is not None else n)
        self._run("probe_accuracy", fn, a.data_ptr() if a is not None else None,
                  b.data_ptr() if b is not None else None, base, n, st.data_ptr())

    def unit_pairs(self, seed, first, n):
        y = self.torch.empty(n, dtype=self.torch.float32, device=self.dev)
        x = self.torch.empty(n, dtype=self.torch.float32, device=self.dev)
        self._run("probe_unit_pairs", seed, first, n, y.data_ptr(), x.data_ptr())
        return y, x


@pytest.fixture(scope="module")
def probe(proj):
    with tempfile.TemporaryDirectory(prefix="p2p_probe_") as d:
        yield Probe(load_probe(build_probe(Path(d))))


def _stats(st):
    s = [int(v) for v in st.cpu().tolist()]
    n, cr, und = s[0], s[1], s[2]
    return dict(n=n, correctly_rounded=cr, undecided=und, cr_fraction=cr / max(1, n - und),
                max_ulp=float(np.uint32(s[3]).view(np.float32)), over_1ulp=s[4], nan=s[5])


def _record(name, stats):
    print("DEVICE_MATH " + json.dumps({"function": name, **stats}))


def _mismatch_count(got, want):
    """Elements whose bits differ; two NaNs of any payload agree."""
    import torch

    gb = got.view(torch.int32)
    wb = want.view(torch.int32)
    both_nan = torch.isnan(got) & torch.isnan(want)
    return int(((gb != wb) & ~both_nan).sum().item())


# ---- IEEE sqrt and division ---------------------------------------------------------------------------------------
SQRT_OPERAND_MIN = 0x2B800000   # 2^-40: ss = x^2 + y^2 + f^2 > f^2 with f > 2^-20


@pytest.mark.gpu
def test_sqrt_rn_fast_every_positive_normal(probe):
    """sqrt_rn_fast against __fsqrt_rn on every positive normal float (2^31 - 2^24 inputs): bit-equal on every operand
    the kernels can produce (ss >= 2^-40) and above; the inputs where the residual FMA underflows all lie below 2^-102."""
    res = probe.counters(3, {1: -1})
    probe._run("probe_sqrt", 0x00800000, 0x7F800000, res.data_ptr())
    bad, lo, hi = (int(v) & 0xFFFFFFFF for v in res.cpu().tolist())
    print(f"DEVICE_MATH {json.dumps({'function': 'sqrt_rn_fast', 'mismatches': bad, 'min': hex(lo), 'max': hex(hi)})}")
    assert bad == 0 or hi < 0x0C800000, (bad, hex(lo), hex(hi))
    res = probe.counters(3, {1: -1})
    probe._run("probe_sqrt", SQRT_OPERAND_MIN, 0x7F800000, res.data_ptr())
    assert int(res[0].item()) == 0


@pytest.mark.gpu
def test_div_rn_with_rcp_every_divisor_mantissa(probe):
    """div_rn_with_rcp(a, d, rcp_refined(d)) is bit-equal to __fdiv_rn for every divisor mantissa in [1, 2) (2^23),
    divisor exponents cycling over [-20, 20] (the norm of the ray lies in (2^-20, 2^20.5)), 1,024 numerator mantissas
    per divisor (1.0, all ones, d's own, the one below it, then seeded) of both signs with |a / d| in (2^-25, 1]."""
    res = probe.counters(3)
    step = 1 << 20
    for m0 in range(0, 1 << 23, step):
        probe._run("probe_div", m0, m0 + step, -20, 41, 1024, 0x2024, res.data_ptr())
    bad, a, d = (int(v) for v in res.cpu().tolist())
    assert bad == 0, (bad, hex(a), hex(d))


# ---- cvRound(x * 32) ----------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_round_x32_and_quantise_every_coordinate(probe):
    """round_x32 (the magic-constant FMA) and quantise equal cvRound(f32(x * 32)) = __float2int_rn(__fmul_rn(x, 32))
    for every float x in [0, 32767): every coordinate a panorama of up to 32767 columns or rows can produce."""
    res = probe.counters(2)
    probe._run("probe_round", int(np.float32(32767.0).view(np.uint32)), res.data_ptr())
    assert [int(v) for v in res.cpu().tolist()] == [0, 0]


# ---- NumPy-exact (SVML) arccos / arctan2 ----------------------------------------------------------------------------
@pytest.mark.gpu
def test_acos_svml_every_float(probe):
    """acos_svml equals NumPy's f32 arccos for every one of the 2^32 floats (NaN compared as NaN-ness, +-0 by bits).
    On a host whose NumPy does not use SVML, the reference is oracle/svml_model.py on 2^20 seeded inputs."""
    torch = probe.torch
    if not numpy_uses_svml():
        rng = np.random.default_rng(7)
        x = np.concatenate([rng.integers(0, 1 << 32, 1 << 19, dtype=np.uint64).astype(np.uint32).view(np.float32),
                            rng.uniform(-1, 1, 1 << 19).astype(np.float32)])
        got = probe.eval(1, probe.tensor(x))
        with np.errstate(invalid="ignore"):
            want = torch.from_numpy(svml_model.acos(x).astype(np.float32)).to(probe.dev)
        assert _mismatch_count(got, want) == 0
        return
    chunk = 1 << 26
    idx = np.arange(chunk, dtype=np.uint32)
    bad = 0
    for base in range(0, 1 << 32, chunk):
        x = (idx + np.uint32(base)).view(np.float32)
        with np.errstate(invalid="ignore"):
            want = torch.from_numpy(np.arccos(x)).to(probe.dev)
        got = probe.eval(1, base=base, n=chunk)
        bad += _mismatch_count(got, want)
    assert bad == 0


def atan2_sets():
    """Host-built (y, x) pairs of atan2 input sets (i) - (iii):
    (i)   every 16-bit leading-mantissa pattern of the larger operand (the svml_rcp14 segment key) x 64 ratios
          t = min / max spanning [2^-26, 1] x 4 sign pairs, the larger operand alternating between y and x;
    (ii)  |y| == |x| and its nextafter neighbours (the edge of SVML's |y| < |x| branch), 4 sign pairs;
    (iii) +-0, NaN, +-inf against each other and against ordinary values."""
    rng = np.random.default_rng(11)
    pat = np.arange(1 << 16, dtype=np.uint32)
    e = rng.integers(-12, 1, pat.size).astype(np.int64)
    mx = ((e + 127).astype(np.uint32) << 23) | (pat << 7) | rng.integers(0, 128, pat.size, dtype=np.uint32)
    mx = mx.view(np.float32)
    t = np.exp2(np.linspace(-26.0, 0.0, 64))
    t[1:-1] *= np.exp2(rng.uniform(-0.2, 0.2, 62))
    mn = (mx[:, None].astype(np.float64) * t[None, :]).astype(np.float32)
    big = np.broadcast_to(mx[:, None], mn.shape)
    y_first = (np.arange(64) % 2 == 0)[None, :]
    y1 = np.where(y_first, big, mn).ravel()
    x1 = np.where(y_first, mn, big).ravel()
    m = rng.uniform(1e-6, 1.0, 1 << 16).astype(np.float32)
    lo, hi = np.nextafter(m, np.float32(0)), np.nextafter(m, np.float32(np.inf))
    y2 = np.concatenate([m, lo, hi, m, m])
    x2 = np.concatenate([m, m, m, lo, hi])
    special = np.array([0.0, -0.0, np.nan, np.inf, -np.inf, 1.0, -1.0, 1e-30, 3.0e38, 0.5], np.float32)
    y3, x3 = (a.ravel() for a in np.meshgrid(special, special))
    ys, xs = [], []
    for sy in (1, -1):
        for sx in (1, -1):
            ys += [y1 * np.float32(sy), y2 * np.float32(sy)]
            xs += [x1 * np.float32(sx), x2 * np.float32(sx)]
    ys.append(y3)
    xs.append(x3)
    return np.concatenate(ys).astype(np.float32), np.concatenate(xs).astype(np.float32)


def operand_domain(y, x):
    """Pairs like the kernels' atan2 operands, the components of a unit ray: finite and below 2 in magnitude.
    acos_svml / atan2_svml restate SVML's main path only; SVML sends NaN, inf and operands of extreme exponent to a
    scalar path of its own, which the kernels never reach."""
    return np.isfinite(y) & np.isfinite(x) & (np.abs(y) < 2) & (np.abs(x) < 2)


UNIT_PAIRS = 1 << 30
UNIT_CHUNK = 1 << 25


@pytest.mark.gpu
def test_atan2_svml_against_numpy(probe):
    """atan2_svml equals np.arctan2 on sets (i) - (iii) within the operand domain and on 2^30 seeded pairs shaped like
    the kernels' unit-vector operands (iv); and the pair identity the mirror kernels rely on,
    finish(core(y, x), y, -x) == np.arctan2(y, -x)."""
    torch = probe.torch
    strict = numpy_uses_svml()
    ref = np.arctan2 if strict else svml_model.atan2

    def check(y, x, yt, xt):
        with np.errstate(invalid="ignore"):
            w = torch.from_numpy(np.asarray(ref(y, x), np.float32)).to(probe.dev)
            wm = torch.from_numpy(np.asarray(ref(y, -x), np.float32)).to(probe.dev)
        return _mismatch_count(probe.eval(2, yt, xt), w), _mismatch_count(probe.eval(3, yt, xt), wm)

    y, x = atan2_sets()
    keep = operand_domain(y, x)
    y, x = y[keep], x[keep]
    if not strict:   # the NumPy model is slow: a seeded 2^20 subset
        k = np.random.default_rng(5).choice(y.size, 1 << 20, replace=False)
        y, x = y[k], x[k]
    assert check(y, x, probe.tensor(y), probe.tensor(x)) == (0, 0)
    n_unit = UNIT_PAIRS if strict else 1 << 20
    chunk = min(UNIT_CHUNK, n_unit)
    bad = [0, 0]
    for first in range(0, n_unit, chunk):
        yt, xt = probe.unit_pairs(0x5EED, first, chunk)
        b = check(yt.cpu().numpy(), xt.cpu().numpy(), yt, xt)
        bad = [bad[0] + b[0], bad[1] + b[1]]
    assert bad == [0, 0]


# ---- minimax mode (P2P_OPT_TRIG = 1) ------------------------------------------------------------------------------
@pytest.mark.gpu
def test_acos_fast_accuracy_every_float_in_domain(probe):
    """acos_fast against the device's double acos over every float in [-1, 1]: max error within the documented bound,
    never NaN inside the domain, NaN for |z| > 1, exactly 0 / f32(pi) at +1 / -1; the correctly rounded fraction is
    recorded and bounded."""
    st = probe.counters(6)
    probe.accuracy(0, st, base=0, n=F32_ONE + 1)
    probe.accuracy(0, st, base=NEG, n=F32_ONE + 1)
    s = _stats(st)
    _record("acos_fast", s)
    assert s["n"] == 2 * (F32_ONE + 1) and s["nan"] == 0
    assert s["max_ulp"] <= ACOS_FAST_MAX_ULP and s["cr_fraction"] >= ACOS_FAST_CR_MIN, s
    above = np.nextafter(np.float32(1), np.float32(2))
    z = np.array([1.0, -1.0, 0.0, -0.0, above, -above, 2.0, -7.5, np.inf, -np.inf, np.nan], np.float32)
    got = probe.eval(4, probe.tensor(z)).cpu().numpy()
    assert _bits(got[0]) == 0 and got[1] == F32_PI, got[:2]
    assert got[2] == got[3] == np.float32(np.pi / 2), got[2:4]
    assert np.isnan(got[4:]).all(), got[4:]


@pytest.mark.gpu
def test_atan2_fast_accuracy(probe):
    """atan2_fast against the device's double atan2 on the operand-domain pairs of sets (i) - (iv): max error within the
    documented bound; the correctly rounded fraction is recorded and bounded."""
    y, x = atan2_sets()
    keep = operand_domain(y, x) & ~((x == 0) & np.signbit(x))   # x = -0: see atan2_fast
    st_sets, st_unit = probe.counters(6), probe.counters(6)
    probe.accuracy(1, st_sets, probe.tensor(y[keep]), probe.tensor(x[keep]))
    for first in range(0, UNIT_PAIRS, UNIT_CHUNK):
        yt, xt = probe.unit_pairs(0x5EED, first, UNIT_CHUNK)
        probe.accuracy(1, st_unit, yt, xt)
    _record("atan2_fast sets (i)-(iii)", _stats(st_sets))
    _record("atan2_fast unit pairs (iv)", _stats(st_unit))
    both = (st_sets + st_unit).cpu()
    both[3] = max(int(st_sets[3].item()), int(st_unit[3].item()))
    s = _stats(both)
    _record("atan2_fast", s)
    assert s["nan"] == 0
    assert s["max_ulp"] <= ATAN2_FAST_MAX_ULP and s["cr_fraction"] >= ATAN2_FAST_CR_MIN, s


@pytest.mark.gpu
def test_mirror_phi_fast_every_float_in_domain(probe):
    """mirror_phi_fast(a) = pi - a (compensated) for every float a in [-pi/2, pi/2]: within 1 ulp of RN(pi - a)
    everywhere; the inputs where it is not correctly rounded are counted."""
    st = probe.counters(6)
    probe.accuracy(2, st, base=0, n=F32_HALF_PI + 1)
    probe.accuracy(2, st, base=NEG, n=F32_HALF_PI + 1)
    s = _stats(st)
    s["not_correctly_rounded"] = s["n"] - s["undecided"] - s["correctly_rounded"]
    _record("mirror_phi_fast", s)
    assert s["n"] == 2 * (F32_HALF_PI + 1) and s["nan"] == 0
    assert s["max_ulp"] <= 1.0 and s["over_1ulp"] == 0, s
