"""CPU tests: the oracle against the golden vectors produced by the unmodified reference
(``oracle/gen_golden.py``), and the cv2-free integer model against real ``cv2.remap``."""
import hashlib
import json

import numpy as np
import pytest

from oracle import fixedpoint as fp
from oracle import golden, ref_port, synth


def sha(a):
    return hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()


@pytest.fixture(scope="module")
def same_numpy_path():
    """The golden vectors were produced where NumPy evaluates f32 arccos / arctan2 with SVML (AVX-512).
    On a host where NumPy takes another path the reference itself differs in the last ulp, so the
    bit-exact oracle-vs-golden comparisons do not apply there."""
    from oracle import svml_model

    if not svml_model.host_numpy_uses_svml():
        pytest.skip("host NumPy does not use the AVX-512 SVML arccos / arctan2: reference bits differ here")


@pytest.fixture(scope="module")
def manifest(golden_dir):
    return json.loads((golden_dir / "manifest.json").read_text())


def load(golden_dir, name):
    return golden.load(golden_dir / name)


def test_synthetic_panoramas_are_reproducible(manifest):
    for key, want in manifest["pano_sha256"].items():
        kind, size, seed = key.split("_")
        Wp, Hp = map(int, size.split("x"))
        if Wp * Hp > 2048 * 1024:
            continue  # the big ones are covered by the hash tests below
        assert sha(synth.make(kind, Wp, Hp, int(seed[1:]))) == want, key


def test_golden_files_are_small_and_decode_exactly(golden_dir, tmp_path):
    """Every golden file stays under 1 MB; a file written with the encodings of ``oracle/golden.py`` loads back to exactly
    the arrays it was given, and views that the stored maps do not reproduce are refused."""
    for f in golden_dir.iterdir():
        assert f.stat().st_size < 1 << 20, f.name
    g = load(golden_dir, "c2_small.npz")
    golden.save(tmp_path / "ok.npz", g, dx=("out_smooth",), from_maps=("out_noise",))
    bad = dict(g, out_noise=g["out_noise"].copy())
    bad["out_noise"][1, 2, 5, 7, 0] ^= 1
    with pytest.raises(ValueError, match=r"views \(yaw index, pitch index\) \[\[1, 2\]\] differ"):
        golden.save(tmp_path / "bad.npz", bad, from_maps=("out_noise",))


def test_remap_model_matches_cv2_on_random_maps():
    cv2 = pytest.importorskip("cv2")
    rng = np.random.default_rng(7)
    for (Hs, Ws, H, W) in [(129, 257, 200, 300), (64, 64, 50, 70), (500, 1000, 120, 90)]:
        src = rng.integers(0, 256, (Hs, Ws, 3), dtype=np.uint8)
        U = rng.uniform(-3, Ws + 3, (H, W)).astype(np.float32)
        V = rng.uniform(-3, Hs + 3, (H, W)).astype(np.float32)
        U[0, :10] = np.arange(10)
        V[0, :10] = Hs - 1
        U[1, :5] = Ws - 1
        U[2, 3] = np.nan
        V[3, 4] = np.nan
        U[4, :8] = np.arange(8) + 0.015625  # exactly representable half-steps of the 1/32 grid
        V[4, :8] = np.arange(8) + 0.046875
        want = cv2.remap(src, U, V, interpolation=cv2.INTER_LINEAR, borderMode=cv2.BORDER_CONSTANT)
        assert np.array_equal(fp.remap_fixedpoint(src, U, V), want)


def test_c1_reference_case(golden_dir, same_numpy_path):
    g = load(golden_dir, "c1.npz")
    pano = synth.noise(int(g["Wp"]), int(g["Hp"]), 0)
    W, H, fov = int(g["W"]), int(g["H"]), int(g["fov"])
    ref_port.clear_caches()
    two_pass = ref_port.process_yaw_and_pitchs(pano, 0, [90], W, H, fov)[0]
    assert np.array_equal(two_pass, g["out"][0, 0])
    assert np.array_equal(fp.project_view_single_pass(pano, 0, 90, W, H, fov), g["out"][0, 0])


def test_c2_small_all_views_and_maps(golden_dir, same_numpy_path):
    g = load(golden_dir, "c2_small.npz")
    Wp, Hp, W, H, fov = (int(g[k]) for k in ("Wp", "Hp", "W", "H", "fov"))
    yaws, pitches = list(g["yaws"]), list(g["pitches"])
    for j, p in enumerate(pitches):
        U, V = ref_port.pitch_mapping(W, H, fov, int(p), Wp, Hp)
        assert np.array_equal(U, g["U"][j]) and np.array_equal(V, g["V"][j])
        Us, Vs = fp.pitch_coords_scalar_model(W, H, fov, int(p), Wp, Hp)
        assert np.array_equal(Us, g["U"][j]) and np.array_equal(Vs, g["V"][j])
    ref_port.clear_caches()
    for kind in ("noise", "smooth"):
        pano = synth.make(kind, Wp, Hp, 0)
        for i, y in enumerate(yaws):
            two_pass = ref_port.process_yaw_and_pitchs(pano, int(y), [int(p) for p in pitches], W, H, fov)
            for j, p in enumerate(pitches):
                want = g[f"out_{kind}"][i, j]
                assert np.array_equal(two_pass[j], want)
                assert np.array_equal(fp.project_view_single_pass(pano, int(y), int(p), W, H, fov), want)


def test_c5_small_cube_faces_and_poles(golden_dir, same_numpy_path):
    g = load(golden_dir, "c5_small.npz")
    Wp, Hp, W, H, fov = (int(g[k]) for k in ("Wp", "Hp", "W", "H", "fov"))
    pano = synth.noise(Wp, Hp, 0)
    for k, (y, p) in enumerate(g["views"]):
        assert np.array_equal(fp.project_view_single_pass(pano, int(y), int(p), W, H, fov), g["out"][k]), (y, p)
    for j, p in enumerate(g["map_pitches"]):
        U, V = fp.pitch_coords_scalar_model(W, H, fov, int(p), Wp, Hp)
        assert np.array_equal(U, g["U"][j], equal_nan=True) and np.array_equal(V, g["V"][j], equal_nan=True)


def test_fractional_yaw_two_stage(golden_dir, same_numpy_path):
    g = load(golden_dir, "frac_yaw.npz")
    Wp, Hp, W, H, fov = (int(g[k]) for k in ("Wp", "Hp", "W", "H", "fov"))
    pano = synth.noise(Wp, Hp, 0)
    for i, y in enumerate(g["yaws"]):
        assert np.array_equal(ref_port.yaw_row(Wp, int(y)), g["yaw_rows"][i])
        for j, p in enumerate(g["pitches"]):
            assert np.array_equal(fp.project_view_single_pass(pano, int(y), int(p), W, H, fov), g["out"][i, j]), (y, p)
    ix, fx = fp.yaw_column_table(Wp, 360)
    assert fp.yaw_table_is_roll(ix, fx) == 0
    ix, fx = fp.yaw_column_table(Wp, 30)
    assert fp.yaw_table_is_roll(ix, fx) is None


def test_nan_coordinate_gives_black_pixel(golden_dir, same_numpy_path):
    g = load(golden_dir, "nan_case.npz")
    Wp, Hp, W, H, fov = (int(g[k]) for k in ("Wp", "Hp", "W", "H", "fov"))
    pano = synth.smooth(Wp, Hp, 0)
    nan_px = g["nan_px"]
    assert len(nan_px) >= 1
    for j, p in enumerate(g["pitches"]):
        out = fp.project_view_single_pass(pano, 0, int(p), W, H, fov)
        assert np.array_equal(out, g["out"][0, j])
    for (j, v, u) in nan_px:
        assert (g["out"][0, j, v, u] == 0).all()
        U, V = fp.pitch_coords_scalar_model(W, H, fov, int(g["pitches"][j]), Wp, Hp)
        assert np.isnan(V[v, u])


def test_fma32_is_correctly_rounded():
    rng = np.random.default_rng(3)
    a = rng.standard_normal(200000).astype(np.float32)
    b = rng.standard_normal(200000).astype(np.float32)
    c = (-(a.astype(np.float64) * b.astype(np.float64)) * (1 + rng.standard_normal(200000) * 1e-7)).astype(np.float32)
    got = fp.fma32(a, b, c)
    # exact value with integer arithmetic on the mantissas via Python fractions on a subsample
    from fractions import Fraction

    for i in range(0, 200000, 997):
        exact = Fraction(float(a[i])) * Fraction(float(b[i])) + Fraction(float(c[i]))
        lo = np.nextafter(got[i], np.float32(-np.inf))
        hi = np.nextafter(got[i], np.float32(np.inf))
        d = abs(Fraction(float(got[i])) - exact)
        assert d <= abs(Fraction(float(lo)) - exact) and d <= abs(Fraction(float(hi)) - exact)


def test_full_size_c2_hashes(manifest, same_numpy_path):
    """BASELINE config 2 at full size: 8192x4096 -> 12 x 1920x1080; the single-pass oracle must
    reproduce the reference bit for bit (sha256 of every view)."""
    want = manifest["hashes"]["c2_noise"]
    pano = synth.noise(8192, 4096, 0)
    assert sha(pano) == manifest["pano_sha256"]["noise_8192x4096_s0"]
    for i, y in enumerate([0, 90, 180, 270]):
        for j, p in enumerate([30, 60, 90]):
            if (i + j) % 2:  # half of the views keeps the CPU suite short; the rest run on the GPU box
                continue
            assert sha(fp.project_view_single_pass(pano, y, p, 1920, 1080, 120)) == want[i][j], (y, p)


def test_full_size_c5_pole_face_hash(manifest, same_numpy_path):
    want = manifest["hashes"]["c5_noise"]
    pano = synth.noise(8192, 4096, 0)
    faces = [(0, 90), (90, 90), (180, 90), (270, 90), (0, 0), (0, 180)]
    for k in (1, 5):  # the seam face and a pole face
        y, p = faces[k]
        assert sha(fp.project_view_single_pass(pano, y, p, 2048, 2048, 90)) == want[k]


def test_exact_bilinear_oracle_arithmetic_model():
    """The optional exact-bilinear mode is pinned against scipy.ndimage.map_coordinates(order=1); this
    checks the arithmetic the CUDA kernel implements (double precision, weights 1 - frac and
    1 - (1 - frac), C-order taps, row weight then column weight, +0.5 and truncation) against scipy."""
    pytest.importorskip("scipy")
    from oracle import exact_bilinear as eb

    rng = np.random.default_rng(0)
    Wp, Hp, W, H = 257, 129, 300, 200
    pano = synth.noise(Wp, Hp, 1)
    U = rng.uniform(0, Wp - 1, (H, W)).astype(np.float32)
    V = rng.uniform(0, Hp - 1, (H, W)).astype(np.float32)
    U[0, :] = Wp - 1
    V[1, :] = Hp - 1
    U[2, :8] = np.arange(8) + 0.5
    V[2, :8] = np.arange(8) + 0.5
    want = eb.sample_view_exact(pano, U, V, 5)
    r = np.roll(pano, -5, axis=1).astype(np.float64)
    xf, yf = np.floor(U), np.floor(V)
    ix, iy = xf.astype(int), yf.astype(int)
    fx, fy = (U - xf).astype(np.float64), (V - yf).astype(np.float64)
    wy0 = 1 - fy
    wy1 = 1 - wy0
    wx0 = 1 - fx
    wx1 = 1 - wx0
    ix1, iy1 = np.minimum(ix + 1, Wp - 1), np.minimum(iy + 1, Hp - 1)
    acc = np.zeros((H, W, 3))
    for yy, xx, wy, wx in ((iy, ix, wy0, wx0), (iy, ix1, wy0, wx1), (iy1, ix, wy1, wx0), (iy1, ix1, wy1, wx1)):
        acc = acc + (r[yy, xx] * wy[..., None]) * wx[..., None]
    got = np.minimum(np.where(acc > 0, acc + 0.5, 0), 255).astype(np.uint8)
    assert np.array_equal(got, want)


def test_svml_model_reproduces_numpy_arccos_arctan2():
    """NumPy evaluates f32 arccos / arctan2 with Intel SVML on AVX-512 hosts; the operation-by-operation
    model (which the CUDA kernels restate) must agree bit for bit, including +-1, +-0, |x| > 1 and NaN."""
    from oracle import svml_model as sm

    if not sm.host_numpy_uses_svml():
        pytest.skip("this host's NumPy does not take the AVX-512 SVML path")
    rng = np.random.default_rng(0)
    z = np.concatenate([rng.uniform(-1, 1, 1_500_000), 1 - np.logspace(-7.5, -1, 100_000),
                        -1 + np.logspace(-7.5, -1, 100_000),
                        [1, -1, 0, -0.0, 0.5, -0.5, 0.25, 1.0000001, -1.0000001, np.nan]]).astype(np.float32)
    with np.errstate(invalid="ignore"):
        want = np.arccos(z)
    got = sm.acos(z)
    assert np.array_equal(want.view(np.uint32)[~np.isnan(want)], got.view(np.uint32)[~np.isnan(want)])
    assert np.array_equal(np.isnan(want), np.isnan(got))
    y = np.concatenate([rng.uniform(-1, 1, 1_500_000), rng.uniform(-1e-6, 1e-6, 100_000),
                        [0, 0, -0.0, 0.3, -0.3, 0, -0.0]]).astype(np.float32)
    x = np.concatenate([rng.uniform(-1, 1, 1_500_000), rng.uniform(-1, 1, 100_000),
                        [0, -0.0, 0.0, 0, -0.0, 0.5, -0.5]]).astype(np.float32)
    assert np.array_equal(np.arctan2(y, x).view(np.uint32), sm.atan2(y, x).view(np.uint32))
    # and the golden maps of the reference follow from it (rotated ray from the scalar model)
