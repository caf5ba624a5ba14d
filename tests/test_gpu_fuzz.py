"""Randomised differential test: the CUDA path against the CPU oracle over random panorama sizes,
output sizes, FOVs, pitches and yaws (integer rolls and fractional), including sizes that take the
byte-store fallback, the per-pixel kernel and the mirror kernel."""
import numpy as np
import pytest

from oracle import fixedpoint as fp
from oracle import ref_port, svml_model, synth

pytestmark = pytest.mark.gpu


def _cases(n, seed):
    rng = np.random.default_rng(seed)
    out = []
    for _ in range(n):
        Wp = int(rng.choice([360, 720, 1000, 1024, 1536, 2048, 2880, 4096]))
        Hp = Wp // 2 if rng.random() < 0.8 else int(rng.integers(64, Wp))
        W = int(rng.choice([8, 30, 64, 72, 100, 128, 200, 256, 333, 400, 512]))
        H = int(rng.integers(5, 300))
        fov = int(rng.choice([20, 45, 60, 90, 100, 120, 150, 170]))
        pitches = sorted({int(x) for x in rng.choice([0, 1, 15, 30, 45, 60, 89, 90, 91, 120, 150, 179, 180], 3)})
        yaws = [int(x) for x in rng.choice([0, 90, 180, 270, 360, 45, 30, 1, 359, -90, 123], 3)]
        out.append((Wp, Hp, W, H, fov, yaws, pitches))
    return out


@pytest.mark.parametrize("case", _cases(24, 2024))
def test_random_configs_against_oracle(proj, case):
    Wp, Hp, W, H, fov, yaws, pitches = case
    noise = synth.noise(Wp, Hp, Wp + H)
    smooth = synth.smooth(Wp, Hp, Wp + H)
    got_n = proj.project_image(noise, yaws, pitches, W, H, fov)
    got_s = proj.project_image(smooth, yaws, pitches, W, H, fov)
    # When this host's NumPy evaluates arccos / arctan2 with SVML (AVX-512), the default device path is
    # bit-identical to the oracle; otherwise the reference itself differs in the last ulp on this host.
    strict = svml_model.host_numpy_uses_svml()
    with proj.slots(1) as (s,):
        proj.upload(s, noise)
        for j, p in enumerate(pitches):
            U, V = ref_port.pitch_mapping(W, H, fov, p, Wp, Hp)
            if strict:   # the default coordinates are NumPy's, bit for bit (NaN as NaN)
                Ud, Vd = proj.coords(W, H, fov, p, Wp, Hp)
                assert np.array_equal(Ud, U, equal_nan=True) and np.array_equal(Vd, V, equal_nan=True), (case, p)
            # sampler stage with the oracle's maps: bit-exact for every integer-roll yaw
            for y in yaws:
                ix, fx = fp.yaw_column_table(Wp, y)
                shift = fp.yaw_table_is_roll(ix, fx)
                if shift is not None:
                    assert np.array_equal(proj.sample_with_maps(s, shift, U, V),
                                          fp.sample_view(noise, U, V, yaw_shift=shift)), (case, y, p)
    total = exact = 0
    for i, y in enumerate(yaws):
        for j, p in enumerate(pitches):
            want_n = fp.project_view_single_pass(noise, y, p, W, H, fov)
            want_s = fp.project_view_single_pass(smooth, y, p, W, H, fov)
            # gradient-bounded panorama: <= 1 LSB, except on the rounding-chaotic seam half row where the
            # reference itself flips between the first and the last column (SURVEY App. A)
            d = np.abs(got_s[i, j].astype(np.int16) - want_s.astype(np.int16)).max(axis=-1)
            U, _ = ref_port.pitch_mapping(W, H, fov, p, Wp, Hp)
            seam = (U <= 1.0) | (U >= Wp - 2.0) | np.isnan(U)
            assert d[~seam].max(initial=0) <= 1, (case, y, p, int(d[~seam].max(initial=0)))
            if strict:
                assert np.array_equal(got_n[i, j], want_n) and np.array_equal(got_s[i, j], want_s), (case, y, p)
            same = (got_n[i, j] == want_n).all(axis=-1)
            total += same.size
            exact += int(same.sum())
    # small, strongly magnified or pole views have few pixels per 1/32-px bin edge: gate on the whole case
    assert exact / total >= 0.93, (case, exact / total)
