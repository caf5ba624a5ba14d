"""GPU tests of fractional yaws (no integer column roll, ``yaw_table(...)[2] is None``) through the flat view list
(``p2p_project_view_list_tables``: table groups of the row-segment kernel), its row bands and partial slots, the view-list
file entries (``p2p_process_view_list_jpeg`` / ``_png``), the front end's files flows and the split of one image over
several GPUs.  The yardstick is the existing one-pass fractional API (``project_tables``, itself pinned to the two
materialised remap passes) and, for integer rolls, ``project``."""
import ctypes as C
import shutil
import subprocess
from pathlib import Path

import numpy as np
import pytest

from oracle import fixedpoint as fp
from oracle import golden, svml_model, synth

pytestmark = pytest.mark.gpu

ROOT = Path(__file__).resolve().parent.parent


def _reference(pkg, proj, slot, tables, consts, W, H):
    """[n_yaw, n_pitch] views of a resident panorama through the per-product APIs: project (integer rolls) and
    project_tables (fractional yaws)."""
    out = np.empty((len(tables), len(consts), H, W, 3), np.uint8)
    for k, t in enumerate(tables):
        if t[2] is None:
            out[k] = proj.project_tables(slot, [t], consts, W, H)[0]
        else:
            out[k] = proj.project(slot, [t[2]], consts, W, H)[0]
        proj.sync(slot)
    return out


CASES = [   # Wp, Hp, W, H, fov, yaws, pitches
    (1000, 500, 200, 121, 100, [0.5, 37, 90, 181, 359.9, 30], [0, 1, 90, 179, 180]),
    (1024, 512, 256, 135, 120, [0, 30, 45, 60, 90, 359.9, 0.1], [30, 90, 150]),
    (777, 388, 64, 63, 90, [359, 1, 123, 200, 271, 33, 77], [0, 60, 180]),
    (2040, 1020, 163, 91, 120, [45, 10.25, 100, 90], [1, 90, 179]),
]


@pytest.mark.parametrize("trig", [0, 1])
@pytest.mark.parametrize("case", range(len(CASES)))
def test_list_tables_equal_per_view_apis(pkg, proj, case, trig):
    """Mixed integer / fractional lists in shuffled order with duplicates: same bytes as project_tables / project and as
    project_any; pole pitches, the clipped last columns (yaws next to 0 / 360: ix = Wp - 1), W % 8 != 0 (per-view
    fallback), odd H, both trig modes."""
    Wp, Hp, W, H, fov, yaws, pitches = CASES[case]
    pano = synth.noise(Wp, Hp, Wp + case)
    tables = [pkg.yaw_table(Wp, y) for y in yaws]
    consts = [pkg.pitch_constants(W, fov, p) for p in pitches]
    assert any(t[2] is None for t in tables)
    proj.set_option(pkg._lib.OPT_TRIG, trig)
    try:
        with proj.slots(1) as (s,):
            proj.upload(s, pano)
            want = _reference(pkg, proj, s, tables, consts, W, H)
            assert np.array_equal(proj.project_any(s, tables, consts, W, H), want)
            rng = np.random.default_rng(case)
            views = [(k, j) for k in range(len(yaws)) for j in range(len(pitches))]
            order = list(rng.permutation(len(views))) + [0, 0, len(views) - 1]
            got = proj.project_list_tables(s, [tables[views[i][0]] for i in order],
                                           [consts[views[i][1]] for i in order], W, H)
            proj.sync(s)
        for n, i in enumerate(order):
            k, j = views[i]
            assert np.array_equal(got[n], want[k, j]), (case, trig, yaws[k], pitches[j])
    finally:
        proj.set_option(pkg._lib.OPT_TRIG, 0)


def test_more_than_48_groups_and_launch_counts(pkg, proj):
    """A fractional-only list of <= 48 groups is one launch, a mixed list two; 64 table groups split over launches and
    still equal project_tables."""
    Wp, Hp, W, H, fov = 1000, 500, 64, 40, 100
    pano = synth.noise(Wp, Hp, 3)
    frac = [pkg.yaw_table(Wp, y) for y in (1.5, 30, 61, 95.5, 130, 170, 210.25, 250, 290, 330, 355, 359.9, 12.3)]
    assert all(t[2] is None for t in frac)
    consts = [pkg.pitch_constants(W, fov, p) for p in range(10, 170, 10)]   # 16 pitches x 13 yaws = 64 groups
    with proj.slots(1) as (s,):
        proj.upload(s, pano)
        want = proj.project_tables(s, frac, consts, W, H)
        proj.sync(s)
        flat_t = [t for t in frac for _ in consts]
        flat_c = consts * len(frac)
        got = proj.project_list_tables(s, flat_t, flat_c, W, H)
        proj.sync(s)
        assert np.array_equal(got.reshape(want.shape), want)
        n0 = proj.launches
        proj.project_list_tables(s, frac[:8], consts[:1] * 8, W, H)           # 2 groups
        proj.sync(s)
        assert proj.launches - n0 == 1
        n0 = proj.launches
        mixed = [frac[0], pkg.yaw_table(Wp, 90), frac[1], pkg.yaw_table(Wp, 180)] * 3
        proj.project_list_tables(s, mixed, consts[:3] * 4, W, H)
        proj.sync(s)
        assert proj.launches - n0 == 2


def test_pinned_values_oracle_and_golden(pkg, proj):
    """Fractional views of the list entry against the oracle's single-pass model and the reference's stored outputs."""
    Wp, Hp, W, H, fov = 1024, 512, 240, 136, 120
    pano = synth.noise(Wp, Hp, 0)
    views = [(33.3, 60), (0, 90), (123.3, 30), (60, 150), (33.3, 150)]
    strict = svml_model.host_numpy_uses_svml()
    with proj.slots(1) as (s,):
        proj.upload(s, pano)
        got = proj.project_list_tables(s, [pkg.yaw_table(Wp, y) for y, _ in views],
                                       [pkg.pitch_constants(W, fov, p) for _, p in views], W, H)
        proj.sync(s)
    for i, (y, p) in enumerate(views):
        want = fp.project_view_single_pass(pano, y, p, W, H, fov)
        frac = float((got[i] == want).all(axis=-1).mean())
        assert frac >= (1.0 if strict else 0.96), (y, p, frac)
    g = golden.load(ROOT / "tests" / "golden" / "frac_yaw.npz")
    Wp, Hp, W, H, fov = (int(g[k]) for k in ("Wp", "Hp", "W", "H", "fov"))
    yaws, pitches = [int(y) for y in g["yaws"]], [int(p) for p in g["pitches"]]
    with proj.slots(1) as (s,):
        proj.upload(s, synth.noise(Wp, Hp, 0))
        got = proj.project_list_tables(s, [pkg.yaw_table(Wp, y) for y in yaws for _ in pitches],
                                       [pkg.pitch_constants(W, fov, p) for _ in yaws for p in pitches], W, H)
        proj.sync(s)
    got = got.reshape(g["out"].shape)
    for i in range(len(yaws)):
        for j in range(len(pitches)):
            if strict:
                assert np.array_equal(got[i, j], g["out"][i, j]), (yaws[i], pitches[j])
            else:
                assert float((got[i, j] == g["out"][i, j]).all(axis=-1).mean()) >= 0.96


@pytest.mark.parametrize("W,H", [(256, 135), (250, 99)])
def test_row_bands_partial_slots_and_refusals(pkg, proj, W, H):
    from p2p_b200 import shard

    Wp, Hp, fov = 1000, 500, 100
    pano = synth.noise(Wp, Hp, 7)
    views = [(30, 45), (90, 45), (181.5, 90), (30, 135)]
    tables = [pkg.yaw_table(Wp, y) for y, _ in views]
    consts = [pkg.pitch_constants(W, fov, p) for _, p in views]
    with proj.slots(2) as (s, b):
        proj.upload(s, pano)
        full = proj.project_list_tables(s, tables, consts, W, H)
        proj.sync(s)
        for world in (2, 3):
            out = np.full((len(views), H, W, 3), 0xAB, np.uint8)
            for r in range(world):
                proj.project_list_tables(s, tables, consts, W, H, rows=shard.shard_rows(H, r, world), out=out)
                proj.sync(s)
            assert np.array_equal(out, full), world
        # a slot holding only the rows the views touch; one row short is refused
        lo, hi = proj.view_row_range(consts, W, H, Wp, Hp)
        proj.upload_rows(b, synth.noise(64, 32, 1), 0, 10)   # another size first: b forgets what it held
        proj.upload_rows(b, pano, lo + 1, hi + 1)
        with pytest.raises(pkg.P2PError) as e:
            proj.project_list_tables(b, tables, consts, W, H)
        assert e.value.code == -4
        proj.upload_rows(b, pano, lo, lo + 1)        # the missing row: the slot now holds rows lo .. hi
        got = proj.project_list_tables(b, tables, consts, W, H)
        proj.sync(b)
        assert np.array_equal(got, full)
        # bad tables
        ix, fx, _ = tables[0]
        for bad in ((np.full_like(ix, Wp), fx), (ix, np.full_like(fx, 32)), (ix, -np.ones_like(fx))):
            with pytest.raises(pkg.P2PError) as e:
                proj.project_list_tables(s, [(bad[0], bad[1], None)], consts[:1], W, H)
            assert e.value.code == -1 and "out of range" in str(e.value)
        lib = pkg._lib.load()
        P = C.POINTER(C.c_int32)
        sh = (C.c_int32 * 1)(-1)
        outb = np.empty((1, H, W, 3), np.uint8)
        rc = lib.p2p_project_view_list_tables(proj.ctx, s, 1, sh, (P * 1)(), (P * 1)(), proj._consts_array(consts[:1]),
                                              W, H, 0, H, outb.ctypes.data, 0)
        assert rc == -1 and lib.p2p_last_error(proj.ctx) == b"null yaw table"
        rc = lib.p2p_project_view_list_tables(proj.ctx, s, 1, sh, None, None, proj._consts_array(consts[:1]),
                                              W, H, 0, H, outb.ctypes.data, 0)
        assert rc == -1
        # the exact-bilinear mode stays integer-roll only
        proj.set_option(pkg._lib.OPT_INTERP, 1)
        try:
            with pytest.raises(pkg.P2PError) as e:
                proj.project_list_tables(s, tables[:1], consts[:1], W, H)
            assert e.value.code == -1
        finally:
            proj.set_option(pkg._lib.OPT_INTERP, 0)


@pytest.mark.parametrize("Wp,Hp,W,H", [(1000, 500, 200, 120), (1000, 500, 1, 1), (1000, 500, 8, 2), (8192, 4096, 1920, 1080)])
def test_view_list_files_equal_cv2(pkg, proj, Wp, Hp, W, H):
    """Files of process_view_list_jpeg / _png = cv2.imencode of the project_tables / project views: panorama decoded into
    the slot from a JPEG and from a PNG file, and host pixels with partial upload."""
    cv2 = pytest.importorskip("cv2")
    big = Wp >= 8192
    pano = synth.smooth(Wp, Hp, 2)
    yaws, pitches = ([33.3, 90], [60]) if big else ([33.3, 90, 30], [60, 120])
    tables = [pkg.yaw_table(Wp, y) for y in yaws]
    consts = [pkg.pitch_constants(W, 100, p) for p in pitches]
    flat_t = [t for t in tables for _ in consts]
    flat_c = consts * len(tables)
    sources = [("host", pano)]
    for ext in ((".jpg",) if big else (".jpg", ".png")):
        ok, enc = cv2.imencode(ext, pano)
        assert ok
        sources.append((ext, enc.tobytes()))
    for name, src in sources:
        with proj.slots(1) as (s,):
            if name == "host":
                img, pix = src, src
            else:
                proj.upload_encoded(s, src)
                img, pix = None, cv2.imdecode(np.frombuffer(src, np.uint8), cv2.IMREAD_COLOR)
            jpg = proj.process_view_list_jpeg(s, img, flat_t, flat_c, W, H)
            png, pixels = proj.process_view_list_png(s, img, flat_t, flat_c, W, H, want_pixels=True)
            with proj.slots(1) as (r,):
                proj.upload(r, pix)
                want = _reference(pkg, proj, r, tables, consts, W, H).reshape(-1, H, W, 3)
        assert np.array_equal(pixels, want), name
        for i in range(len(flat_t)):
            assert jpg[i] == cv2.imencode(".jpg", want[i])[1].tobytes(), (name, i)
            assert png[i] == cv2.imencode(".png", want[i])[1].tobytes(), (name, i)


@pytest.mark.parametrize("fmt", ["png", "jpg"])
def test_front_end_fractional_files_stay_on_device(pkg, tmp_path, monkeypatch, fmt):
    """``main`` over a folder (and a single file) of JPEG and PNG panoramas with fractional yaws: the files equal cv2 of
    process_yaw_and_pitchs, and no pixels reach the host (the host-pixel routes are patched to raise)."""
    cv2 = pytest.importorskip("cv2")
    src = tmp_path / "in"
    src.mkdir()
    Wp, Hp, W, H, fov = 1024, 512, 200, 120, 100
    yaws, pitches = [0, 30, 45, 60, 90], [60, 120]
    for i, ext in enumerate(("jpg", "png", "jpg")):
        assert cv2.imwrite(str(src / f"p{i}.{ext}"), synth.smooth(Wp, Hp, i))
    want = {}
    for f in sorted(src.iterdir()):
        img = cv2.imread(str(f))
        for y in yaws:
            for p, v in zip(pitches, pkg.process_yaw_and_pitchs(img, y, pitches, W, H, fov)):
                name = f"{f.stem}_{W}x{H}_yaw_{y}_pitch_{p}.{fmt}"
                want[name] = cv2.imencode("." + fmt, v)[1].tobytes()

    def boom(*a, **k):
        raise AssertionError("pixels went through the host")

    for name in ("decode_encoded", "project_image", "encode_jpeg", "encode_png"):
        monkeypatch.setattr(pkg.Projector, name, boom)
    out = tmp_path / "out"
    pkg.main(str(src), str(out), yaws, pitches, W, H, num_workers=2, output_format=fmt, fov_deg=fov)
    one = tmp_path / "one"
    pkg.main(str(src / "p1.png"), str(one), yaws, pitches, W, H, num_workers=2, output_format=fmt, fov_deg=fov)
    assert sorted(p.name for p in out.iterdir()) == sorted(want)
    for p in out.iterdir():
        assert p.read_bytes() == want[p.name], p.name
    for p in one.iterdir():
        assert p.read_bytes() == want[p.name], p.name
    assert len(list(one.iterdir())) == len(yaws) * len(pitches)


def _device_sets(pkg):
    n = pkg._lib.load().p2p_device_count()
    return [[0, 0]] + ([list(range(min(n, 4)))] if n >= 2 else [])


def test_split_with_fractional_yaws_identical(pkg, tmp_path):
    """One image split over devices (a device listed twice plays two GPUs) with fractional yaws: pixels and files equal
    the single-device path."""
    cv2 = pytest.importorskip("cv2")
    from p2p_b200 import panorama_to_plane_pitch as front

    Wp, Hp, W, H, fov = 1000, 500, 200, 120, 100
    yaws, pitches = [0, 30, 90, 33.3], [60, 120]
    pano = synth.noise(Wp, Hp, 11)
    one = front._project(pkg.get_projector(), pano, yaws, pitches, W, H, fov, devices=[])
    f = tmp_path / "pano.jpg"
    assert cv2.imwrite(str(f), synth.smooth(Wp, Hp, 4))
    for fmt in ("png", "jpg"):
        ref = tmp_path / f"ref_{fmt}"
        ref.mkdir()
        pkg.process_single_image(f, ref, yaws, pitches, W, H, num_workers=2, output_format=fmt, fov_deg=fov)
        names = sorted(p.name for p in ref.iterdir())
        assert len(names) == len(yaws) * len(pitches)
        for i, devs in enumerate(_device_sets(pkg)):
            out = tmp_path / f"split_{fmt}_{i}"
            out.mkdir()
            pkg.process_single_image(f, out, yaws, pitches, W, H, num_workers=2, output_format=fmt, fov_deg=fov,
                                     devices=devs)
            assert sorted(p.name for p in out.iterdir()) == names
            for n in names:
                assert (out / n).read_bytes() == (ref / n).read_bytes(), (devs, n)
    for devs in _device_sets(pkg):
        got = front._project(pkg.get_projector(), pano, yaws, pitches, W, H, fov, devices=devs)
        assert np.array_equal(got, one), devs


def test_plain_c_consumer_of_the_list_entry(pkg, tmp_path):
    gcc = shutil.which("gcc")
    if gcc is None:
        pytest.skip("gcc not available")
    exe = tmp_path / "c_fractional_list"
    libdir = pkg._lib.LIB_PATH.parent
    subprocess.run([gcc, "-std=c99", "-O1", f"-I{ROOT / 'include'}", str(ROOT / "tests" / "c_fractional_list.c"), "-o",
                    str(exe), f"-L{libdir}", "-lp2p_b200", f"-Wl,-rpath,{libdir}"], check=True)
    Wp, Hp, W, H, fov = 1000, 500, 200, 120, 100
    out_file = tmp_path / "out.bin"
    run = subprocess.run([str(exe), str(Wp), str(Hp), str(W), str(H), str(fov), str(out_file)], capture_output=True,
                         text=True)
    assert run.returncode == 0, run.stderr
    s, vals = 12345, np.empty(Wp * Hp * 3, np.uint8)
    for i in range(vals.size):  # same LCG as the C program
        s = (s * 1664525 + 1013904223) & 0xFFFFFFFF
        vals[i] = s >> 24
    pano = vals.reshape(Hp, Wp, 3)
    got = np.fromfile(out_file, np.uint8).reshape(4, H, W, 3)
    want = pkg.Projector(0, n_slots=1).project_image(pano, [0, 33.3, 90], [60, 120], W, H, fov)
    for i, (k, j) in enumerate([(0, 0), (1, 0), (2, 1), (1, 1)]):
        assert np.array_equal(got[i], want[k, j]), i
