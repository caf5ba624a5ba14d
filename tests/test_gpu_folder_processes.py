"""A folder over several devices runs one worker process per listed device (``folder_pool``): the same file names and
bytes as one device, for a mixed folder (JPEG and PNG panoramas of two sizes, a progressive JPEG, a damaged JPEG the device
decoder declines, a file nothing can read), to JPEG and to PNG files.  On a one-GPU box the device is listed twice."""
import logging

import numpy as np
import pytest

from oracle import synth

pytestmark = pytest.mark.gpu

W, H, FOV, YAWS, PITCHES = 200, 120, 100, [0, 90, 45], [60, 120]   # yaw 45 is a column table on 1000-wide panoramas


def _alive(pid):
    from pathlib import Path

    try:
        stat = Path(f"/proc/{pid}/stat").read_text()
    except OSError:
        return False
    return stat.rsplit(")", 1)[1].split()[0] != "Z"


def _gone(pids, seconds=15.0):
    import time

    end = time.monotonic() + seconds
    while time.monotonic() < end and any(_alive(p) for p in pids):
        time.sleep(0.05)
    return not any(_alive(p) for p in pids)


@pytest.fixture(scope="module")
def folder(tmp_path_factory):
    cv2 = pytest.importorskip("cv2")
    src = tmp_path_factory.mktemp("mixed")
    for i in range(6):
        wh = (2048, 1024) if i % 3 == 0 else (1000, 500)
        ext = "png" if i % 2 else "jpg"
        assert cv2.imwrite(str(src / f"p{i}.{ext}"), synth.smooth(*wh, i))
    assert cv2.imwrite(str(src / "prog.jpg"), synth.noise(1024, 512, 7), [cv2.IMWRITE_JPEG_PROGRESSIVE, 1])
    assert cv2.imwrite(str(src / "deep.png"), synth.smooth(1024, 512, 8).astype(np.uint16) * 257)
    good = cv2.imencode(".jpg", synth.smooth(1024, 512, 9), [cv2.IMWRITE_JPEG_RST_INTERVAL, 8])[1].tobytes()
    seq = bytearray(good)
    seq[good.find(b"\xff\xd2", good.find(b"\xff\xda")) + 1] = 0xD5     # restart marker out of sequence
    (src / "seq.jpg").write_bytes(bytes(seq))
    (src / "broken.png").write_bytes(b"not an image")
    assert cv2.imread(str(src / "seq.jpg")) is not None and cv2.imread(str(src / "broken.png")) is None
    return src


def _device_lists(pkg):
    n = pkg._lib.load().p2p_device_count()
    return [[0, 0]] + ([list(range(n))] if n >= 2 else [])


def _bytes(out):
    return {p.name: p.read_bytes() for p in sorted(out.iterdir())}


@pytest.mark.parametrize("fmt", ["jpg", "png"])
def test_mixed_folder_same_files_as_one_device(pkg, folder, tmp_path, fmt, caplog):
    ref = tmp_path / "one"
    ref.mkdir()
    with caplog.at_level(logging.ERROR):
        read_one = pkg.process_image_batch(sorted(folder.iterdir()), ref, YAWS, PITCHES, W, H, num_workers=4,
                                           output_format=fmt, fov_deg=FOV)
    assert any("Failed to read image" in r.message and "broken.png" in r.message for r in caplog.records)
    want = _bytes(ref)
    assert len(want) == 9 * len(YAWS) * len(PITCHES)
    assert read_one[folder / "seq.jpg"] == "cv2.imread" and read_one[folder / "broken.png"] is None
    assert read_one[folder / "p0.jpg"] == read_one[folder / "p1.png"] == read_one[folder / "prog.jpg"] == "device"
    from p2p_b200 import folder_pool

    try:
        for i, devs in enumerate(_device_lists(pkg)):
            out = tmp_path / f"d{i}"
            out.mkdir()
            caplog.clear()
            with caplog.at_level(logging.ERROR):
                read = pkg.process_image_batch(sorted(folder.iterdir()), out, YAWS, PITCHES, W, H, num_workers=4,
                                               output_format=fmt, fov_deg=FOV, devices=devs)
            # a child's log lines are emitted by the parent's handlers
            assert [r.message for r in caplog.records if "broken.png" in r.message] == \
                [f"Failed to read image: {folder / 'broken.png'}"]
            assert read == read_one, devs
            got = _bytes(out)
            assert sorted(got) == sorted(want), devs
            for n in want:
                assert got[n] == want[n], (devs, n)
            # the CLI flag takes the same route
            out = tmp_path / f"cli{i}"
            pkg.cli(["--input_path", str(folder), "--output_path", str(out), "--FOV", str(FOV), "--output_width", str(W),
                     "--output_height", str(H), "--yaw_angles", *map(str, YAWS), "--pitch_angles", *map(str, PITCHES),
                     "--output_format", fmt, "--num_workers", "4", "--devices", *map(str, devs)])
            assert _bytes(out) == want, devs
    finally:
        folder_pool.close_shared()


def test_pool_is_kept_and_png_formats_reach_the_workers(pkg, folder, tmp_path, caplog):
    """A second call with the same devices reuses the worker processes; ``set_png_formats`` between calls reaches them
    (the 16-bit PNG is read by cv2.imread before, on the device after: same pixels, so only the decoder tells); the info
    lines of the workers appear in the parent; ``close`` leaves no worker behind."""
    from p2p_b200 import folder_pool

    files, deep = sorted(folder.iterdir()), folder / "deep.png"
    (tmp_path / "a").mkdir()
    (tmp_path / "b").mkdir()
    try:
        with caplog.at_level(logging.INFO):
            read = pkg.process_image_batch(files, tmp_path / "a", YAWS, PITCHES, W, H, num_workers=4, output_format="png",
                                           fov_deg=FOV, devices=[0, 0])
        assert read[deep] == "cv2.imread"
        assert sorted(r.message for r in caplog.records if r.message.startswith("Loading image: ")) == \
            sorted(f"Loading image: {f}" for f in files)
        pool = folder_pool.shared([0, 0], pkg.panorama_to_plane_pitch._folder_worker_body)
        pids = pool.pids
        assert len(pids) == 2 and all(_alive(p) for p in pids)
        pkg.set_png_formats(True)
        read = pkg.process_image_batch(files, tmp_path / "b", YAWS, PITCHES, W, H, num_workers=4, output_format="png",
                                       fov_deg=FOV, devices=[0, 0])
        assert read[deep] == "device"
        assert folder_pool.shared([0, 0], pkg.panorama_to_plane_pitch._folder_worker_body).pids == pids
        assert _bytes(tmp_path / "a") == _bytes(tmp_path / "b")
    finally:
        pkg.set_png_formats(False)
        folder_pool.close_shared()
    assert _gone(pids)
