"""The worker-process pool of the directory front end (``folder_pool``), with stand-in bodies that call no GPU code: every
file handled exactly once whatever the number of workers, a worker that dies or raises is reported in the caller and its
files are not given to another worker, and no worker outlives ``close()`` or its parent."""
import logging
import os
import signal
import subprocess
import sys
import textwrap
import time
from pathlib import Path

import pytest


def marker_body(device, job, take, confirm):
    """Appends one line to a marker file per file it takes (the file's name and this worker's device and pid): a file
    handled twice leaves two lines."""
    out = Path(job["out"])
    while (f := take()) is not None:
        if job.get("log"):
            logging.info(f"marker for {Path(f).name}")
        with open(out / (Path(f).name + ".done"), "a") as m:
            m.write(f"{Path(f).name} {device} {os.getpid()}\n")
        confirm(f, ("marker", device))


def copy_body(device, job, take, confirm):
    """Copies every file it takes into ``job["out"]`` (paths as the caller gave them, relative ones too) and confirms with
    its working directory and one environment variable."""
    while (f := take()) is not None:
        Path(job["out"], Path(f).name).write_bytes(Path(f).read_bytes())
        confirm(f, (os.getcwd(), os.environ.get("P2P_FOLDER_POOL_TEST")))


def exit_body(device, job, take, confirm):
    """The worker of device 1 takes one file and ends with exit code 3; the others wait until it has, then behave like
    ``marker_body``."""
    flag = Path(job["out"]) / "taken"
    if device == 1:
        flag.write_text(str(Path(take()).name))
        os._exit(3)
    end = time.monotonic() + 60
    while not flag.exists() and time.monotonic() < end:
        time.sleep(0.01)
    marker_body(device, job, take, confirm)


def raise_body(device, job, take, confirm):
    if device == 1:
        raise ValueError("no such device in this test")
    marker_body(device, job, take, confirm)


@pytest.fixture
def folder_pool(pkg):
    return pkg.folder_pool


def _alive(pid):
    """True while ``pid`` runs (a zombie has ended: it only waits to be reaped)."""
    try:
        stat = Path(f"/proc/{pid}/stat").read_text()
    except OSError:
        return False
    return stat.rsplit(")", 1)[1].split()[0] != "Z"


def _wait_gone(pids, seconds=10.0):
    end = time.monotonic() + seconds
    while time.monotonic() < end and any(_alive(p) for p in pids):
        time.sleep(0.05)
    return [p for p in pids if _alive(p)]


def _files(tmp_path, n):
    src = tmp_path / "in"
    src.mkdir()
    for i in range(n):
        (src / f"f{i:03d}.jpg").write_bytes(b"")
    return sorted(src.iterdir())


def test_every_file_once_for_1_2_4_workers(folder_pool, tmp_path):
    files = _files(tmp_path, 37)
    results = []
    for n in (1, 2, 4):
        out = tmp_path / f"out{n}"
        out.mkdir()
        pool = folder_pool.FolderPool(list(range(n)), marker_body)
        try:
            pids = pool.pids
            assert len(set(pids)) == n
            done = pool.run({"out": str(out)}, files)
            (tmp_path / f"again{n}").mkdir()
            again = pool.run({"out": str(tmp_path / f"again{n}")}, files[:5])     # a second call: the same processes
            assert pool.pids == pids and sorted(again) == files[:5]
        finally:
            pool.close()
        assert sorted(done) == files and all(info[0] == "marker" and 0 <= info[1] < n for info in done.values())
        names = sorted(p.name for p in out.iterdir())
        assert names == sorted(f.name + ".done" for f in files)
        for p in out.iterdir():
            lines = p.read_text().splitlines()
            assert len(lines) == 1, (p.name, lines)         # handled exactly once
            name, dev, pid = lines[0].split()
            assert name + ".done" == p.name and int(pid) in pids and done[files[0].parent / name] == ("marker", int(dev))
        results.append({f.name: (out / (f.name + ".done")).exists() for f in files})
        assert _wait_gone(pids) == []
    assert results[0] == results[1] == results[2]


def test_worker_that_exits_is_reported_and_not_retried(folder_pool, tmp_path, caplog):
    files = _files(tmp_path, 12)
    out = tmp_path / "out"
    out.mkdir()
    pool = folder_pool.FolderPool([0, 1], exit_body)
    pids = pool.pids
    with caplog.at_level(logging.ERROR), pytest.raises(folder_pool.WorkerExited) as e:
        pool.run({"out": str(out)}, files)
    assert "exited with code 3" in str(e.value)
    lost = [r.message for r in caplog.records if r.message.startswith("Error processing ")]
    assert len(lost) == 1 and "exited with code 3" in lost[0]
    name = (out / "taken").read_text()
    assert lost[0].startswith(f"Error processing {files[0].parent / name}:")
    # every other file was handled by the worker that stayed, the lost one by nobody
    assert sorted(p.name for p in out.iterdir() if p.name != "taken") == sorted(f.name + ".done" for f in files if f.name != name)
    assert pool.closed and _wait_gone(pids) == []


def test_exception_in_body_is_raised_in_caller(folder_pool, tmp_path):
    files = _files(tmp_path, 6)
    out = tmp_path / "out"
    out.mkdir()
    pool = folder_pool.FolderPool([0, 1], raise_body)
    pids = pool.pids
    with pytest.raises(ValueError, match="no such device in this test") as e:
        pool.run({"out": str(out)}, files)
    assert any("folder worker process" in n for n in getattr(e.value, "__notes__", []))
    assert len(list(out.iterdir())) == len(files)       # the other worker handled every file
    assert pool.closed and _wait_gone(pids) == []


def test_workers_follow_the_callers_directory_and_environment(folder_pool, tmp_path, monkeypatch):
    """Relative input and output paths of a call, and the environment, are the caller's at the time of the call, also
    when it changed directory or environment after the pool's processes started."""
    for d in ("A", "B"):
        (tmp_path / d / "in").mkdir(parents=True)
        (tmp_path / d / "out").mkdir()
        for i in range(5):
            (tmp_path / d / "in" / f"f{i}.jpg").write_text(f"{d}{i}")
    files = [Path("in") / f"f{i}.jpg" for i in range(5)]
    monkeypatch.chdir(tmp_path / "A")
    monkeypatch.setenv("P2P_FOLDER_POOL_TEST", "a")
    pool = folder_pool.FolderPool([0, 0], copy_body)
    try:
        got_a = pool.run({"out": "out"}, files)
        monkeypatch.chdir(tmp_path / "B")
        monkeypatch.setenv("P2P_FOLDER_POOL_TEST", "b")
        got_b = pool.run({"out": "out"}, files)
        monkeypatch.delenv("P2P_FOLDER_POOL_TEST")
        got_c = pool.run({"out": "out"}, files[:1])
    finally:
        pool.close()
    assert got_a == {f: (str(tmp_path / "A"), "a") for f in files}
    assert got_b == {f: (str(tmp_path / "B"), "b") for f in files}
    assert got_c == {files[0]: (str(tmp_path / "B"), None)}
    for d in ("A", "B"):
        assert {p.name: p.read_text() for p in (tmp_path / d / "out").iterdir()} == {f"f{i}.jpg": f"{d}{i}" for i in range(5)}


def test_worker_log_records_reach_the_parent_handlers(folder_pool, tmp_path, caplog):
    files = _files(tmp_path, 4)
    out = tmp_path / "out"
    out.mkdir()
    pool = folder_pool.FolderPool([0, 0], marker_body)
    try:
        with caplog.at_level(logging.INFO):
            pool.run({"out": str(out), "log": True}, files)
    finally:
        pool.close()
    assert sorted(r.message for r in caplog.records if r.message.startswith("marker for")) == \
        sorted(f"marker for {f.name}" for f in files)


def test_shared_pool_is_kept_per_device_list(folder_pool):
    try:
        a = folder_pool.shared([0, 0], marker_body)
        assert folder_pool.shared([0, 0], marker_body) is a
        pids = a.pids
        b = folder_pool.shared([0, 1], marker_body)
        assert b is not a and a.closed and _wait_gone(pids) == []
        pids = b.pids
    finally:
        folder_pool.close_shared()
    assert _wait_gone(pids) == []


def test_shared_calls_from_threads_run_one_after_the_other(folder_pool, tmp_path):
    """Two threads calling the kept pool with different device lists: the second call waits for the first instead of
    replacing the pool under it; both handle all their files."""
    import threading

    files = _files(tmp_path, 40)
    outs = [tmp_path / "o0", tmp_path / "o1"]
    errors, done = [], {}

    def call(k, devices):
        try:
            outs[k].mkdir()
            done[k] = folder_pool.run_shared(devices, marker_body, {"out": str(outs[k])}, files)
        except BaseException as e:   # noqa: BLE001
            errors.append(e)

    try:
        threads = [threading.Thread(target=call, args=(k, devs)) for k, devs in enumerate(([0, 0], [0, 1, 2]))]
        for t in threads:
            t.start()
        for t in threads:
            t.join(120)
        assert errors == [] and sorted(done[0]) == sorted(done[1]) == files
        for out in outs:
            assert sorted(p.name for p in out.iterdir()) == sorted(f.name + ".done" for f in files)
    finally:
        folder_pool.close_shared()


def test_no_worker_outlives_a_killed_parent(pkg, tmp_path):
    """A parent that is killed (no atexit, no close) leaves no worker behind: the workers read end-of-file and leave."""
    root = Path(__file__).resolve().parent.parent
    script = textwrap.dedent(f"""
        import sys, time
        sys.path[:0] = [{str(root)!r}, {str(Path(__file__).parent)!r}]
        if __name__ == "__main__":
            import __graft_entry__ as g
            from test_folder_pool import marker_body
            pool = g.load_package().folder_pool.FolderPool([0, 0, 0], marker_body)
            print(" ".join(map(str, pool.pids)), flush=True)
            time.sleep(300)
    """)
    path = tmp_path / "parent.py"
    path.write_text(script)
    proc = subprocess.Popen([sys.executable, str(path)], stdout=subprocess.PIPE, text=True)
    try:
        pids = [int(p) for p in proc.stdout.readline().split()]
        assert len(pids) == 3 and all(_alive(p) for p in pids)
    finally:
        proc.send_signal(signal.SIGKILL)
        proc.wait()
    assert _wait_gone(pids) == []
