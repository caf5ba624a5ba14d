"""Worker processes for the directory front end: one per listed device, fed one file at a time from the caller's queue.

One Python process drives a folder at about 1.3 ms of host time per image (reading files, destuffing, creating the output
files under the GIL), so a folder over several GPUs is only faster with a process per GPU (DESIGN §6).  ``FolderPool``
starts those processes with the ``spawn`` method (never ``fork``: the caller may hold a CUDA context) and keeps them for
later calls, so a long-lived caller pays CUDA context creation once per worker.

The parent never touches a device.  Per call it sends every worker ``(device, job)`` with the caller's working directory
and environment variables, which the worker takes over for the call (relative paths and settings read from the
environment mean what they mean in the caller); a worker's threads ask for files
(``take``), the parent hands out the next one from its queue and records which worker took it, the worker confirms each
file once its outputs are written (``confirm``).  Log records of the workers are emitted by the parent's own handlers.
A worker blocks reading its control pipe and leaves on end-of-file, so no worker outlives its parent.

As with any spawn-started process, a script that runs a pool needs the ``if __name__ == "__main__":`` guard: a worker
imports the caller's main script as ``__mp_main__`` when it starts.  Calls of the kept pool (``run_shared``) run one at
a time.
"""
from __future__ import annotations

import atexit
import collections
import copy
import importlib.util
import logging
import multiprocessing
import os
import pickle
import queue
import runpy
import sys
import threading
import traceback
from multiprocessing import connection

_WORKER_RUN_NAME = "__p2p_folder_worker__"   # the name this file runs under in a worker (see the end of the file)


class WorkerExited(RuntimeError):
    """A worker process ended in the middle of a call; the files it had taken and not confirmed were not processed."""


class _Worker:
    __slots__ = ("device", "proc", "conn", "taken")

    def __init__(self, device, proc, conn):
        self.device, self.proc, self.conn, self.taken = device, proc, conn, []


class FolderPool:
    """One worker process per entry of ``devices`` (an entry may repeat: two processes on one GPU).

    ``body(device, job, take, confirm)`` runs in each worker for every ``run``: ``take()`` returns the next file or None
    when the queue is empty, ``confirm(file, info)`` reports a file as done.  ``body`` is pickled by reference and resolved
    in the worker after the package is loaded there under the parent's package name."""

    def __init__(self, devices, body):
        self.devices = [int(d) for d in devices]
        self.body = body
        self._lock = threading.RLock()
        self._workers = []
        ctx = multiprocessing.get_context("spawn")
        package = __name__.rpartition(".")[0]
        package_dir = os.path.dirname(os.path.abspath(__file__))
        try:
            for d in self.devices:
                ours, theirs = ctx.Pipe()
                # runpy.run_path is importable in a fresh interpreter; the package may not be (its directory name is not
                # an identifier, and it may be loaded under another name): the worker runs this file by its path
                proc = ctx.Process(target=runpy.run_path, args=(os.path.abspath(__file__),),
                                   kwargs={"run_name": _WORKER_RUN_NAME,
                                           "init_globals": {"_WORKER_ARGS": (package, package_dir, theirs)}},
                                   name=f"p2p-folder-worker-{d}", daemon=True)
                proc.start()
                theirs.close()
                self._workers.append(_Worker(d, proc, ours))
                ours.send(body)
        except BaseException:
            self.close()
            raise

    @property
    def pids(self) -> list:
        return [w.proc.pid for w in self._workers]

    @property
    def closed(self) -> bool:
        return not self._workers

    @property
    def ready(self) -> bool:
        """Open, and every worker process alive."""
        return bool(self._workers) and all(w.proc.is_alive() for w in self._workers)

    def run(self, job, files) -> dict:
        """Process ``files`` with every worker and return {file: info} of the confirmed files.  Files are handed out one at
        a time to whichever worker asks first, each file exactly once.  Raises, once every worker has stopped, the first
        exception that escaped a worker's ``body``, or ``WorkerExited`` if a worker process ended; the pool is closed
        then.  A file a worker had taken when it ended is logged as ``Error processing <file>`` and not given to
        another worker."""
        with self._lock:
            if self.closed:
                raise RuntimeError("the folder pool is closed")
            try:
                return self._run(job, files)
            except BaseException:
                self.close()
                raise

    def _run(self, job, files):
        pending = collections.deque(files)
        level = logging.getLogger().getEffectiveLevel()
        where = (os.getcwd(), dict(os.environ))
        for w in self._workers:
            w.taken = []
            w.conn.send(("call", w.device, job, level, where))
        running = list(self._workers)
        done, errors = {}, []

        def handle(w, msg):
            kind = msg[0]
            if kind == "take":
                f = pending.popleft() if pending else None
                if f is not None:
                    w.taken.append(f)
                w.conn.send(("file", f))
            elif kind == "done":
                w.taken.remove(msg[1])
                done[msg[1]] = msg[2]
            elif kind == "log":
                record = msg[1]
                logging.getLogger(record.name).handle(record)
            else:   # "finished"
                running.remove(w)
                if msg[1] is not None:
                    errors.append(msg[1])

        def lost(w):
            try:                    # what it sent before it ended still counts
                while w in running and w.conn.poll():
                    handle(w, w.conn.recv())
            except (EOFError, OSError):
                pass
            if w not in running:
                return
            running.remove(w)
            w.proc.join()
            code = w.proc.exitcode
            for f in w.taken:
                logging.error(f"Error processing {f}: the worker process of device {w.device} exited with code {code}")
            errors.append(WorkerExited(f"the folder worker of device {w.device} (pid {w.proc.pid}) exited with code {code}; "
                                       f"{len(w.taken)} files it had taken were not processed"))

        while running:
            by_handle = {}
            for w in running:
                by_handle[w.conn] = by_handle[w.proc.sentinel] = w
            for r in connection.wait(list(by_handle)):
                w = by_handle[r]
                if w not in running:
                    continue
                if r is w.proc.sentinel:
                    lost(w)
                    continue
                try:
                    handle(w, w.conn.recv())
                except (EOFError, OSError):   # (a reply to a worker that has just ended)
                    lost(w)
        if errors:
            if pending:
                errors[0].add_note(f"{len(pending)} files were not handed to any worker")
            raise errors[0]
        return done

    def close(self, timeout: float = 10.0) -> None:
        """End every worker (end-of-file on its pipe; killed if it has not left after ``timeout`` seconds) and wait for it.
        Waits for a ``run`` in progress in another thread to end first."""
        with self._lock:
            workers, self._workers = self._workers, []
        for w in workers:
            w.conn.close()
        for w in workers:
            w.proc.join(timeout)
            if w.proc.is_alive():
                w.proc.kill()
                w.proc.join()


_shared: FolderPool | None = None
_shared_lock = threading.RLock()


def shared(devices, body) -> FolderPool:
    """The pool kept for later calls: reused while the device list and ``body`` stay the same, else replaced."""
    global _shared
    devices = [int(d) for d in devices]
    with _shared_lock:
        if _shared is not None and not (_shared.ready and _shared.devices == devices and _shared.body is body):
            _shared.close()
            _shared = None
        if _shared is None:
            _shared = FolderPool(devices, body)
        return _shared


def run_shared(devices, body, job, files) -> dict:
    """``run`` of the kept pool for ``devices`` and ``body``.  Calls from several threads run one after the other, so a
    call with another device list never replaces the pool under a call in progress."""
    with _shared_lock:
        return shared(devices, body).run(job, files)


def close_shared() -> None:
    """Close the kept pool, if there is one."""
    global _shared
    with _shared_lock:
        if _shared is not None:
            _shared.close()
            _shared = None


def _close_shared_at_exit():
    # a call still running in a daemon thread keeps the lock: its workers then leave on end-of-file when this process ends
    if _shared_lock.acquire(blocking=False):
        try:
            close_shared()
        finally:
            _shared_lock.release()


atexit.register(_close_shared_at_exit)


# ----------------------------------------------------------------------------------------------------------------------
# the worker side
# ----------------------------------------------------------------------------------------------------------------------
class _ForwardHandler(logging.Handler):
    """Sends every record to the parent with its message already formatted (arguments may not pickle)."""

    def __init__(self, send):
        super().__init__()
        self._send = send

    def emit(self, record):
        try:
            r = copy.copy(record)
            r.msg, r.args = record.getMessage(), None
            if record.exc_info:
                r.exc_text = logging.Formatter().formatException(record.exc_info)
            r.exc_info = None
            self._send(("log", r))
        except Exception:   # noqa: BLE001
            self.handleError(record)


def _portable(e: BaseException) -> BaseException:
    """``e`` with the worker's traceback as a note, or a RuntimeError with its text if ``e`` does not pickle."""
    tb = "".join(traceback.format_exception(e))
    try:
        e.add_note(f"in a folder worker process (pid {os.getpid()}):\n{tb}")
        pickle.loads(pickle.dumps(e))
        return e
    except Exception:   # noqa: BLE001
        return RuntimeError(f"in a folder worker process (pid {os.getpid()}):\n{tb}")


def _run_call(body, device, job, where, files, send):
    def take():
        send(("take",))
        return files.get()

    def confirm(f, info=None):
        send(("done", f, info))

    err = None
    try:
        cwd, env = where      # the caller's: its relative paths and environment settings mean the same here
        os.chdir(cwd)
        if env != os.environ:
            os.environ.clear()
            os.environ.update(env)
        body(device, job, take, confirm)
    except BaseException as e:   # noqa: BLE001 - raised in the caller
        err = _portable(e)
    send(("finished", err))


def _serve(conn):
    lock = threading.Lock()

    def send(msg):
        with lock:
            conn.send(msg)

    root = logging.getLogger()
    for h in list(root.handlers):
        root.removeHandler(h)
    root.addHandler(_ForwardHandler(send))
    files = queue.SimpleQueue()
    call = None
    try:
        body = conn.recv()
        while True:
            msg = conn.recv()
            if msg[0] == "file":
                files.put(msg[1])
            else:   # ("call", device, job, level, (cwd, environment))
                _, device, job, level, where = msg
                root.setLevel(level)
                call = threading.Thread(target=_run_call, args=(body, device, job, where, files, send), daemon=True)
                call.start()
    except EOFError:    # the parent closed the pool, or is gone
        if call is not None and call.is_alive():
            os._exit(1)


def _worker_main(package, package_dir, conn):
    """Load the package under the parent's name (as ``__graft_entry__.load_package`` does), then serve the pipe."""
    if package not in sys.modules:
        spec = importlib.util.spec_from_file_location(package, os.path.join(package_dir, "__init__.py"),
                                                      submodule_search_locations=[package_dir])
        mod = importlib.util.module_from_spec(spec)
        sys.modules[package] = mod
        spec.loader.exec_module(mod)
    _serve(conn)


if __name__ == _WORKER_RUN_NAME:
    _worker_main(*_WORKER_ARGS)  # noqa: F821 - given by FolderPool through runpy's init_globals
