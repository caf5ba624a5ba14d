"""The device JPEG encoder (csrc/p2p_jpeg.cuh) on the images of tests/jpeg_symbols.py, which reach every DC category and
AC symbol of both Huffman tables, ZRL chains, coefficients at zig-zag 63, padding that completes an 0xFF and blocks at
every bit of an emit word (tests/test_jpeg_symbols_oracle.py shows that on the CPU).  Every file must be the bytes
cv2.imencode('.jpg') writes at the same quality: one image per call, same-size batches, images read from device memory
at every byte alignment, every quality from four threads while the table cache is rebuilt, and a batch in which one
file does not fit its output buffer."""
import ctypes as C
import threading

import numpy as np
import pytest

import jpeg_symbols as js

pytestmark = pytest.mark.gpu

CORPUS = js.corpus()
BY_NAME = {c[0]: c for c in CORPUS}
P2P_ERR_LIMIT = -5


@pytest.fixture(scope="module")
def jctx(pkg):
    """A context of this module's own, with 4 slots: the quality sweep below counts on starting from an empty table
    cache and on owning every slot."""
    p = pkg.Projector(0, n_slots=4)
    yield p
    p.close()


def encode_raw(ctx, slot, ptr, on_device, n, W, H, quality, stride):
    """p2p_encode_jpeg through the C ABI: (return code, sizes, files as bytes or None for size 0)"""
    out = np.zeros((n, stride), np.uint8)
    sizes = (C.c_size_t * n)()
    rc = ctx.lib.p2p_encode_jpeg(ctx.ctx, slot, ptr, on_device, n, W, H, quality, out.ctypes.data, stride, sizes)
    return rc, list(sizes), [out[i, :sizes[i]].tobytes() if sizes[i] else None for i in range(n)]


@pytest.mark.parametrize("name", list(BY_NAME))
def test_symbol_image_equals_cv2(jctx, name):
    _, img, quality = BY_NAME[name]
    assert jctx.encode_jpeg(img, quality)[0] == js.cv2_jpeg(img, quality), name


def _batch():
    """every 128 x 128 image of the corpus (flat and saturated ones included), at least 12"""
    imgs = [(n, img) for n, img, _ in CORPUS if img.shape[:2] == (js.SIZE, js.SIZE)]
    assert len(imgs) >= 12 and {"flat-gray", "saturated-noise"} <= {n for n, _ in imgs}
    return [n for n, _ in imgs], np.stack([img for _, img in imgs])


@pytest.mark.parametrize("quality", [50, 90, 100])
def test_batch_of_one_size_equals_cv2(jctx, quality):
    names, imgs = _batch()
    files = jctx.encode_jpeg(imgs, quality)
    for name, f, img in zip(names, files, imgs):
        assert f == js.cv2_jpeg(img, quality), name


@pytest.mark.parametrize("offset", [0, 1, 2, 3])
def test_device_input_at_every_alignment(jctx, offset):
    """Device pointers with on_device = 1 at byte offsets 0 .. 3: 128-pixel rows (W * 3 % 4 == 0) take the word loads of
    jpeg_dct_kernel's staging only when the pointer is 4-byte aligned, odd widths never."""
    import torch

    names, imgs = _batch()
    groups = [(names, imgs, 100)]
    groups += [([n], img[None], q) for n, img, q in CORPUS if img.shape[1] * 3 % 4 != 0]
    assert len(groups) >= 3
    for gnames, g, quality in groups:
        n, H, W, _ = g.shape
        buf = torch.zeros(offset + g.nbytes, dtype=torch.uint8, device="cuda:0")
        buf[offset:] = torch.from_numpy(np.ascontiguousarray(g).reshape(-1)).to("cuda:0")
        torch.cuda.synchronize()        # the encoder runs on its slot's own stream
        rc, _, files = encode_raw(jctx, 0, buf.data_ptr() + offset, 1, n, W, H, quality, W * H * 3 + 4096)
        assert rc == 0, jctx.lib.p2p_last_error(jctx.ctx).decode()
        for name, f, img in zip(gnames, files, g):
            assert f == js.cv2_jpeg(img, quality), (name, offset)


def test_every_quality_from_four_threads(jctx):
    """Qualities 0 .. 100 and -1, 101, 1000 (clamped to 1 .. 100 by build_tables as by cv2) on two images of different
    sizes, from 4 threads on the 4 slots of one context: 208 (size, quality) entries, so the table cache passes its 64
    entries and is rebuilt three times while the other slots have work in flight."""
    imgs = [BY_NAME["ac0-q100-0"][1], BY_NAME["dc-edge3-44x52"][1]]
    jobs = [(i, q) for q in list(range(101)) + [-1, 101, 1000] for i in range(2)]
    got, errors = {}, []

    def work(slot):
        try:
            for i, q in jobs[slot::4]:
                got[(i, q)] = jctx.encode_jpeg(imgs[i], q, slot=slot)[0]
        except Exception as e:   # reported below: an exception in a thread would otherwise pass silently
            errors.append(repr(e))

    threads = [threading.Thread(target=work, args=(s,)) for s in range(4)]
    for t in threads:
        t.start()
    for t in threads:
        t.join()
    assert not errors, errors
    wrong = [(i, q) for (i, q) in jobs if got.get((i, q)) != js.cv2_jpeg(imgs[i], q)]
    assert not wrong, wrong


def test_batch_with_one_file_too_large(jctx):
    """One file of the batch does not fit out_stride: P2P_ERR_LIMIT, size 0 for that file, and every other file still
    arrives, identical to cv2's."""
    names = ["flat-gray", "saturated-noise", "ac0-q100-0", "dc0-q100", "ac1-q100-0"]
    imgs = np.stack([BY_NAME[n][1] for n in names])
    refs = [js.cv2_jpeg(img, 100) for img in imgs]
    stride = max(len(r) for n, r in zip(names, refs) if n != "saturated-noise")
    assert len(refs[1]) > stride
    rc, sizes, files = encode_raw(jctx, 1, imgs.ctypes.data, 0, len(imgs), js.SIZE, js.SIZE, 100, stride)
    assert rc == P2P_ERR_LIMIT
    assert sizes[1] == 0 and files[1] is None
    for i, name in enumerate(names):
        if i != 1:
            assert files[i] == refs[i], name
    # the context stays usable, and the same batch with room for every file succeeds
    rc, _, files = encode_raw(jctx, 1, imgs.ctypes.data, 0, len(imgs), js.SIZE, js.SIZE, 100, js.SIZE * js.SIZE * 3 + 4096)
    assert rc == 0 and files == refs
