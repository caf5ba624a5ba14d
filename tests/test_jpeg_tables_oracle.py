"""Huffman tables and file layouts cv2 does not write by default (tests/jpeg_writer.py), on the CPU: the writer against
cv2's own bytes, the oracle and the library's host stage against cv2.imdecode, and the exact tables the device Huffman
stage receives (``p2p_jpeg_device_tables``) decoded code by code the way its kernels read them."""
import ctypes as C

import cv2
import numpy as np
import pytest

import jpeg_writer as jw
from oracle import jpeg_decode_model as jd
from oracle import synth

SAMPLING = {"420": cv2.IMWRITE_JPEG_SAMPLING_FACTOR_420, "422": cv2.IMWRITE_JPEG_SAMPLING_FACTOR_422,
            "444": cv2.IMWRITE_JPEG_SAMPLING_FACTOR_444}


def _image(kind, w, h, seed):
    if kind == "noise":
        return synth.noise(w, h, seed)
    if kind == "sat":
        return (np.random.default_rng(seed).integers(0, 2, (h, w, 3)) * 255).astype(np.uint8)
    return synth.smooth(w, h, seed)


def writer_cases():
    for (w, h) in [(1, 1), (2, 3), (17, 33), (67, 45), (120, 90)]:
        for sname in ("420", "422", "444", "gray"):
            for rst in (0, 1, 7):
                kind = ("noise", "smooth", "sat")[(w + rst) % 3]
                yield f"{w}x{h}_{sname}_rst{rst}_{kind}", w, h, sname, rst, kind


@pytest.mark.parametrize("name,w,h,sname,rst,kind", list(writer_cases()), ids=[c[0] for c in writer_cases()])
def test_writer_reproduces_cv2_bytes(name, w, h, sname, rst, kind):
    """Annex K tables give exactly cv2.imencode's default file, optimal tables exactly its IMWRITE_JPEG_OPTIMIZE file
    (the two files of one image carry the same coefficients)."""
    img = _image(kind, w, h, w * 31 + h)
    if sname == "gray":
        img = np.ascontiguousarray(img[..., 1])
    params = [cv2.IMWRITE_JPEG_QUALITY, 90, cv2.IMWRITE_JPEG_RST_INTERVAL, rst]
    if sname != "gray":
        params += [cv2.IMWRITE_JPEG_SAMPLING_FACTOR, SAMPLING[sname]]
    default = cv2.imencode(".jpg", img, params)[1].tobytes()
    optimised = cv2.imencode(".jpg", img, params + [cv2.IMWRITE_JPEG_OPTIMIZE, 1])[1].tobytes()
    source = jw.read_coefficients(default)
    assert jw.write(default, source=source) == default
    assert jw.write(default, tables="optimal", source=source) == optimised
    assert jw.write(optimised, tables="annex_k") == default


def table_corpus():
    """(label, file): cv2 OPTIMIZE files, luma / chroma qualities that differ, and every jpeg_writer policy and layout on
    smooth and noise content"""
    for k, (w, h) in enumerate([(1, 1), (17, 33), (67, 45)]):
        for sname in ("420", "422", "444", "gray"):
            q, rst, kind = ((20, 0, "smooth"), (75, 7, "noise"), (95, 1, "sat"), (100, 0, "noise"))[(k + len(sname)) % 4]
            img = _image(kind, w, h, k)
            params = [cv2.IMWRITE_JPEG_QUALITY, q, cv2.IMWRITE_JPEG_RST_INTERVAL, rst, cv2.IMWRITE_JPEG_OPTIMIZE, 1]
            if sname == "gray":
                img = np.ascontiguousarray(img[..., 0])
            else:
                params += [cv2.IMWRITE_JPEG_SAMPLING_FACTOR, SAMPLING[sname]]
            yield f"optimize {w}x{h} {sname} q{q} rst{rst} {kind}", cv2.imencode(".jpg", img, params)[1].tobytes()
    img = synth.smooth(67, 45, 4)
    for lq, cq in ((95, 30), (20, 100)):
        yield f"luma q{lq} chroma q{cq}", cv2.imencode(".jpg", img, [cv2.IMWRITE_JPEG_LUMA_QUALITY, lq,
                                                                     cv2.IMWRITE_JPEG_CHROMA_QUALITY, cq])[1].tobytes()
    for kind, (w, h) in (("smooth", (67, 45)), ("noise", (40, 24))):
        img = _image(kind, w, h, 3)
        for sname, src in (("420", img), ("444", img), ("gray", np.ascontiguousarray(img[..., 2]))):
            params = [cv2.IMWRITE_JPEG_QUALITY, 93]
            if sname != "gray":
                params += [cv2.IMWRITE_JPEG_SAMPLING_FACTOR, SAMPLING[sname]]
            data = cv2.imencode(".jpg", src, params)[1].tobytes()
            source = jw.read_coefficients(data)
            for label, kw in jw.variants(1 if sname == "gray" else 3):
                yield f"{kind} {sname} {label}", jw.write(data, source=source, **kw)


CORPUS = list(table_corpus())


def _host_stage(lib, data):
    lay = (C.c_int32 * 10)()
    if lib.p2p_jpeg_coefficients(data, len(data), None, 0, lay):
        return None
    shapes = [(lay[5 + 2 * k], lay[4 + 2 * k], 64) for k in range(3)]
    coef = np.zeros(sum(a * b * c for a, b, c in shapes), np.int16)
    if lib.p2p_jpeg_coefficients(data, len(data), coef.ctypes.data, coef.size, lay):
        return None
    planes, off = [], 0
    for sh in shapes:
        n = sh[0] * sh[1] * 64
        planes.append(coef[off:off + n].astype(np.int64).reshape(sh))
        off += n
    return planes


@pytest.mark.parametrize("label,data", CORPUS, ids=[c[0] for c in CORPUS])
def test_oracle_and_host_stage_equal_cv2(pkg, label, data):
    ref = cv2.imdecode(np.frombuffer(data, np.uint8), cv2.IMREAD_COLOR)
    assert ref is not None
    assert np.array_equal(jd.decode(data), ref)
    p = jd.parse(data)
    want, _ = jd.entropy_decode(p)
    got = _host_stage(pkg._lib.load(), data)
    assert got is not None, "the host stage declined"
    for a, b in zip(got, want):
        assert np.array_equal(a, b)
    assert np.array_equal(jd.reconstruct(p, got[:len(want)]), ref)


# ---- the tables the device receives ----------------------------------------------------------------------------------
def device_tables(lib, data):
    """(DevHuff fields per component, SyncLut e / w, masks) as p2p_jpeg_device_tables exports them"""
    lay = (C.c_int32 * 16)()
    assert lib.p2p_jpeg_device_tables(data, len(data), None, 0, lay) == 0
    size, huff = lay[0], lay[1]
    buf = np.zeros(size, np.uint8)
    assert lib.p2p_jpeg_device_tables(data, len(data), buf.ctypes.data, size - 1, lay) == -1   # capacity checked
    assert lib.p2p_jpeg_device_tables(data, len(data), buf.ctypes.data, size, lay) == 0
    fast = 1 << lay[15]
    n_dc, n_ac = lay[11], lay[12]

    def arr(c, off, dtype, n):
        o = c * huff + off
        return buf[o:o + n * np.dtype(dtype).itemsize].view(dtype)

    comps = []
    for c in range(3):
        comps.append(dict(
            dc=dict(look=arr(c, lay[2], np.uint16, 512), maxcode=arr(c, lay[3], np.int32, 18), valoff=arr(c, lay[4], np.int32, 18),
                    vals=arr(c, lay[5], np.uint8, n_dc), mask=n_dc - 1),
            ac=dict(fast=arr(c, lay[6], np.int32, fast), look=arr(c, lay[7], np.uint16, 512), maxcode=arr(c, lay[8], np.int32, 18),
                    valoff=arr(c, lay[9], np.int32, 18), vals=arr(c, lay[10], np.uint8, n_ac), mask=n_ac - 1)))
    L = lay[13]
    e = buf[L:L + 3 * 2 * fast * 2].view(np.uint16).reshape(3, 2, fast)
    w = buf[L + lay[14]:L + lay[14] + 3 * 2 * fast * 4].view(np.uint32).reshape(3, 2, fast)
    return comps, e, w, lay[15]


def dht_codes(bits, vals):
    """plain decode of a DHT: [(length, code, symbol)] - a value listed twice decodes from each of its codes"""
    out, code, k = [], 0, 0
    for ln in range(1, 17):
        for _ in range(bits[ln - 1]):
            out.append((ln, code, vals[k]))
            code += 1
            k += 1
        code <<= 1
    return out


def kernel_symbol(t, win):
    """huff_decode_range / huff_sync_fast_kernel / huff_write_fast_kernel: 9-bit look-up, then slow_symbol over
    maxcode / valoff / vals (index masked like the kernels); -> (symbol, length)"""
    e = int(t["look"][win >> 23])
    if e:
        return e & 0xFF, e >> 8
    w16 = win >> 16
    for ln in range(10, 17):
        code = w16 >> (16 - ln)
        if code <= int(t["maxcode"][ln]):
            return int(t["vals"][(code + int(t["valoff"][ln])) & t["mask"]]), ln
    return -1, 16


def extend(v, s):
    return v - (1 << s) + 1 if v < (1 << (s - 1)) else v


def check_device_tables(lib, data):
    p = jd.parse(data)
    comps, E, Wt, fb = device_tables(lib, data)
    scan = p["scan"] * 3 if len(p["scan"]) == 1 else p["scan"]
    for c, (_, td, ta) in enumerate(scan):
        for cls, tid in ((0, td), (1, ta)):
            bits, vals = p["huff"][(cls << 4) | tid]
            t = comps[c]["ac" if cls else "dc"]
            codes = dht_codes(bits, vals)
            for ln, code, sym in codes:
                # every code, with value bits 0..0 and 1..1 behind it: the symbol and the length the kernels decode
                for tail in (0, (1 << (32 - ln)) - 1):
                    win = (code << (32 - ln)) | tail
                    assert kernel_symbol(t, win) == (sym, ln), (c, cls, ln, code, sym)
            # every 10-bit window: 9-bit look-up, combined AC look-up, the synchronisation / write-pass look-ups
            prefix = {}
            for ln, code, sym in codes:
                if ln <= fb:
                    for i in range(code << (fb - ln), (code + 1) << (fb - ln)):
                        prefix[i] = (ln, sym)
            for i in range(1 << fb):
                ln, sym = prefix.get(i, (0, -1))
                if i % 2 == 0:
                    want = (ln << 8) | sym if 0 < ln <= 9 else 0
                    assert int(t["look"][i >> 1]) == want, (c, cls, i)
                if sym < 0:
                    assert E[c, cls, i] == 0 and Wt[c, cls, i] == 0, (c, cls, i)
                    if cls:
                        assert t["fast"][i] == 0
                    continue
                if cls == 0:
                    s, adv = min(sym, 15), 1
                else:
                    r, s = sym >> 4, sym & 15
                    adv = r + 1 if s else (16 if r == 15 else 64)
                    if s and ln + s <= fb:
                        v = (i >> (fb - ln - s)) & ((1 << s) - 1)
                        want = ((extend(v, s) & 0xFFFFFF) << 8) | (r << 4) | (ln + s)
                        assert int(t["fast"][i]) & 0xFFFFFFFF == want, (c, i, sym)
                    else:
                        assert t["fast"][i] == 0, (c, i, sym)
                assert E[c, cls, i] == (ln + s) | (adv << 5), (c, cls, i, ln, sym)
                assert Wt[c, cls, i] == ln | (s << 5) | (adv << 9), (c, cls, i, ln, sym)
        # the all-ones prefix is no code: the kernels report it (16 bits consumed)
        assert kernel_symbol(comps[c]["ac"], 0xFFFFFFFF)[0] == -1 and kernel_symbol(comps[c]["dc"], 0xFFFFFFFF)[0] == -1


@pytest.mark.parametrize("label,data", CORPUS, ids=[c[0] for c in CORPUS])
def test_device_tables_decode_every_code(pkg, label, data):
    """The exact bytes the device Huffman stage uploads, read the way its kernels read them: every code of every table in
    use gives the DHT's symbol and length; every 10-bit window of the look-ups gives the code + value bits consumed and the
    zigzag advance of a plain decode of the DHT."""
    check_device_tables(pkg._lib.load(), data)


def test_device_tables_cover_the_table_edges(pkg):
    """The corpus reaches the boundaries the look-up paths switch on: 9 against 10 bits, length + size of 10 against 11,
    16-bit codes, DC codes of 10 bits or more at symbol index 16 or higher."""
    seen = set()
    for label, data in CORPUS:
        p = jd.parse(data)
        for (tc_th, (bits, vals)) in p["huff"].items():
            for ln, code, sym in dht_codes(bits, vals):
                seen.add(("len", ln))
                if tc_th >> 4 and sym & 15:
                    seen.add(("len+size", ln + (sym & 15)))
            if not tc_th >> 4 and len(vals) > 16 and bits[9]:
                seen.add("dc index >= 16")
    for want in [("len", 9), ("len", 10), ("len", 16), ("len+size", 10), ("len+size", 11), "dc index >= 16"]:
        assert want in seen, want
    lay = (C.c_int32 * 16)()
    prog = cv2.imencode(".jpg", synth.smooth(64, 48, 1), [cv2.IMWRITE_JPEG_PROGRESSIVE, 1])[1].tobytes()
    assert pkg._lib.load().p2p_jpeg_device_tables(prog, len(prog), None, 0, lay) == -6   # no device stage for these
