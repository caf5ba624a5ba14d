"""Test-only JPEG writer: re-encodes the quantised coefficients of a baseline file with any legal Huffman tables, table
ids, restart interval and segment layout - the files the decoder meets in the wild (optimised tables from stitchers,
``cjpeg -optimize``, PIL ``optimize=True``, progressive-era libjpeg-turbo) and edge cases no encoder writes by default.

The coefficients come from ``oracle.jpeg_decode_model`` (or, for large files, from the library's host stage, which the
CPU tests pin against the oracle), so a re-encoded file holds exactly the coefficients of its source and cv2 decodes both
to the same pixels.  The entropy coder is jchuff.c's (DC differences per component, reset at restart markers; runs of
zeros as ZRL + (run, size) symbols, EOB; value bits as HUFF_EXTEND expects; 1-bit padding; 0xFF stuffing), vectorised
with NumPy so that panoramas are re-encoded in seconds.  With ``tables="annex_k"`` the output is byte for byte the file
``cv2.imencode`` writes, with ``tables="optimal"`` the one ``cv2.imencode(..., [IMWRITE_JPEG_OPTIMIZE, 1])`` writes.

Table policies (``tables=`` one policy for every table, or a dict ``{("dc" | "ac", component): policy}``; a policy is a
name below or an explicit ``(bits, vals)``):
  annex_k        the Annex K tables (luma for table 0, chroma for the others), as cv2 writes them
  optimal        jchuff.c jpeg_gen_optimal_table over the symbol counts of the blocks that use the table
  all_len(n)     every used symbol gets an n-bit code
  fast_ac_edge   AC codes whose length + value size is exactly 10 or 11 (the decoder's 10-bit combined lookup edge);
                 DC optimal
  dc_dup         DC: 16 five-bit codes of category 0, then categories 0..11 as 10-bit codes at indices 16..27 (a table
                 with more than 16 entries; the symbols in use sit at index 16 or higher); AC optimal
  eob_alias      size-0 symbols 0x10 .. 0xE0 used as end of block (libjpeg ends the block for any run below 15);
                 tables optimal over those counts
"""
from __future__ import annotations

import ctypes as C
import re

import numpy as np

from oracle import jpeg_decode_model as jd
from oracle import jpeg_model as jm
from oracle.jpeg_model import ZIGZAG

LAYOUTS = ("dht_one_segment", "dqt_one_segment", "tables_after_sof", "dri_before_dqt", "extra_segments", "fill_bytes")


# ---- coefficients of a file ----------------------------------------------------------------------------------------
def read_coefficients(data: bytes, lib=None):
    """(header dict of ``jd.parse``, coefficient planes [by, bx, 64] natural order per component).  ``lib``: the loaded
    library - its host stage (``p2p_jpeg_coefficients``) instead of the bit-serial oracle, for large files."""
    p = jd.parse(data)
    ncomp = len(p["frame"]["comps"])
    if lib is None:
        planes, _ = jd.entropy_decode(p)
        return p, planes
    lay = (C.c_int32 * 10)()
    if lib.p2p_jpeg_coefficients(data, len(data), None, 0, lay) != 0:
        raise ValueError("the host stage declines the source file")
    shapes = [(lay[5 + 2 * k], lay[4 + 2 * k], 64) for k in range(3)]
    coef = np.zeros(sum(a * b * c for a, b, c in shapes), np.int16)
    if lib.p2p_jpeg_coefficients(data, len(data), coef.ctypes.data, coef.size, lay) != 0:
        raise ValueError("the host stage declines the source file")
    planes, off = [], 0
    for sh in shapes[:ncomp]:
        n = sh[0] * sh[1] * 64
        planes.append(coef[off:off + n].astype(np.int64).reshape(sh))
        off += n
    return p, planes


# ---- Huffman tables ------------------------------------------------------------------------------------------------
def gen_optimal_table(freq):
    """jchuff.c jpeg_gen_optimal_table: (bits[16], vals) for the symbol counts ``freq[0..255]`` (pseudo-symbol 256
    reserves the all-ones code; code lengths limited to 16 bits)."""
    freq = [int(f) for f in freq[:256]] + [1]
    codesize, others = [0] * 257, [-1] * 257
    while True:
        c1, v = -1, 1 << 62
        for i in range(257):          # smallest non-zero count; ties: the larger symbol
            if freq[i] and freq[i] <= v:
                v, c1 = freq[i], i
        c2, v = -1, 1 << 62
        for i in range(257):
            if freq[i] and freq[i] <= v and i != c1:
                v, c2 = freq[i], i
        if c2 < 0:
            break
        freq[c1] += freq[c2]
        freq[c2] = 0
        codesize[c1] += 1
        while others[c1] >= 0:
            c1 = others[c1]
            codesize[c1] += 1
        others[c1] = c2
        codesize[c2] += 1
        while others[c2] >= 0:
            c2 = others[c2]
            codesize[c2] += 1
    bits = [0] * 33
    for i in range(257):
        if codesize[i]:
            bits[codesize[i]] += 1
    for i in range(32, 16, -1):       # JPEG allows no code longer than 16 bits
        while bits[i] > 0:
            j = i - 2
            while bits[j] == 0:
                j -= 1
            bits[i] -= 2
            bits[i - 1] += 1
            bits[j + 1] += 2
            bits[j] -= 1
    i = 16
    while bits[i] == 0:               # drop the pseudo-symbol from the longest length
        i -= 1
    bits[i] -= 1
    vals = [j for ln in range(1, 33) for j in range(256) if codesize[j] == ln]
    return bits[1:17], vals


def lengths_to_table(lengths: dict):
    """{symbol: code length} -> (bits, vals), symbols of one length in increasing order"""
    bits = [0] * 16
    for ln in lengths.values():
        bits[ln - 1] += 1
    vals = sorted(lengths, key=lambda s: (lengths[s], s))
    return bits, vals


def check_table(bits, vals):
    """jdhuff.c jpeg_make_d_derived_tbl's conditions: every length fits with the all-ones code unused."""
    code = 0
    for ln in range(1, 17):
        code += bits[ln - 1]
        assert code < (1 << ln) or bits[ln - 1] == 0, "over-subscribed code length"
        code <<= 1
    assert sum(bits) == len(vals) <= 256


def fast_ac_edge_table(freq):
    """AC code lengths such that length + size is 10 or 11 for every used symbol (alternating by symbol), lengthened
    from the shortest where the code space would overflow."""
    used = [s for s in range(256) if freq[s]]
    ln = {s: min(16, max(1, (10 + (s & 1)) - (s & 15))) for s in used}
    while sum(2.0 ** -v for v in ln.values()) > 1 - 2.0 ** -16:
        s = min(ln, key=lambda t: (ln[t], -t))
        ln[s] += 1
    return lengths_to_table(ln)


def make_table(policy, cls: str, table_id: int, freq):
    if isinstance(policy, tuple):
        return policy
    if policy == "annex_k":
        if cls == "dc":
            return jm.DC_LUMA if table_id == 0 else jm.DC_CHROMA
        return jm.AC_LUMA if table_id == 0 else jm.AC_CHROMA
    m = re.fullmatch(r"all_len\((\d+)\)", policy)
    if m:
        n = int(m.group(1))
        used = [s for s in range(256) if freq[s]]
        assert len(used) < (1 << n), (n, len(used))
        return lengths_to_table({s: n for s in used})
    if policy == "dc_dup" and cls == "dc":
        return [0, 0, 0, 0, 16, 0, 0, 0, 0, 12, 0, 0, 0, 0, 0, 0], [0] * 16 + list(range(12))
    if policy == "fast_ac_edge" and cls == "ac":
        return fast_ac_edge_table(freq)
    if policy in ("optimal", "dc_dup", "fast_ac_edge", "eob_alias"):
        return gen_optimal_table(freq)
    raise ValueError(f"unknown table policy {policy!r}")


def derive_codes(bits, vals, pick: str):
    """symbol -> (code, length); a symbol listed twice takes its ``pick`` ("first" / "last") code"""
    codes, code, k = {}, 0, 0
    for ln in range(1, 17):
        for _ in range(bits[ln - 1]):
            if pick == "last" or vals[k] not in codes:
                codes[vals[k]] = (code, ln)
            code += 1
            k += 1
        code <<= 1
    co, si = np.zeros(256, np.int64), np.zeros(256, np.int64)
    for s, (c, ln) in codes.items():
        co[s], si[s] = c, ln
    return co, si


# ---- entropy-coded data --------------------------------------------------------------------------------------------
def nbits(v):
    a = np.abs(v)
    s = np.zeros(a.shape, np.int64)
    for b in range(16):
        s += a >= (1 << b)
    return s


def value_bits(v, s):
    """HUFF_EXTEND's inverse: v >= 0 as is, v < 0 as v - 1, in s bits"""
    return np.where(v < 0, v - 1, v) & ((np.int64(1) << s) - 1)


def scan_symbols(planes, comps, restart: int, eob_alias: bool):
    """Blocks in scan order -> token stream without codes: per token (block, order key, table class, symbol, value
    bits, value size, extra ZRL count)."""
    ncomp = len(comps)
    if ncomp == 1:
        pl = planes[0]
        blocks = pl.reshape(-1, 64)
        comp = np.zeros(len(blocks), np.int64)
        mcu = np.arange(len(blocks))
    else:
        h0, v0 = comps[0][1], comps[0][2]
        Y = planes[0]
        mcuy, mcux = Y.shape[0] // v0, Y.shape[1] // h0
        Y = Y.reshape(mcuy, v0, mcux, h0, 64).transpose(0, 2, 1, 3, 4).reshape(mcuy * mcux, v0 * h0, 64)
        parts = [Y] + [pl.reshape(mcuy * mcux, 1, 64) for pl in planes[1:]]
        blocks = np.concatenate(parts, axis=1)
        nb = blocks.shape[1]
        blocks = blocks.reshape(-1, 64)
        comp = np.tile(np.array([0] * (v0 * h0) + [1, 2]), mcuy * mcux)
        mcu = np.repeat(np.arange(mcuy * mcux), nb)
    nblk = len(blocks)
    Z = blocks[:, ZIGZAG].astype(np.int64)
    ivl = mcu // restart if restart else np.zeros(nblk, np.int64)
    # DC differences per component, predictors reset at every restart interval
    dc = Z[:, 0]
    diff = np.empty(nblk, np.int64)
    for c in range(ncomp):
        idx = np.nonzero(comp == c)[0]
        prev = np.concatenate([[0], dc[idx[:-1]]])
        first = np.concatenate([[True], ivl[idx[1:]] != ivl[idx[:-1]]])
        prev[first] = 0
        diff[idx] = dc[idx] - prev
    s = nbits(diff)
    tok = [dict(blk=np.arange(nblk), key=np.zeros(nblk, np.int64), cls=np.zeros(nblk, np.int64), sym=s,
                vb=value_bits(diff, s), vs=s, zrl=np.zeros(nblk, np.int64))]
    # AC: (run, size) symbols, ZRL for runs of 16, EOB (or an alias of it) after the last non-zero coefficient
    b, k = np.nonzero(Z[:, 1:])
    k = k + 1
    v = Z[b, k]
    kp = np.concatenate([[0], k[:-1]])
    kp[np.concatenate([[True], b[1:] != b[:-1]])] = 0
    run = k - kp - 1
    sz = nbits(v)
    tok.append(dict(blk=b, key=1 + 2 * k, cls=np.ones(len(b), np.int64), sym=((run & 15) << 4) | sz, vb=value_bits(v, sz),
                    vs=sz, zrl=run >> 4))
    last = np.zeros(nblk, np.int64)
    np.maximum.at(last, b, k)
    e = np.nonzero(last < 63)[0]
    eob = ((e % 15) << 4) if eob_alias else np.zeros(len(e), np.int64)
    tok.append(dict(blk=e, key=np.full(len(e), 200), cls=np.ones(len(e), np.int64), sym=eob, vb=np.zeros(len(e), np.int64),
                    vs=np.zeros(len(e), np.int64), zrl=np.zeros(len(e), np.int64)))
    T = {f: np.concatenate([t[f] for t in tok]) for f in tok[0]}
    order = np.lexsort((T["key"], T["blk"]))
    T = {f: a[order] for f, a in T.items()}
    T["comp"] = comp[T["blk"]]
    T["ivl"] = ivl[T["blk"]]
    return T, int(ivl[-1]) + 1


def pack_bits(code, length):
    """concatenate the codes MSB first -> 0/1 uint8 array"""
    out = []
    step = 1 << 19
    for a in range(0, len(code), step):
        c, ln = code[a:a + step], length[a:a + step]
        tot = int(ln.sum())
        if tot == 0:
            continue
        t = np.repeat(np.arange(len(c)), ln)
        j = np.arange(tot) - np.repeat(np.cumsum(ln) - ln, ln)
        out.append(((c[t] >> (ln[t] - 1 - j)) & 1).astype(np.uint8))
    return np.concatenate(out) if out else np.zeros(0, np.uint8)


def entropy_code(T, n_ivl, dc_codes, ac_codes, fill: int):
    """token stream -> entropy-coded segment (stuffed, with RSTn markers between intervals)"""
    n = len(T["sym"])
    co, si = np.zeros(n, np.int64), np.zeros(n, np.int64)
    for cls, codes in ((0, dc_codes), (1, ac_codes)):
        for c, (cc, ss) in codes.items():
            m = (T["cls"] == cls) & (T["comp"] == c)
            co[m], si[m] = cc[T["sym"][m]], ss[T["sym"][m]]
            assert (ss[T["sym"][m]] > 0).all(), "a symbol in use has no code"
    zco, zsi = np.zeros(n, np.int64), np.zeros(n, np.int64)
    for c, (cc, ss) in ac_codes.items():
        m = T["comp"] == c
        zco[m], zsi[m] = cc[0xF0], ss[0xF0]
    # per token: ZRL codes (0..3 of them), then the symbol's code, then its value bits
    nz = T["zrl"]
    assert (zsi[nz > 0] > 0).all(), "ZRL in use without a code"
    pieces_c = [np.where(nz > r, zco, 0) for r in range(3)] + [co, T["vb"]]
    pieces_l = [np.where(nz > r, zsi, 0) for r in range(3)] + [si, T["vs"]]
    code = np.stack(pieces_c, 1).reshape(-1)
    length = np.stack(pieces_l, 1).reshape(-1)
    ivl = np.repeat(T["ivl"], 5)
    # every interval ends byte-aligned, padded with 1-bits (jchuff.c flush_bits)
    per = np.bincount(ivl, weights=length, minlength=n_ivl).astype(np.int64)
    pad = (-per) % 8
    ends = np.searchsorted(ivl, np.arange(n_ivl), side="right")
    code = np.insert(code, ends, (1 << pad) - 1)
    length = np.insert(length, ends, pad)
    raw = np.packbits(pack_bits(code, length))
    nbytes = (per + pad) // 8
    bounds = np.cumsum(nbytes)[:-1]
    ff = np.nonzero(raw == 0xFF)[0]
    stuffed = np.insert(raw, ff + 1, 0)
    if n_ivl > 1:
        at = bounds + np.searchsorted(ff, bounds)
        mk = [[0xFF] * (1 + fill) + [0xD0 + (i & 7)] for i in range(n_ivl - 1)]
        stuffed = np.insert(stuffed, np.repeat(at, len(mk[0])), np.array(mk, np.uint8).reshape(-1))
    return stuffed.tobytes()


# ---- the file ------------------------------------------------------------------------------------------------------
def segment(marker: int, payload: bytes, fill: int = 0) -> bytes:
    return b"\xff" * fill + bytes([0xFF, marker]) + (len(payload) + 2).to_bytes(2, "big") + payload


EXIF_ORIENTATION_1 = (b"Exif\x00\x00MM\x00\x2a\x00\x00\x00\x08\x00\x01\x01\x12\x00\x03\x00\x00\x00\x01\x00\x01\x00\x00"
                      b"\x00\x00\x00\x00")
ICC_LIKE = b"ICC_PROFILE\x00\x01\x01" + bytes(range(128))


def write(data: bytes, tables="annex_k", pick: str = "last", ids=None, restart=None, layout=(), cids=None, lib=None,
          source=None) -> bytes:
    """Re-encode the baseline file ``data``.

    tables   a policy for every table, or ``{("dc" | "ac", component): policy}`` (see the module docstring)
    pick     which code a symbol listed twice in a table is written with: "first" or "last"
    ids      per component (dc table id, ac table id, quantisation table id), 0..3; default: as in the source.
             SOF1 is written when a Huffman table id is above 1 (as libjpeg does)
    restart  restart interval in MCUs (default: the source's; 0 = none)
    layout   any of LAYOUTS: every DHT in one segment, every DQT in one segment, the tables behind SOF, DRI before the
             DQTs, COM + APP2 (ICC-style) + APP1 (EXIF orientation 1) segments, 0xFF fill bytes before every marker
    cids     component ids of the frame / scan (default: the source's)
    lib      the loaded library: read the coefficients with its host stage (large files)
    source   (header, planes) of ``read_coefficients``, when the caller already has them
    """
    for f in layout:
        assert f in LAYOUTS, f
    p, planes = source if source is not None else read_coefficients(data, lib)
    frame = p["frame"]
    comps = frame["comps"]
    ncomp = len(comps)
    if ncomp == 1:
        comps = [(comps[0][0], 1, 1, comps[0][3])]
    sel = {cid: (td, ta) for cid, td, ta in p["scan"]}
    if ids is None:
        ids = [(sel[c[0]][0], sel[c[0]][1], c[3]) for c in comps]
    cids = list(cids) if cids is not None else [c[0] for c in frame["comps"]]
    restart = p["dri"] if restart is None else restart
    fill = 2 if "fill_bytes" in layout else 0
    pol = tables if isinstance(tables, dict) else None
    T, n_ivl = scan_symbols(planes, comps, restart, tables == "eob_alias" or (pol is not None and "eob_alias" in pol.values()))
    # one table per (class, id), from the symbol counts of every component that uses it
    built = {}
    codes = ({}, {})
    for cls_i, cls in enumerate(("dc", "ac")):
        for c in range(ncomp):
            tid = ids[c][cls_i]
            if (cls, tid) not in built:
                users = [k for k in range(ncomp) if ids[k][cls_i] == tid]
                m = (T["cls"] == cls_i) & np.isin(T["comp"], users)
                freq = np.bincount(T["sym"][m], minlength=256)
                if cls == "ac":
                    freq[0xF0] += int(T["zrl"][np.isin(T["comp"], users)].sum())
                policy = pol.get((cls, c), "annex_k") if pol is not None else tables
                bits, vals = make_table(policy, cls, tid, freq)
                check_table(bits, vals)
                built[(cls, tid)] = (list(bits), list(vals))
            codes[cls_i][c] = derive_codes(*built[(cls, tid)], pick)
    ecs = entropy_code(T, n_ivl, codes[0], codes[1], fill)

    # markers, in libjpeg's order unless the layout says otherwise
    out = b"\xff\xd8"
    j = 2
    while data[j] == 0xFF and 0xE0 <= data[j + 1] <= 0xEF:   # the source's APPn segments
        L = (data[j + 2] << 8) | data[j + 3]
        out += b"\xff" * fill + data[j:j + 2 + L]
        j += 2 + L
    if "extra_segments" in layout:
        out += segment(0xFE, b"re-encoded test file", fill) + segment(0xE2, ICC_LIKE, fill) + segment(0xE1, EXIF_ORIENTATION_1, fill)
    dri = segment(0xDD, restart.to_bytes(2, "big"), fill) if restart else b""
    q_order = []
    for c in range(ncomp):
        if ids[c][2] not in q_order:
            q_order.append(ids[c][2])
    qsrc = {ids[c][2]: p["qt"][comps[c][3]] for c in range(ncomp)}
    qtabs = [bytes([t]) + bytes(int(x) for x in qsrc[t][ZIGZAG]) for t in q_order]
    dqt = segment(0xDB, b"".join(qtabs), fill) if "dqt_one_segment" in layout else b"".join(segment(0xDB, q, fill) for q in qtabs)
    htabs = []
    for c in range(ncomp):
        for cls_i, cls in enumerate(("dc", "ac")):
            t = (cls, ids[c][cls_i])
            if t not in [h[0] for h in htabs]:
                bits, vals = built[t]
                htabs.append((t, bytes([(cls_i << 4) | t[1]]) + bytes(bits) + bytes(vals)))
    dht = (segment(0xC4, b"".join(h for _, h in htabs), fill) if "dht_one_segment" in layout
           else b"".join(segment(0xC4, h, fill) for _, h in htabs))
    sof_marker = 0xC1 if any(i[0] > 1 or i[1] > 1 for i in ids) else 0xC0
    sof = segment(sof_marker, bytes([8]) + frame["H"].to_bytes(2, "big") + frame["W"].to_bytes(2, "big") + bytes([ncomp]) +
                  b"".join(bytes([cids[c], (frame["comps"][c][1] << 4) | frame["comps"][c][2], ids[c][2]]) for c in range(ncomp)),
                  fill)
    sos = segment(0xDA, bytes([ncomp]) + b"".join(bytes([cids[c], (ids[c][0] << 4) | ids[c][1]]) for c in range(ncomp)) +
                  bytes([0, 63, 0]), fill)
    if "dri_before_dqt" in layout:
        out += dri
        dri = b""
    if "tables_after_sof" in layout:
        out += sof + dqt + dht
    else:
        out += dqt + sof + dht
    return out + dri + sos + ecs + b"\xff" * fill + b"\xff\xd9"


def variants(ncomp: int = 3):
    """(label, ``write`` keyword arguments): every table policy, table id assignment and segment layout of this module"""
    for pol in ("annex_k", "optimal", "all_len(9)", "all_len(10)", "all_len(16)", "fast_ac_edge", "dc_dup", "eob_alias"):
        yield pol, dict(tables=pol)
    yield "dc_dup pick first", dict(tables="dc_dup", pick="first")
    yield "dc_dup rst 1", dict(tables="dc_dup", restart=1)
    yield "all_len(16) rst 7", dict(tables="all_len(16)", restart=7)
    yield "eob_alias rst 3", dict(tables="eob_alias", restart=3)
    if ncomp == 3:
        yield "Cr on tables 2", dict(tables="optimal", ids=[(0, 0, 0), (1, 1, 1), (2, 2, 2)])
        yield "tables 3 2 1", dict(tables="all_len(10)", ids=[(3, 2, 1), (2, 3, 0), (1, 0, 3)])
        yield "per component", dict(ids=[(0, 0, 0), (1, 1, 1), (2, 2, 2)], tables={
            ("dc", 0): "dc_dup", ("ac", 0): "all_len(16)", ("dc", 1): "all_len(10)", ("ac", 1): "fast_ac_edge",
            ("dc", 2): "optimal", ("ac", 2): "eob_alias"})
    else:
        yield "table 3", dict(tables="optimal", ids=[(3, 3, 3)])
    for lay in LAYOUTS:
        yield lay, dict(tables="optimal", layout=(lay,), restart=0 if lay == "fill_bytes" else None)
        if lay in ("fill_bytes", "dri_before_dqt"):
            yield lay + " rst 2", dict(tables="optimal", layout=(lay,), restart=2)
    yield "every layout, dc_dup, rst 2", dict(tables="dc_dup", layout=LAYOUTS, restart=2)
    yield "component ids 0 1 2", dict(tables="optimal", cids=[0, 1, 2][:ncomp])
