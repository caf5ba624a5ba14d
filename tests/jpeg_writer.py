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
    return pack_intervals(code, length, np.repeat(T["ivl"], 5), n_ivl, fill)


def pack_intervals(code, length, ivl, n_ivl: int, fill: int):
    """bit pieces (code, length; interval of each, non-decreasing) -> entropy-coded segment: every interval padded with
    1-bits to a byte, 0xFF stuffed, RSTn markers (``fill`` 0xFF fill bytes in front of each) between intervals"""
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


# ---- progressive files (jcphuff.c) ---------------------------------------------------------------------------------
# A scan is (component indices in scan order, Ss, Se, Ah, Al); a script is a list of scans.  The entropy coder is
# jcphuff.c's: DC first with the point transform (an arithmetic shift) and a predictor per component, DC refinement as raw
# bits, AC first with end-of-band runs (EOBRUN), AC refinement with the correction bits buffered in the run (BE) or since
# the last symbol (BR); a run is forced out at 0x7FFF, when its buffered bits could overflow jcphuff.c's MAX_CORR_BITS
# buffer during the next block, in front of a restart marker and at the end of the scan.  With the "simple" script and
# optimal tables (every scan gets its own, as jcphuff.c's statistics pass makes them) the output is byte for byte the file
# cv2.imencode(..., [IMWRITE_JPEG_PROGRESSIVE, 1]) writes.
MAX_EOBRUN = 0x7FFF
MAX_CORR_BITS = 1000


def script(name: str, ncomp: int = 3):
    """the scans of a named script (SCRIPTS); a gray file (one component) keeps the scans of component 0"""
    Y, Cb, Cr, ALL = (0,), (1,), (2,), (0, 1, 2)
    if name in ("simple", "rst_everywhere", "table_churn"):
        if ncomp == 1:   # jcparam.c jpeg_simple_progression, the all-purpose script
            return [(Y, 0, 0, 0, 1), (Y, 1, 5, 0, 2), (Y, 6, 63, 0, 2), (Y, 1, 63, 2, 1), (Y, 0, 0, 1, 0), (Y, 1, 63, 1, 0)]
        return [(ALL, 0, 0, 0, 1), (Y, 1, 5, 0, 2), (Cr, 1, 63, 0, 1), (Cb, 1, 63, 0, 1), (Y, 6, 63, 0, 2),
                (Y, 1, 63, 2, 1), (ALL, 0, 0, 1, 0), (Cr, 1, 63, 1, 0), (Cb, 1, 63, 1, 0), (Y, 1, 63, 1, 0)]
    if name == "mozjpeg_like":       # one DC scan per component, luma bands split
        s = [(Y, 0, 0, 0, 1), (Cb, 0, 0, 0, 1), (Cr, 0, 0, 0, 1), (Y, 1, 8, 0, 2), (Y, 9, 63, 0, 2), (Cb, 1, 63, 0, 0),
             (Cr, 1, 63, 0, 0), (Y, 1, 63, 2, 1), (Y, 1, 63, 1, 0), (Y, 0, 0, 1, 0), (Cb, 0, 0, 1, 0), (Cr, 0, 0, 1, 0)]
    elif name == "spectral_only":    # spectral selection without successive approximation
        s = [(ALL, 0, 0, 0, 0), (Y, 1, 5, 0, 0), (Y, 6, 63, 0, 0), (Cb, 1, 63, 0, 0), (Cr, 1, 63, 0, 0)]
    elif name == "deep_sa":          # three refinement levels: Ah 3 -> 2 -> 1 -> 0 for DC and AC
        s = [(ALL, 0, 0, 0, 3), (Y, 1, 63, 0, 3), (Cb, 1, 63, 0, 3), (Cr, 1, 63, 0, 3)]
        for al in (2, 1, 0):
            s += [(ALL, 0, 0, al + 1, al), (Y, 1, 63, al + 1, al), (Cb, 1, 63, al + 1, al), (Cr, 1, 63, al + 1, al)]
    elif name == "single_coef":      # bands of one or two coefficients (Ss == Se)
        s = [(ALL, 0, 0, 0, 0)] + [(Y, k, k, 0, 0) for k in range(1, 21)] + [(Y, k, k + 1, 0, 0) for k in range(21, 63, 2)]
        s += [(Y, 63, 63, 0, 0), (Cb, 1, 1, 0, 0), (Cb, 2, 63, 0, 0), (Cr, 1, 2, 0, 0), (Cr, 3, 63, 0, 0)]
    elif name == "dc_subset":        # interleaved DC scans over a subset of the components
        s = [(Y, 0, 0, 0, 1), ((1, 2), 0, 0, 0, 1), (Y, 1, 63, 0, 1), (Cb, 1, 63, 0, 0), (Cr, 1, 63, 0, 0),
             ((1, 2), 0, 0, 1, 0), (Y, 1, 63, 1, 0), (Y, 0, 0, 1, 0)]
    elif name == "chroma_first":     # DC refinement right after DC first, every chroma scan before luma AC
        s = [(ALL, 0, 0, 0, 1), (ALL, 0, 0, 1, 0), (Cr, 1, 63, 0, 1), (Cb, 1, 63, 0, 1), (Cr, 1, 63, 1, 0),
             (Cb, 1, 63, 1, 0), (Y, 1, 63, 0, 1), (Y, 1, 63, 1, 0)]
    elif name == "over_cap":         # 65 scans and more: one per luma coefficient
        s = [(ALL, 0, 0, 0, 1), (ALL, 0, 0, 1, 0)] + [(Y, k, k, 0, 0) for k in range(1, 64)] + [(Cb, 1, 63, 0, 0), (Cr, 1, 63, 0, 0)]
    else:
        raise ValueError(f"unknown script {name!r}")
    if ncomp == 1:
        s = [((0,), ss, se, ah, al) for comps, ss, se, ah, al in s if 0 in comps]
    return s


def named(name: str, ncomp: int = 3) -> dict:
    """``write_progressive`` keyword arguments of a named script: the scans, and for rst_everywhere a restart interval per
    scan (1, a prime, none, ...; DRI written whenever it changes), for table_churn table ids 0-3 rotating over the scans
    with a decoy DHT before every scan that redefines a slot the scan does not use (the next scan using it sends its own)"""
    s = script(name, ncomp)
    kw = dict(script=s)
    if name == "rst_everywhere":
        kw["restart"] = [(1, 13, 0, 7, 1, 0)[k % 6] for k in range(len(s))]
    if name == "table_churn":
        kw["slots"] = [[(k + j) % 4 for j in range(len(sc[0]))] for k, sc in enumerate(s)]
        kw["decoy"] = True
    return kw


SCRIPTS = ("simple", "mozjpeg_like", "spectral_only", "deep_sa", "single_coef", "dc_subset", "chroma_first",
           "rst_everywhere", "table_churn", "over_cap")


def _frame_geometry(p):
    """(normalised frame components [(id, h, v, tq)], hmax, vmax)"""
    comps = p["frame"]["comps"]
    if len(comps) == 1:
        comps = [(comps[0][0], 1, 1, comps[0][3])]
    return comps, max(c[1] for c in comps), max(c[2] for c in comps)


def _scan_blocks(planes, comps, hmax, vmax, W, H, sc):
    """blocks of a scan in coding order -> (zigzag coefficients [n, 64], component of each block, MCU of each block).
    One component: its own ceil(width / 8) x ceil(height / 8) blocks; several: MCUs of the frame, padding blocks included."""
    if len(sc) == 1:
        c = sc[0]
        wc, hc = -(-W * comps[c][1] // hmax), -(-H * comps[c][2] // vmax)
        blocks = planes[c][:-(-hc // 8), :-(-wc // 8)].reshape(-1, 64)
        return blocks[:, ZIGZAG].astype(np.int64), np.full(len(blocks), c), np.arange(len(blocks))
    mcuy, mcux = -(-H // (8 * vmax)), -(-W // (8 * hmax))
    parts, owner = [], []
    for c in sc:
        h, v = comps[c][1], comps[c][2]
        parts.append(planes[c].reshape(mcuy, v, mcux, h, 64).transpose(0, 2, 1, 3, 4).reshape(mcuy * mcux, v * h, 64))
        owner += [c] * (v * h)
    blocks = np.concatenate(parts, axis=1)
    nb = blocks.shape[1]
    return (blocks.reshape(-1, 64)[:, ZIGZAG].astype(np.int64), np.tile(np.array(owner), mcuy * mcux),
            np.repeat(np.arange(mcuy * mcux), nb))


class _Pieces:
    """bit pieces of a scan: Huffman symbols (table slot, symbol) or raw bits (value, length), with a sort key
    (block, position, sub-order, order)"""

    def __init__(self):
        self.parts = []

    def add(self, blk, pos, sub, order, slot, sym, val, ln):
        n = len(blk)
        f = lambda x: np.broadcast_to(np.asarray(x, np.int64), (n,))
        self.parts.append([f(blk), f(pos), f(sub), f(order), f(slot), f(sym), f(val), f(ln)])

    def sorted(self):
        a = [np.concatenate([p[i] for p in self.parts]) for i in range(8)]
        o = np.lexsort((a[3], a[2], a[1], a[0]))
        return [x[o] for x in a]


def _previous_true(nz):
    """per position of a [n, w] mask: index of the previous True strictly before it in its row (-1 if none)"""
    n, w = nz.shape
    idx = np.where(nz, np.arange(w), -1)
    prev = np.maximum.accumulate(idx, axis=1)
    return np.concatenate([np.full((n, 1), -1), prev[:, :-1]], axis=1)


def _ac_pieces(P, Z, Ss, Se, Ah, Al, slot, chunk=1 << 16):
    """AC first / refinement scan of one component: symbol pieces of every block; returns per block (has a symbol, ends
    in an end-of-band, count of correction bits for the run buffer) and the buffered bits (block, order, bit)"""
    w = Se - Ss + 1
    n = len(Z)
    has_sym, trailing, be = np.zeros(n, bool), np.zeros(n, bool), np.zeros(n, np.int64)
    be_parts = []
    jj = np.arange(w)
    for c0 in range(0, n, chunk):
        A = Z[c0:c0 + chunk, Ss:Se + 1]
        a = np.abs(A) >> Al
        m = len(A)
        if Ah == 0:
            nz = a != 0
            last = np.where(nz.any(1), w - 1 - np.argmax(nz[:, ::-1], 1), -1)
            prev = _previous_true(nz)
            b, j = np.nonzero(nz)
            run = j - prev[b, j] - 1
            nzrl = run >> 4
            rb = np.repeat(b, nzrl)
            P.add(c0 + rb, Ss + np.repeat(j, nzrl), 0, np.arange(len(rb)), slot, 0xF0, 0, 0)
            s = nbits(a[b, j])
            v = np.where(A[b, j] < 0, -a[b, j], a[b, j])
            P.add(c0 + b, Ss + j, 3, 0, slot, ((run & 15) << 4) | s, 0, 0)
            P.add(c0 + b, Ss + j, 4, 0, -1, 0, value_bits(v, s), s)
        else:
            new, old, zero = a == 1, a > 1, a == 0
            last = np.where(new.any(1), w - 1 - np.argmax(new[:, ::-1], 1), -1)
            before_last = jj[None, :] <= last[:, None]
            cz = np.cumsum(zero, axis=1)
            base = np.maximum.accumulate(np.where(new, cz, 0), axis=1)          # zeros up to the latest new coefficient
            base = np.concatenate([np.zeros((m, 1), np.int64), base[:, :-1]], axis=1)
            zr = cz - base                                                      # zeros since the last symbol
            F = zr >> 4                                                         # ZRLs emitted up to here
            nzm = (new | old) & before_last                                     # ZRLs only up to the last new one
            prev = _previous_true(new | old)
            pc = np.clip(prev, 0, None)
            rows = np.arange(m)[:, None]
            same_seg = (prev >= 0) & old[rows, pc]
            zrl_at = np.where(nzm, F - np.where(same_seg, F[rows, pc], 0), 0)
            event = nzm & ((zrl_at > 0) | new)
            # correction bits up to the last new coefficient go out behind the first code of the next event
            nxt = np.where(event, jj, w)
            nxt = np.minimum.accumulate(nxt[:, ::-1], axis=1)[:, ::-1]
            nxt = np.concatenate([nxt[:, 1:], np.full((m, 1), w)], axis=1)    # next event strictly after
            b, j = np.nonzero(zrl_at > 0)
            P.add(c0 + b, Ss + j, 0, 0, slot, 0xF0, 0, 0)
            more = zrl_at[b, j] - 1
            rb, rj = np.repeat(b, more), np.repeat(j, more)
            P.add(c0 + rb, Ss + rj, 2, np.arange(len(rb)), slot, 0xF0, 0, 0)
            b, j = np.nonzero(new)
            P.add(c0 + b, Ss + j, 3, 0, slot, ((zr[b, j] & 15) << 4) | 1, 0, 0)
            P.add(c0 + b, Ss + j, 4, 0, -1, 0, (A[b, j] > 0).astype(np.int64), 1)
            b, j = np.nonzero(old & before_last)
            t = nxt[b, j]
            P.add(c0 + b, Ss + t, np.where(zrl_at[b, t] > 0, 1, 5), j, -1, 0, a[b, j] & 1, 1)
            b, j = np.nonzero(old & ~before_last)                              # behind the last new one: the run's buffer
            be_parts.append((c0 + b, j, a[b, j] & 1))
            be[c0:c0 + m] = np.bincount(b, minlength=m)
        has_sym[c0:c0 + m] = last >= 0
        trailing[c0:c0 + m] = last < w - 1
    return has_sym, trailing, be, be_parts


def _eob_runs(P, has_sym, trailing, be, be_parts, ivl, slot):
    """jcphuff.c's end-of-band runs: blocks that end in an end-of-band join the pending run, which is sent (EOBn symbol,
    run bits, then its buffered correction bits) in front of the next block with a symbol, in front of a restart marker,
    at the end of the scan, and as soon as it reaches 0x7FFF blocks or more than MAX_CORR_BITS - 63 buffered bits"""
    n = len(has_sym)
    start = has_sym.copy()
    start[0] = True
    start[1:] |= ivl[1:] != ivl[:-1]
    g = np.cumsum(start) - 1
    gs = np.nonzero(start)[0]
    ge = np.append(gs[1:], n) - 1
    t = trailing.astype(np.int64)
    ct, cb = np.cumsum(t), np.cumsum(be)
    gcnt, gbe = np.bincount(g, weights=t).astype(np.int64), np.bincount(g, weights=be).astype(np.int64)
    limit = MAX_CORR_BITS - 64 + 1
    light = (gcnt > 0) & (gcnt < MAX_EOBRUN) & (gbe <= limit)
    his = [ge[light]]
    for k in np.nonzero(((gcnt >= MAX_EOBRUN) | (gbe > limit)))[0]:
        cur, end = gs[k], ge[k]
        while cur <= end:
            bt, bb = (ct[cur - 1], cb[cur - 1]) if cur else (0, 0)
            j = min(np.searchsorted(ct, bt + MAX_EOBRUN, "left"), np.searchsorted(cb, bb + limit, "right"))
            if j > end:
                if ct[end] > bt:
                    his.append([end])
                break
            his.append([j])
            cur = j + 1
    hi = np.sort(np.concatenate([np.asarray(h, np.int64) for h in his]))
    lo = np.append(0, hi[:-1] + 1)
    cnt = ct[hi] - np.where(lo > 0, ct[np.maximum(lo - 1, 0)], 0)
    nb = nbits(cnt) - 1
    P.add(hi, 1000, 0, 0, slot, nb << 4, 0, 0)
    P.add(hi, 1000, 1, 0, -1, 0, cnt & ((1 << nb) - 1), nb)
    for b, j, bit in be_parts:
        h = hi[np.searchsorted(hi, b, "left")]
        P.add(h, 1000, 2, b * 64 + j, -1, 0, bit, 1)


def _encode_scan(planes, comps, hmax, vmax, W, H, sc, Ss, Se, Ah, Al, slots, restart, tables, fill):
    """one scan -> (entropy-coded bytes, {(class, slot): (bits, vals)} of the tables it uses)"""
    Z, owner, mcu = _scan_blocks(planes, comps, hmax, vmax, W, H, sc)
    n = len(Z)
    ivl = mcu // restart if restart else np.zeros(n, np.int64)
    n_ivl = int(ivl[-1]) + 1
    P = _Pieces()
    blk = np.arange(n)
    if Ss == 0 and Ah == 0:
        v = Z[:, 0] >> Al
        diff = np.empty(n, np.int64)
        for c in sc:
            idx = np.nonzero(owner == c)[0]
            prev = np.concatenate([[0], v[idx[:-1]]])
            prev[np.concatenate([[True], ivl[idx[1:]] != ivl[idx[:-1]]])] = 0
            diff[idx] = v[idx] - prev
        s = nbits(diff)
        slot_of = np.zeros(3, np.int64)
        slot_of[list(sc)] = slots
        P.add(blk, 0, 0, 0, slot_of[owner], s, 0, 0)
        P.add(blk, 0, 1, 0, -1, 0, value_bits(diff, s), s)
    elif Ss == 0:
        P.add(blk, 0, 0, 0, -1, 0, (Z[:, 0] >> Al) & 1, 1)
    else:
        has_sym, trailing, be, be_parts = _ac_pieces(P, Z, Ss, Se, Ah, Al, slots[0])
        _eob_runs(P, has_sym, trailing, be, be_parts, ivl, slots[0])
    pb, _, _, _, pslot, psym, pval, pln = P.sorted()
    cls = "dc" if Ss == 0 else "ac"
    built, code, length = {}, pval.copy(), pln.copy()
    for sl in sorted(set(slots)) if not (Ss == 0 and Ah) else []:
        m = pslot == sl
        freq = np.bincount(psym[m], minlength=256)
        bits, vals = make_table(tables, cls, sl, freq)
        check_table(bits, vals)
        co, si = derive_codes(bits, vals, "last")
        assert (si[psym[m]] > 0).all(), "a symbol in use has no code"
        code[m], length[m] = co[psym[m]], si[psym[m]]
        built[(cls, sl)] = (list(bits), list(vals))
    return pack_intervals(code, length, ivl[pb], n_ivl, fill), built


def write_progressive(data: bytes, script="simple", restart=None, slots=None, decoy=False, tables="optimal", layout=(),
                      lib=None, source=None) -> bytes:
    """Re-encode the coefficients of ``data`` (any file ``read_coefficients`` takes) as a progressive (SOF2) file.

    script   a name of SCRIPTS or a list of scans (components, Ss, Se, Ah, Al); component indices in scan order
    restart  restart interval in MCUs for every scan, or a list with one per scan (default: the source's); a DRI segment
             is written in front of a scan whenever the interval changes, as libjpeg does
    slots    per scan, the table id of each of its components (default: libjpeg's - 0 for luma, 1 for chroma)
    decoy    a DHT before every scan that redefines a table slot the scan does not use
    tables   a table policy of ``make_table`` for every table of every scan ("optimal": jcphuff.c's per-scan tables)
    layout   any of LAYOUTS; "extra_segments" also puts a COM segment between the scans, "fill_bytes" puts 0xFF fill
             bytes before every marker, restart markers included
    """
    for f in layout:
        assert f in LAYOUTS, f
    p, planes = source if source is not None else read_coefficients(data, lib)
    comps, hmax, vmax = _frame_geometry(p)
    ncomp = len(comps)
    kw = named(script, ncomp) if isinstance(script, str) else dict(script=script)
    scans = kw["script"]
    restart = kw.get("restart", restart)
    slots = kw.get("slots", slots)
    decoy = kw.get("decoy", decoy)
    W, H = p["frame"]["W"], p["frame"]["H"]
    restarts = restart if isinstance(restart, (list, tuple)) else [p["dri"] if restart is None else restart] * len(scans)
    if slots is None:
        slots = [[0 if c == 0 else 1 for c in sc[0]] for sc in scans]
    fill = 2 if "fill_bytes" in layout else 0

    out = b"\xff\xd8"
    j = 2
    while data[j] == 0xFF and 0xE0 <= data[j + 1] <= 0xEF:   # the source's APPn segments
        L = (data[j + 2] << 8) | data[j + 3]
        out += b"\xff" * fill + data[j:j + 2 + L]
        j += 2 + L
    if "extra_segments" in layout:
        out += segment(0xFE, b"re-encoded test file", fill) + segment(0xE2, ICC_LIKE, fill) + segment(0xE1, EXIF_ORIENTATION_1, fill)
    qts = []
    for c in comps:
        if c[3] not in qts:
            qts.append(c[3])
    qtabs = [bytes([t]) + bytes(int(x) for x in p["qt"][t][ZIGZAG]) for t in qts]
    dqt = segment(0xDB, b"".join(qtabs), fill) if "dqt_one_segment" in layout else b"".join(segment(0xDB, q, fill) for q in qtabs)
    sof = segment(0xC2, bytes([8]) + H.to_bytes(2, "big") + W.to_bytes(2, "big") + bytes([ncomp]) +
                  b"".join(bytes([c[0], (c[1] << 4) | c[2], c[3]]) for c in comps), fill)
    last_dri = 0
    if "dri_before_dqt" in layout and restarts[0]:
        out += segment(0xDD, restarts[0].to_bytes(2, "big"), fill)
        last_dri = restarts[0]
    out += sof + dqt if "tables_after_sof" in layout else dqt + sof
    for k, ((sc, Ss, Se, Ah, Al), rst, sl) in enumerate(zip(scans, restarts, slots)):
        ecs, built = _encode_scan(planes, comps, hmax, vmax, W, H, sc, Ss, Se, Ah, Al, sl, rst, tables, fill)
        if k and "extra_segments" in layout:
            out += segment(0xFE, b"between scans %d and %d" % (k - 1, k), fill)
        if decoy:
            free = [s for s in range(4) if s not in sl][0]
            out += segment(0xC4, bytes([(0 if Ss else 1) << 4 | free]) + bytes([0] * 7 + [255] + [0] * 8) + bytes(range(255)), fill)
        htabs = []
        for c, s in zip(sc, sl):
            for cls_i, cls in enumerate(("dc", "ac")):
                if (cls, s) in built and (cls, s) not in [h[0] for h in htabs]:
                    bits, vals = built[(cls, s)]
                    htabs.append(((cls, s), bytes([(cls_i << 4) | s]) + bytes(bits) + bytes(vals)))
        if htabs:
            out += (segment(0xC4, b"".join(h for _, h in htabs), fill) if "dht_one_segment" in layout
                    else b"".join(segment(0xC4, h, fill) for _, h in htabs))
        if rst != last_dri:
            out += segment(0xDD, rst.to_bytes(2, "big"), fill)
            last_dri = rst
        sel = b"".join(bytes([comps[c][0], ((s if Ss == 0 and Ah == 0 else 0) << 4) | (s if Ss else 0)]) for c, s in zip(sc, sl))
        out += segment(0xDA, bytes([len(sc)]) + sel + bytes([Ss, Se, (Ah << 4) | Al]), fill) + ecs
    return out + b"\xff" * fill + b"\xff\xd9"
