"""The designed PNG-encoder corpus (tests/png_streams.py) on the CPU: the oracle's deflate equals zlib's and its files equal
cv2.imencode's for every designed stream, and the corpus reaches each rare path of zlib's deflate_rle / trees.c it is
designed for - read from the oracle's per-block records and the runs of the stream, never assumed."""
import zlib

import cv2
import numpy as np
import pytest

import png_streams as ps
from oracle import png_model as pm

CORPUS = ps.corpus()


@pytest.fixture(scope="module")
def records():
    """family -> [(name, W, F, per-block records)]"""
    out = {}
    for fam, name, W, F in CORPUS:
        out.setdefault(fam, []).append((name, W, F, ps.deflate_records(F)[1]))
    return out


def blocks(records, fam):
    return [r for _, _, _, st in records[fam] for r in st]


@pytest.mark.parametrize("fam,name,W,F", CORPUS, ids=[f"{c[0]}-{c[1]}" for c in CORPUS])
def test_designed_stream_oracle_equals_zlib_and_cv2(fam, name, W, F):
    img = ps.image_from_filtered(F, W)              # asserts sub_filter(img) == F
    co = zlib.compressobj(1, zlib.DEFLATED, 15, 8, zlib.Z_RLE)
    stats = []
    assert pm.deflate_rle(F.tobytes(), stats=stats)[0] == co.compress(F.tobytes()) + co.flush()
    assert pm.encode_png(img) == cv2.imencode(".png", img)[1].tobytes()
    assert sum(r["bytes"] for r in stats) == len(F)
    assert stats[-1]["last"] == 1 and all(r["last"] == 0 for r in stats[:-1])


def test_records_leave_the_stream_unchanged():
    F = CORPUS[0][3].tobytes()
    assert pm.deflate_rle(F, stats=[]) == pm.deflate_rle(F)


def test_literal_tree_repair(records):
    ovf = {r["l_overflow"] for r in blocks(records, "lit_overflow")}
    assert {2, 4, 6} <= ovf
    # match-length symbols among the deep leaves of a repaired tree (length codes 257 .. 285 in the chain)
    with_lengths = [r for name, _, _, st in records["lit_overflow"] if "lengths" in name for r in st]
    assert any(r["l_overflow"] and 258 in r["lengths"] and 3 in r["lengths"] for r in with_lengths)
    assert any(r["l_overflow"] and len(r["lengths"]) >= 11 for r in with_lengths)


def test_bit_length_tree_repair(records):
    assert any(r["bl_overflow"] for r in blocks(records, "bl_overflow"))


def test_static_blocks(records):
    st = blocks(records, "static")
    flat = [r for r in st if r["kind"] == "static" and len(r["lengths"]) >= 29]
    assert flat, "a static block holding matches of every length code"
    lc = {pm.length_code[L - 3] for r in flat for L in r["lengths"]}
    assert lc == set(range(29)) and any(258 in r["lengths"] for r in flat)
    _, _, F, recs = next(x for x in records["static"] if x[0] == "flat")
    assert set(F[1:].tolist()) >= set(range(256)) - {1}
    dyn_then = next(x[3] for x in records["static"] if x[0] == "dynamic_then_flat")
    assert [r["kind"] for r in dyn_then][0] == "dynamic"
    assert any(r["kind"] == "static" and r["last"] for fam in records for r in blocks(records, fam))


def test_largest_tree_description(records):
    hdr = max(r["hdr_bits"] for r in blocks(records, "big_header"))
    print(f"largest dynamic header reached: {hdr} bits")
    assert hdr > 1000
    assert hdr <= 71 + 288 * 7 < 80 * 32                 # the device's BlockInfo.hdr holds 80 words


def test_stored_blocks(records):
    allb = [r for fam in records for r in blocks(records, fam)]
    stored = [r for r in allb if r["kind"] == "stored"]
    residues = set()
    for fam in records:
        for _, _, _, st in records[fam]:
            for a, b in zip(st, st[1:]):
                if b["kind"] == "stored" and a["kind"] != "stored":
                    residues.add(b["start_bit"] % 8)
            if any(a["kind"] == b["kind"] == "stored" for a, b in zip(st, st[1:])):
                residues.add("after_stored")
    assert residues >= set(range(8)) | {"after_stored"}, residues
    assert any(r["kind"] == "stored" and r["last"] for r in allb)
    # DESIGN's claim (p2p_png.cuh, stored-block comment): every stored block has < 16383 + 1300 bytes
    assert max(r["bytes"] for r in stored) < 16383 + 1300


def test_exact_block_fills(records):
    fills = {name: st for name, _, _, st in records["fill"]}
    for name in ("runfree14x381", "runfree42x258"):
        st = fills[name]
        assert st[-1]["tokens"] == 0 and st[-1]["kind"] == "static" and all(r["tokens"] == 16383 for r in st[:-1])
    assert sum(r["tokens"] for r in fills["runfree2730x2"]) == 16382
    assert sum(r["tokens"] for r in fills["runfree5x1024"]) == 16384
    st = fills["match258_last"]
    assert st[0]["tokens"] == 16383 and 258 in st[0]["lengths"]
    _, _, F, _ = next(x for x in records["fill"] if x[0] == "match258_last")
    toks = pm.tokenize_rle(F.tobytes())
    assert toks[16382] == ("M", 258)


def test_runs_at_tokeniser_edges(records):
    items = {name: (W, F) for name, W, F, _ in records["runs"]}
    for r in range(4):
        W, F = items[f"ramp{r}"]
        assert (F == 1).all() and (len(F) - 1) % 258 == r
    residues, ends_behind, long_runs, short_runs = set(), set(), False, set()
    for name, (W, F) in items.items():
        for s, e in ps.runs(F):
            for B in range((s // ps.TILE + 1) * ps.TILE, e, ps.TILE):
                residues.add((B - s - 1) % 258)                 # the run crosses tile boundary B
            B = (e - 1) // ps.TILE * ps.TILE                      # the run ends d bytes behind the tile boundary B
            if s < B:
                ends_behind.add(e - B)
            if e - s > ps.TILE + ps.LOOK:
                long_runs = True
            short_runs.add(e - s)
        if name == "tile_ends":
            assert F[-1] == F[-2] and ps.runs(F)[-1][1] == len(F)   # a run ending at N
    assert residues == set(range(258))
    assert {1, 2, 256, 257, 258, 288, 289} <= ends_behind, sorted(ends_behind)[:20]
    # matches starting at a tile's last byte whose length the look-ahead decides (run ends 250 .. 258 bytes behind it)
    W, F = items["tile_ends"]
    toks, at, seen = pm.tokenize_rle(F.tobytes()), 0, set()
    for t, v in toks:
        if t == "M" and at % ps.TILE == ps.TILE - 1:
            seen.add(v)
        at += 1 if t == "L" else v
    assert {255, 256, 257, 258} <= seen, sorted(seen)
    assert long_runs and {2, 3, 4} <= short_runs
    W, F = items["width1"]
    assert W == 1 and F[0] == 0 and any(e - s > 4 * 3 for s, e in ps.runs(F))   # runs across rows of 4 bytes
