"""Designed deflate streams (tests/deflate_writer.py) on the CPU: every stream inflates with zlib to its designed bytes,
the shapes each design claims to reach are read back from its block records, and the library's host model of the PNG
decoder (``p2p_png_decode_host``: the device pipeline's routines run serially) decodes every file like ``cv2.imdecode``
and finds every dynamic block with its block-start search.  No GPU needed."""
import ctypes as C
import zlib

import cv2
import numpy as np
import pytest

import deflate_writer as D

HOST_DECLINES = {"decline:max_syms", "decline:cinfo_window"}   # the host model has no caps and no host budget


def cv2_decode(data: bytes):
    return cv2.imdecode(np.frombuffer(data, np.uint8), cv2.IMREAD_COLOR)


@pytest.fixture(scope="module")
def host_decode(pkg):
    lib = pkg._lib.load()

    def run(data: bytes):
        w, h = C.c_int(), C.c_int()
        assert lib.p2p_png_probe(data, len(data), C.byref(w), C.byref(h)) == 0
        out = np.zeros((h.value, w.value, 3), np.uint8)
        stats = (C.c_uint64 * 4)()
        rc = lib.p2p_png_decode_host(data, len(data), out.ctypes.data, out.strides[0], h.value, stats)
        return rc, out, list(stats)

    return run


def recs_of(*families):
    c = D.corpus()
    return [(d, i, r) for f in families for d in c[f] for i, r in enumerate(d.recs)]


def dyn(*families):
    return [(d, i, r) for d, i, r in recs_of(*families) if r.kind == "dynamic"]


ALL = list(D.corpus())


@pytest.mark.parametrize("design", D.all_designs(), ids=lambda d: d.name)
def test_every_stream_inflates_to_its_designed_bytes(design):
    if design.expect == "invalid":
        with pytest.raises(zlib.error):
            zlib.decompress(design.z)
    else:
        assert zlib.decompress(design.z) == design.data
    assert sum(r.out_len for r in design.recs) == len(design.data)
    assert design.recs[-1].final and not any(r.final for r in design.recs[:-1])
    assert design.recs[0].start == 16
    for a, b in zip(design.recs, design.recs[1:]):
        assert a.end == b.start
    assert (design.recs[-1].end + 7) // 8 + 4 == len(design.z)


def test_header_shapes_are_reached():
    R = [r for _, _, r in dyn(*ALL)]
    assert {257, 286} <= {r.hlit for r in R} and {1, 30} <= {r.hdist for r in R}
    assert set(range(5, 20)) <= {r.hclen for r in R}
    # a code-length code with a 7-bit code in use
    assert any(max(r.cl_lens[s] for s, _ in r.cl_runs) == 7 for r in R)
    # distance trees: empty (HDIST 1 and 30), a single code of length 1; a literal tree holding only end-of-block
    assert any(r.hdist == 1 and not any(r.distlens) and r.n_tokens for r in R)
    assert any(r.hdist == 30 and not any(r.distlens) for r in R)
    assert any(sorted(l for l in r.distlens if l) == [1] and r.dsyms for r in R)
    assert any([l for l in r.litlens if l] == [1] and r.litlens[256] == 1 and r.out_len == 0 for r in R)
    # code-length repeats crossing from the literal / length lengths into the distance lengths: a zero run and a 16 run
    crossing = set()
    for r in R:
        at = 0
        for s, e in r.cl_runs:
            n = 1 if s < 16 else (3 if s < 18 else 11) + e
            if s >= 16 and at < r.hlit < at + n:
                crossing.add(s)
            at += n
    assert {16, 18} <= crossing or {16, 17} <= crossing, crossing
    assert any((18, 127) in r.cl_runs for r in R)
    # literal / length codes of every length 1 .. 15 and distance codes of 9 .. 15 bits actually used
    lit_used, dist_used = set(), set()
    for r in R:
        lit_used |= {r.litlens[s] for s in r.lits | {ls for ls, _ in r.lsyms} | {256}}
        dist_used |= {r.distlens[ds] for ds, _ in r.dsyms}
    assert set(range(1, 16)) <= lit_used
    assert set(range(9, 16)) <= dist_used


def test_every_length_and_distance_symbol_at_both_extra_ends():
    lsyms, dsyms, dists = set(), set(), set()
    for d, _, r in recs_of(*ALL):
        lsyms |= r.lsyms
        dsyms |= r.dsyms
        dists |= {D.match_dist(c, e) for c, e in r.dsyms}
    for k in range(29):
        assert {(257 + k, 0), (257 + k, (1 << D.LEN_EXTRA[k]) - 1)} <= lsyms, 257 + k
    for c in range(30):
        assert {(c, 0), (c, (1 << D.DIST_EXTRA[c]) - 1)} <= dsyms, c
    assert (284, 31) in lsyms and 32768 in dists


def test_layouts_are_reached():
    recs = recs_of(*ALL)
    assert {r.start % 32 for _, _, r in recs if r.kind == "dynamic"} == set(range(32))
    assert any(i == 0 and r.kind == "dynamic" for _, i, r in recs)
    # a fixed block between dynamic ones; empty fixed blocks in the middle; stored blocks of LEN 0 and 65535
    assert any(0 < i < len(d.recs) - 1 and r.kind == "fixed" and d.recs[i - 1].kind == "dynamic" and d.recs[i + 1].kind == "dynamic"
               for d, i, r in recs)
    assert any(r.kind == "fixed" and r.out_len == 0 and not r.final for _, _, r in recs)
    assert {0, 65535} <= {r.out_len for _, _, r in recs if r.kind == "stored"}
    # stored blocks behind Huffman blocks that end at every residue of a stream word
    ends = {d.recs[i - 1].end % 32 for d, i, r in recs if r.kind == "stored" and i and d.recs[i - 1].kind != "stored"}
    assert ends == set(range(32))
    # empty final blocks of every kind; the shortest final dynamic block, ending in the last word before the Adler-32
    assert {"stored", "fixed", "dynamic"} <= {r.kind for _, _, r in recs if r.final and r.out_len == 0}
    assert any(r.final and r.kind == "dynamic" and (len(d.z) - 4) * 8 - r.end < 8 and r.end - r.start < 128 for d, _, r in recs)


def test_history_shapes_are_reached():
    recs = dyn("history")
    # sources straddling the block start with distance at most the length, a source at exactly the block's first byte
    straddle = {dist for _, i, r in recs if i for o, dist, L in r.match_srcs if o < dist <= L}
    assert {1, 2, 3, 31, 32, 33, 257, 258} <= straddle
    assert any(o == dist for _, i, r in recs if i for o, dist, _ in r.match_srcs)
    # blocks of exactly 32767 / 32768 / 32769 bytes, each followed by distance-32768 matches
    for n in (32767, 32768, 32769):
        assert any(r.out_len == n and any(dist == 32768 for _, dist, _ in d.recs[i + 1].match_srcs) for d, i, r in recs)
    # a distance-32768 match opening a block whose source is the first byte of the last 32 KiB of a longer block in front
    assert any(r.out_len > 32768 and (d.recs[i + 1].out_len, d.recs[i + 2].match_srcs[0][:2]) == (0, (0, 32768))
               for d, i, r in recs if i + 2 < len(d.recs))
    # k^2 - 1, k^2, k^2 + 1 blocks; in every such stream with groups beyond the first a mark at exactly a group start and
    # one in front of it, and a mark in front of every group start but the first (a chain through every group)
    by_nb = {d.n_blocks: d for d in D.corpus()["history"] if d.name.startswith("groups_")}
    for k in (2, 3, 5, 8):
        for nb in (k * k - 1, k * k, k * k + 1):
            d = by_nb[nb]
            per = D.group_size(nb)
            starts = [r.out_off for r in d.recs]
            gs_hits, gs1_hits, crossing = set(), set(), set()
            for i, r in enumerate(d.recs):
                g0 = starts[(i // per) * per]
                for o, dist, L in r.match_srcs:
                    if o >= dist:
                        continue   # inside the block: no mark
                    src = r.out_off + o - dist
                    gs_hits |= {i // per} if src == g0 and i % per else set()
                    gs1_hits |= {i // per} if src == g0 - 1 and i % per else set()
                    if src < g0:
                        crossing.add(i // per)
            ng = (nb + per - 1) // per
            assert set(range(1, ng)) <= crossing, (nb, crossing)
            assert set(range(ng)) - {ng - 1 if nb % per == 1 else ng} <= gs_hits, (nb, gs_hits)   # groups of 2+ blocks
            assert set(range(1, ng)) - {ng - 1 if nb % per == 1 else ng} <= gs1_hits, (nb, gs1_hits)
    assert {1, 2, 3} <= {d.n_blocks for d in D.corpus()["history"]}


def test_named_declines_sit_at_the_limits():
    c = {d.name: d for d in D.corpus()["declines"]}
    n = [r.n_tokens + 1 for r in c["max_syms_exact"].recs if r.kind == "dynamic"]
    assert n == [D.MAX_SYMS]
    assert [r.n_tokens + 1 for r in c["max_syms_plus1"].recs if r.kind == "dynamic"] == [D.MAX_SYMS + 1]
    for name, bits in (("host_budget_under", D.HOST_BUDGET), ("host_budget_over", D.HOST_BUDGET + 1)):
        r = c[name].recs[0]
        assert r.kind == "fixed" and r.end - r.start == bits and c[name].recs[1].kind == "fixed"
    for name, over in (("blocks_at_cap", 0), ("blocks_over_cap", 1)):
        d = c[name]
        assert d.n_blocks == D.cap_blocks(len(d.z), len(d.data)) + over
    d = c["distance_beyond_cinfo_window"]
    assert d.z[0] >> 4 == 0 and max(dist for _, dist, _ in d.recs[0].match_srcs) > 256


@pytest.mark.parametrize("design", D.all_designs(), ids=lambda d: d.name)
def test_host_model_equals_cv2_and_finds_every_dynamic_block(host_decode, design):
    """The host model decodes what cv2 decodes (declining only the shapes it declines on purpose), and every dynamic block
    is a candidate of its search: the chain walk measures only the stored and fixed blocks (stats[3])."""
    ref = cv2_decode(design.png)
    rc, out, stats = host_decode(design.png)
    if design.expect == "invalid":
        assert ref is None and rc == -6
        return
    if design.expect in HOST_DECLINES:
        assert rc == -6
        return
    assert ref is not None
    assert rc == 0 and np.array_equal(out, ref), (rc, stats)
    n_quick, n_cand, n_blocks, n_host = stats
    assert n_blocks == design.n_blocks
    assert n_host == sum(r.kind != "dynamic" for r in design.recs)
    if design.name.startswith("decoys_cand"):
        cap = D.cap_cand(len(design.z))
        assert (0.85 * cap < n_cand <= cap) if design.expect == "decode" else (cap < n_cand < 1.3 * cap), (n_cand, cap)
    if design.name.startswith("decoys_list"):
        cap = D.cap_list(len(design.z))
        assert (0.85 * cap < n_quick <= cap) if design.expect == "decode" else (cap < n_quick < 1.3 * cap), (n_quick, cap)
    if design.name.startswith("decoy") and not design.name.startswith("decoys_list"):
        assert n_cand > sum(r.kind == "dynamic" for r in design.recs)   # the false candidates are there


def test_decoys_measure_as_designed():
    """Every false candidate placed on purpose, measured by a one-block inflate the way the decoder measures a candidate:
    'block' decoys end at an end-of-block (a different block), 'bad' ones at a code the tree does not have, the 'long' one
    after 2^20 symbols without end-of-block (PD_LONG).  The decoys between true blocks sit at every residue of a stream
    word.  The same inflate gives every true dynamic block of the small designs its recorded end and length."""
    want = {"block": "ok", "bad": "bad", "long": "long"}
    kinds = set()
    for d in D.corpus()["decoys"]:
        bits = D.stream_bits(d.z)
        for bit, kind in d.decoys:
            assert D.measure(bits, bit, len(d.data))[0] == want[kind], (d.name, bit, kind)
            kinds.add(kind)
    assert kinds == set(want)
    every = next(d for d in D.corpus()["decoys"] if d.name == "decoys_every_shift")
    assert {bit % 32 for bit, _ in every.decoys} == set(range(32))
    for d in D.all_designs():
        if d.expect != "decode" or len(d.z) > 200000:
            continue
        bits = D.stream_bits(d.z)
        for r in d.recs:
            if r.kind == "dynamic":
                assert D.measure(bits, r.start, len(d.data), 256 << (d.z[0] >> 4)) == ("ok", r.end, r.out_len), d.name
