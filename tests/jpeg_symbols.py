"""Seeded BGR images whose JPEG files reach named paths of the device JPEG encoder (csrc/p2p_jpeg.cuh), and a counter of
what a file actually reaches.

The encoder's rare paths sit in the entropy coder and the byte stuffing, not in the pixels: DC categories up to 11 (a
quantiser of 1 and a jump of >= 128 in block mean), all 160 AC (run, size) symbols of both tables (sizes 9 and 10 need a
quantiser of 1 or 2), chains of ZRL codes, a non-zero coefficient at zig-zag 63 (no EOB), the 1-bit padding of the last
byte completing an 0xFF, 0xFF at every byte of the stuffing kernel's 16-byte chunks, and blocks starting at every bit of
the emit kernel's 32-bit words.  Noise, smooth and flat images leave most of these to chance; the builders below aim at
each one.

* ``corpus()``: ``(name, bgr, quality)`` items.  Symbol images are 128 x 128 (8 x 8 MCUs): one target per 8 x 8 block,
  everything else flat gray.  A luma target is a gray block (B = G = R gives Y exactly and Cb = Cr = 128); a chroma
  target varies Cb (or Cr) over 2 x 2-constant pixels whose other chroma stays exactly 128.  The block is the inverse
  DCT of the wanted quantised coefficients, rounded with a seeded dither until the exact integer model
  (``oracle/jpeg_model.py``) quantises it to the wanted symbol.
* ``file_stats(data)``: what a file reaches - taken from the coefficients ``oracle/jpeg_decode_model.py`` decodes out of
  the file, not from what a builder intended.
* ``targets()`` / ``reached(stats)``: the named targets; a corpus covers them when the union of ``reached`` over its
  files (encoded by ``cv2.imencode`` at their qualities) contains ``targets()``.
"""
from __future__ import annotations

import functools
from collections import Counter

import cv2
import numpy as np

from oracle import jpeg_decode_model as jd
from oracle import jpeg_model as jm

SIZE = 128            # symbol images: SIZE x SIZE pixels, 8 x 8 MCUs
QUALITIES = (50, 75, 90, 100)   # tried in this order for an AC target: the largest quantiser that reaches it
CHUNK = 16            # bytes per thread of jpeg_ffcount_kernel / jpeg_stuff_kernel
WORD = 32             # bits per word of the emit kernel's bit string


# ---- what a file reaches ---------------------------------------------------------------------------------------------
def _code_lengths():
    return ([jm.derive_codes(*jm.DC_LUMA)[1], jm.derive_codes(*jm.DC_CHROMA)[1]],
            [jm.derive_codes(*jm.AC_LUMA)[1], jm.derive_codes(*jm.AC_CHROMA)[1]])


def _nbits(v) -> int:
    return int(abs(int(v))).bit_length()


def file_stats(data: bytes) -> dict:
    """Symbols, block bit lengths / offsets and the unstuffed scan bytes of a baseline 4:2:0 file (cv2's layout)."""
    p = jd.parse(data)
    planes, (mcux, mcuy, _, _) = jd.entropy_decode(p)
    W, H = p["frame"]["W"], p["frame"]["H"]
    ybw, ybh = (W + 7) // 8, (H + 7) // 8
    dc_len, ac_len = _code_lengths()
    st = dict(dc=[Counter(), Counter()], ac=[Counter(), Counter()], zrl=[0, 0], eob=[0, 0], chains=[Counter(), Counter()],
              runs=[Counter(), Counter()], z63=[Counter(), Counter()], dc_only=[0, 0], dummy_after_dc11=0, bits=[])
    pred, prev_cat = [0, 0, 0], None
    for my in range(mcuy):
        for mx in range(mcux):
            for ci, (h, v) in enumerate(((2, 2), (1, 1), (1, 1))):
                t = min(ci, 1)
                for yi in range(v):
                    for xi in range(h):
                        by, bx = my * v + yi, mx * h + xi
                        zz = planes[ci][by, bx][jm.ZIGZAG]
                        diff = int(zz[0]) - pred[ci]
                        pred[ci] = int(zz[0])
                        cat = _nbits(diff)
                        st["dc"][t][(cat, int(np.sign(diff)))] += 1
                        if ci == 0:
                            if not (bx < ybw and by < ybh) and prev_cat == 11:
                                st["dummy_after_dc11"] += 1
                            prev_cat = cat
                        nbit = int(dc_len[t][cat]) + cat
                        run, last_nz = 0, 0
                        for k in range(1, 64):
                            c = int(zz[k])
                            if c == 0:
                                run += 1
                                continue
                            s = _nbits(c)
                            if run >= 16:
                                st["chains"][t][run // 16] += 1
                                st["zrl"][t] += run // 16
                                nbit += (run // 16) * int(ac_len[t][0xF0])
                            st["runs"][t][run] += 1
                            st["ac"][t][(run & 15, s, 1 if c > 0 else -1)] += 1
                            nbit += int(ac_len[t][((run & 15) << 4) | s]) + s
                            if k == 63:
                                st["z63"][t]["after_zrl" if run >= 16 else ("after_62" if run == 0 else "other")] += 1
                            run, last_nz = 0, k
                        if run:
                            st["eob"][t] += 1
                            nbit += int(ac_len[t][0])
                        if last_nz == 0:
                            st["dc_only"][t] += 1
                        st["bits"].append(nbit)
    bits = np.array(st["bits"], np.int64)
    st["offsets"] = np.concatenate([[0], np.cumsum(bits)[:-1]])
    st["total_bits"] = int(bits.sum())
    ecs = bytes(p["ecs"])
    assert ecs.endswith(b"\xff\xd9")
    scan = ecs[:-2].replace(b"\xff\x00", b"\xff")
    assert len(scan) == (st["total_bits"] + 7) // 8, "decoded bit count does not match the scan length"
    st["scan"] = scan
    return st


# ---- named targets ---------------------------------------------------------------------------------------------------
def _sgn(s: int) -> str:
    return "+" if s > 0 else "-"


def targets() -> set:
    out = {"dc0/dummy_after_cat11"}
    for t in (0, 1):
        out.add(f"dc{t}/cat0")
        out |= {f"dc{t}/cat{c}{_sgn(s)}" for c in range(1, 12) for s in (1, -1)}
        out |= {f"ac{t}/r{r}s{s}{_sgn(g)}" for r in range(16) for s in range(1, 11) for g in (1, -1)}
        out |= {f"ac{t}/zrl", f"ac{t}/eob", f"ac{t}/dc_only", f"ac{t}/z63_after_zrl", f"ac{t}/z63_after_62"}
        out |= {f"ac{t}/zrl_chain{k}" for k in (1, 2, 3)} | {f"ac{t}/run{16 * k}" for k in (1, 2, 3)}
    out |= {"stuff/pad_completes_ff", "stuff/no_padding", "stuff/len_mult32", "stuff/ff_run_across_chunk"}
    out |= {f"stuff/ff_at_{i}" for i in range(CHUNK)}
    out |= {f"sink/offset{i}" for i in range(WORD)} | {"sink/5_blocks_one_word"}
    return out


def reached(st: dict) -> set:
    out = set()
    if st["dummy_after_dc11"]:
        out.add("dc0/dummy_after_cat11")
    for t in (0, 1):
        out |= {f"dc{t}/cat{c}" + (_sgn(s) if c else "") for (c, s) in st["dc"][t]}
        out |= {f"ac{t}/r{r}s{s}{_sgn(g)}" for (r, s, g) in st["ac"][t]}
        for name, hit in (("zrl", st["zrl"][t]), ("eob", st["eob"][t]), ("dc_only", st["dc_only"][t]),
                          ("z63_after_zrl", st["z63"][t]["after_zrl"]), ("z63_after_62", st["z63"][t]["after_62"])):
            if hit:
                out.add(f"ac{t}/{name}")
        out |= {f"ac{t}/zrl_chain{k}" for k in st["chains"][t]}
        out |= {f"ac{t}/run{r}" for r in st["runs"][t] if r in (16, 32, 48)}
    tb, scan = st["total_bits"], st["scan"]
    if tb % 8 and scan[-1] == 0xFF:
        out.add("stuff/pad_completes_ff")
    if tb % 8 == 0:
        out.add("stuff/no_padding")
    if tb % 32 == 0:
        out.add("stuff/len_mult32")
    a = np.frombuffer(scan, np.uint8)
    ff = np.flatnonzero(a == 0xFF)
    out |= {f"stuff/ff_at_{i}" for i in set((ff % CHUNK).tolist())}
    if np.any((a[CHUNK - 1:-1:CHUNK] == 0xFF) & (a[CHUNK::CHUNK] == 0xFF)):
        out.add("stuff/ff_run_across_chunk")
    bits, offs = np.array(st["bits"]), st["offsets"]
    out |= {f"sink/offset{i}" for i in set((offs[bits >= 20] % WORD).tolist())}
    first, last = offs // WORD, (offs + bits - 1) // WORD
    per_word = np.bincount(np.concatenate([np.arange(f, l + 1) for f, l in zip(first, last)]))
    if per_word.max() >= 5:
        out.add("sink/5_blocks_one_word")
    return out


def cv2_jpeg(img: np.ndarray, quality: int) -> bytes:
    return cv2.imencode(".jpg", img, [cv2.IMWRITE_JPEG_QUALITY, int(quality)])[1].tobytes()


# ---- symbol blocks ---------------------------------------------------------------------------------------------------
def _basis() -> np.ndarray:
    """orthonormal 8 x 8 DCT basis by zig-zag position: the islow FDCT of basis k, divided by 8, is ~ 1 at k"""
    c = np.array([np.sqrt(0.125 if u == 0 else 0.25) * np.cos((2 * np.arange(8) + 1) * u * np.pi / 16) for u in range(8)])
    nat = np.einsum("ui,vj->uvij", c, c).reshape(64, 8, 8)   # natural index = vertical * 8 + horizontal frequency
    return nat[jm.ZIGZAG]


BASIS = _basis()


@functools.lru_cache(maxsize=None)
def _chroma_luts():
    """colour per Cb value with Cr == 128 exactly, per Cr value with Cb == 128, and per Cb value with any Cr"""
    v = np.arange(256)
    g, b = (a.ravel() for a in np.meshgrid(v, v, indexing="ij"))
    lut_cb, lut_cr, lut_any = {}, {}, {}
    for r in range(256):
        cb = (-11059 * r - 21709 * g + 32768 * b + (128 << 16) + 32767) >> 16
        cr = (32768 * r - 27439 * g - 5329 * b + (128 << 16) + 32767) >> 16
        for lut, sel, key in ((lut_cb, cr == 128, cb), (lut_cr, cb == 128, cr), (lut_any, np.ones_like(cb, bool), cb)):
            for k, i in zip(key[sel][::-1], np.flatnonzero(sel)[::-1]):
                lut[int(k)] = (int(b[i]), int(g[i]), r)
    return lut_cb, lut_cr, lut_any


def _lut_array(lut: dict) -> np.ndarray:
    a = np.zeros((256, 3), np.uint8)
    for k, c in lut.items():
        a[k] = c
    return a


def _search(coefs: dict, q: np.ndarray, lo: int, hi: int, check, rng, rounds: int = 6, batch: int = 128):
    """An integer 8 x 8 block in [lo, hi] (level-shifted) whose exact quantised coefficients (zig-zag) pass check, or
    None.  Start: the inverse DCT of the wanted quantised coefficients; rounding: seeded dither."""
    base = sum(v * float(q[jm.ZIGZAG[k]]) * BASIS[k] for k, v in coefs.items())
    if base.max() > hi - 0.5 or base.min() < lo + 0.5:
        return None
    for _ in range(rounds):
        P = np.clip(np.floor(base + rng.random((batch, 8, 8))), lo, hi).astype(np.int64)
        zz = jm.quantise(jm.fdct_islow(P), q).reshape(batch, 64)[:, jm.ZIGZAG]
        ok = check(zz)
        if ok.any():
            return P[int(np.argmax(ok))]
    return None


def _size_ok(col: np.ndarray, s: int, sign: int) -> np.ndarray:
    a = np.abs(col)
    return (a >= (1 << (s - 1))) & (a < (1 << s)) & (np.sign(col) == sign)


def _ac_block(t: int, run: int, s: int, sign: int, rng, at63: bool = False, tail62: bool = False):
    """(quality, block) with the AC symbol (run % 16, s) at a coefficient preceded by exactly `run` zeros (ZRLs for
    run >= 16); the coefficient before the run, if any, is non-zero.  at63: the target sits at zig-zag 63; tail62: a
    block with non-zero coefficients at zig-zag 62 and 63."""
    lo, hi = (-128, 127) if t == 0 else (7 - 128, 249 - 128)
    base = jm.STD_LUMA_Q if t == 0 else jm.STD_CHROMA_Q
    for quality in QUALITIES:
        q = jm.quant_table(base, quality)
        cands = [63] if at63 or tail62 else list(rng.permutation(np.arange(run + 1, 64)))[:24]
        for pos in cands:
            prev = pos - run - 1
            if tail62:
                prev = 62
            mag = (1 << (s - 1)) + min(2, (1 << (s - 1)) // 2)   # a margin for the rounding noise at quantiser 1
            coefs = {pos: sign * mag}
            if prev >= 1:
                coefs[prev] = int(rng.choice([-1, 1])) * (1 if q[jm.ZIGZAG[prev]] >= 8 else 3)

            def check(zz, pos=pos, prev=prev):
                ok = _size_ok(zz[:, pos], s, sign) & (zz[:, prev + 1:pos] == 0).all(1)
                return ok & (zz[:, prev] != 0) if prev >= 1 else ok

            blk = _search(coefs, q, lo, hi, check, rng)
            if blk is not None:
                return quality, blk
    raise RuntimeError(f"no block for table {t} run {run} size {s} sign {sign}")


def _ac_targets(t: int):
    """(name, run, size, sign, at63, tail62) of every AC target of table t that needs a designed block"""
    out = [(f"r{r}s{s}{_sgn(g)}", r, s, g, False, False) for r in range(16) for s in range(1, 11) for g in (1, -1)]
    out += [(f"run{16 * k}", 16 * k, 2, 1, False, False) for k in (1, 2, 3)]
    out += [("z63_after_zrl", 20, 3, -1, True, False), ("z63_after_62", 0, 2, 1, False, True)]
    return out


def _place_luma(blocks: list) -> np.ndarray:
    """gray image; block i at luma block position i in MCU scan order (4 per MCU)"""
    y = np.full((SIZE, SIZE), 128, np.int64)
    per_row = SIZE // 16
    for i, blk in enumerate(blocks):
        m, k = divmod(i, 4)
        oy, ox = (m // per_row) * 16 + (k >> 1) * 8, (m % per_row) * 16 + (k & 1) * 8
        y[oy:oy + 8, ox:ox + 8] = blk + 128
    return np.repeat(y.astype(np.uint8)[..., None], 3, axis=2)


def _place_chroma(blocks: list, luts: list) -> np.ndarray:
    """one chroma block per MCU (Cb or Cr per lut), each chroma sample on 2 x 2 equal pixels; the rest gray"""
    img = np.full((SIZE, SIZE, 3), 128, np.uint8)
    per_row = SIZE // 16
    for m, (blk, lut) in enumerate(zip(blocks, luts)):
        px = np.repeat(np.repeat(lut[blk + 128], 2, axis=0), 2, axis=1)
        oy, ox = (m // per_row) * 16, (m % per_row) * 16
        img[oy:oy + 16, ox:ox + 16] = px
    return img


def _ac_images(rng) -> list:
    lut_cb, lut_cr, _ = (_lut_array(x) for x in _chroma_luts())
    out = []
    for t in (0, 1):
        by_q: dict = {}
        for i, (_, run, s, g, at63, tail62) in enumerate(_ac_targets(t)):
            quality, blk = _ac_block(t, run, s, g, rng, at63, tail62)
            by_q.setdefault(quality, []).append((blk, lut_cb if i % 2 == 0 else lut_cr))
        cap = (SIZE // 16) ** 2 * (4 if t == 0 else 1)
        for quality in sorted(by_q):
            items = by_q[quality]
            for j in range(0, len(items), cap):
                part = items[j:j + cap]
                img = _place_luma([b for b, _ in part]) if t == 0 else _place_chroma([b for b, _ in part], [l for _, l in part])
                out.append((f"ac{t}-q{quality}-{j // cap}", img, quality))
    return out


# ---- DC differences --------------------------------------------------------------------------------------------------
def _dc_sequence(rng) -> list:
    """DC values (quantiser 1: DC = sum of the 64 level-shifted samples / 8) whose differences take every category
    0 .. 11 with both signs: each target is a pair (from, to), from the end of the range that leaves room."""
    seq = [0, 0]
    for c in range(1, 12):
        for sign in (1, -1):
            m = int(min(rng.integers(1 << (c - 1), 1 << c), 2040))
            start = -1024 if sign > 0 else 1016
            seq += [start, start + sign * m]
    return seq


def _dc_block(dc: int) -> np.ndarray:
    """level-shifted 8 x 8 block with sum 8 * dc, samples as equal as possible"""
    s = 8 * dc
    a, rem = divmod(s, 64)
    blk = np.full(64, a, np.int64)
    blk[:rem] += 1
    return blk.reshape(8, 8)


def _dc_images(rng) -> list:
    _, _, lut_any = _chroma_luts()
    luma = _place_luma([_dc_block(d) for d in _dc_sequence(rng)])
    lut = _lut_array(lut_any)
    chroma = _place_chroma([_dc_block(d) for d in _dc_sequence(rng)], [lut] * 64)
    out = [("dc0-q100", luma, 100), ("dc1-q100", chroma, 100)]
    # dummy luma blocks (W % 16, H % 16 in 1 .. 8) after real blocks that jump by the whole range: black / white 8 x 8
    # blocks at random
    for k, (w, h) in enumerate([(33, 40), (56, 17), (21, 29), (44, 52), (79, 36)]):
        cells = rng.integers(0, 2, ((h + 7) // 8, (w + 7) // 8)) * 255
        img = np.repeat(np.repeat(cells, 8, axis=0), 8, axis=1)[:h, :w].astype(np.uint8)
        out.append((f"dc-edge{k}-{w}x{h}", np.repeat(img[..., None], 3, axis=2), 100 - k % 3))
    return out


# ---- stuffing and bit sink -------------------------------------------------------------------------------------------
def _random_image(rng, w: int, h: int) -> np.ndarray:
    kind = int(rng.integers(0, 3))
    if kind == 0:
        return rng.integers(0, 256, (h, w, 3), dtype=np.uint8)
    if kind == 1:
        return (rng.integers(0, 2, (h, w, 3)) * 255).astype(np.uint8)
    cells = rng.integers(0, 256, ((h + 3) // 4, (w + 3) // 4, 3))
    return np.repeat(np.repeat(cells, 4, axis=0), 4, axis=1)[:h, :w].astype(np.uint8)


def _stream_images(rng) -> list:
    """Flat and saturated images, then a seeded search over small random images (up to 23 x 23, any quality) for the
    stuffing / bit-sink targets they do not reach yet."""
    flat = np.full((SIZE, SIZE, 3), 128, np.uint8)
    sat = (rng.integers(0, 2, (SIZE, SIZE, 3)) * 255).astype(np.uint8)
    out = [("flat-gray", flat, 95), ("saturated-noise", sat, 100)]
    want = {t for t in targets() if t.startswith(("stuff/", "sink/"))}
    for _, img, q in out:
        want -= reached(file_stats(cv2_jpeg(img, q)))
    for i in range(5000):
        if not want:
            break
        w, h = (int(x) for x in rng.integers(1, 24, 2))
        img, q = _random_image(rng, w, h), int(rng.integers(1, 101))
        data = cv2_jpeg(img, q)
        if want == {"stuff/pad_completes_ff"} and data[-4:-2] != b"\xff\x00":
            continue        # only a file ending FF 00 FF D9 can reach it: skip the decode
        hit = reached(file_stats(data)) & want
        if hit:
            out.append((f"search{i}-{w}x{h}", img, q))
            want -= hit
    return out


@functools.lru_cache(maxsize=None)
def corpus() -> tuple:
    """((name, bgr, quality), ...): fixed seeds, the same images on every call."""
    rng = np.random.default_rng(20261022)
    return tuple(_ac_images(rng) + _dc_images(rng) + _stream_images(rng))
