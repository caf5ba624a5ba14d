"""Designed inputs for the PNG encoder (test-only).

OpenCV writes every row with filter Sub (type 0 for images one pixel wide), so the deflate input of a BGR image is a byte
string F of rows ``filter byte | 3 W filtered bytes``.  ``image_from_filtered`` inverts the filter: it turns a chosen F
into the image whose ``png_model.sub_filter`` is exactly F, so a test chooses the deflate input directly - literal
frequencies, runs, block fills - instead of hoping that ordinary images reach a path of zlib's deflate_rle / trees.c.

``corpus()`` yields the designed images by family.  Which paths they reach is not taken on trust: the tests read it from
``png_model.deflate_rle``'s per-block records (``stats``) and from the runs of F (``runs``).
"""
import numpy as np

from oracle import png_model as pm

TILE = 4096        # the device tokeniser's tile (p2p_png.cuh kTile) and its look-ahead of 18 x 16 bytes (kLookThreads)
LOOK = 288
SYM_PER_BLOCK = 16383


def filter_byte(W):
    return 0 if W == 1 else 1


def image_from_filtered(F, W):
    """The BGR image whose Sub-filtered rows are F (bytes or uint8 array of H rows of 1 + 3 W bytes): per channel the
    cumulative sum mod 256 along the row, channels in RGB order."""
    F = np.frombuffer(bytes(F), np.uint8) if not isinstance(F, np.ndarray) else F.reshape(-1)
    rows = F.reshape(-1, 1 + 3 * W)
    assert (rows[:, 0] == filter_byte(W)).all(), "every row starts with the filter byte OpenCV writes"
    d = rows[:, 1:].reshape(-1, W, 3).astype(np.int64)
    rgb = (np.cumsum(d, axis=1) & 255).astype(np.uint8)
    img = np.ascontiguousarray(rgb[..., ::-1])
    assert pm.sub_filter(img) == rows.tobytes()
    return img


def background(H, W, seed):
    """F of H rows with no two equal neighbours: pixel bytes in 2 .. 255 (a random walk with steps 1 .. 253 mod 254), the
    filter bytes 0 / 1, so the tokeniser sees literals only."""
    rng = np.random.default_rng(seed)
    steps = rng.integers(1, 254, H * 3 * W)
    px = (2 + np.cumsum(steps) % 254).astype(np.uint8).reshape(H, 3 * W)
    F = np.empty((H, 1 + 3 * W), np.uint8)
    F[:, 0] = filter_byte(W)
    F[:, 1:] = px
    return F.reshape(-1)


def runs(F, min_len=2):
    """(start, end) of the maximal runs of equal bytes of F with at least ``min_len`` bytes."""
    F = np.asarray(F).reshape(-1)
    chg = np.flatnonzero(F[1:] != F[:-1]) + 1
    starts = np.concatenate([[0], chg])
    ends = np.concatenate([chg, [len(F)]])
    keep = ends - starts >= min_len
    return list(zip(starts[keep].tolist(), ends[keep].tolist()))


def fill_row(payload, W=None):
    """One row: the filter byte, then ``payload`` (its length is 3 W)."""
    payload = np.asarray(payload, np.uint8)
    W = len(payload) // 3 if W is None else W
    assert len(payload) == 3 * W
    return np.concatenate([[filter_byte(W)], payload]).astype(np.uint8), W


def _arrange(units, rng):
    """Concatenate byte units (arrays of one repeated byte) so that no two neighbouring units share their byte: the units
    grouped by byte, the largest group first (shuffled inside each group), fill the even places, then the odd ones.  That
    works while no byte has more than half of the units."""
    by = {}
    for u in units:
        by.setdefault(int(u[0]), []).append(u)
    groups = sorted(by.values(), key=len, reverse=True)
    assert 2 * len(groups[0]) <= len(units) + 1
    seq = []
    for g in groups:
        seq += [g[i] for i in rng.permutation(len(g))]
    order = [None] * len(seq)
    places = list(range(0, len(seq), 2)) + list(range(1, len(seq), 2))
    for p, u in zip(places, seq):
        order[p] = u
    out = np.concatenate(order)
    assert all(a[-1] != b[0] for a, b in zip(order, order[1:]))
    return out


def fib(n):
    f = [1, 2]
    while len(f) < n:
        f.append(f[-1] + f[-2])
    return f[:n]


def chain_row(n_values, seed, lengths=()):
    """A one-row F whose literal / length frequencies are a Fibonacci chain: END_BLOCK 1, the filter byte 1 (1 time), and
    n_values - 1 further symbols with frequencies 2, 3, 5, 8, ...  ``lengths``: match lengths whose length symbols take
    the lowest places of the chain (each such match is a run of the most frequent literal, which pays for the run's
    first byte).  No two neighbouring units share a byte, so there are no other runs."""
    rng = np.random.default_rng(seed)
    freqs = fib(n_values)[1:]                 # 2, 3, 5, ...: the chain above the filter byte
    values = [v for v in range(2, 256) if v != 0][: len(freqs)]
    top = values[-1]
    units = []
    for L, f in zip(lengths, freqs):
        units += [np.full(L + 1, top, np.uint8)] * f
    n_top = freqs[-1] - sum(f for _, f in zip(lengths, freqs))
    n_top += -(sum(freqs) + sum((L - 1) * f for L, f in zip(lengths, freqs))) % 3   # 3 W bytes: the top leaf takes the slack
    for v, f in list(zip(values, freqs))[len(lengths):]:
        units += [np.array([v], np.uint8)] * (n_top if v == top else f)
    payload = _arrange(units, rng)
    return fill_row(payload)


def deflate_records(F):
    stats = []
    z, _ = pm.deflate_rle(bytes(np.asarray(F).reshape(-1)), stats=stats)
    return z, stats


def with_runs(H, W, seed, spans):
    """background(H, W) with the byte ranges ``spans`` [(start, end)] set to the filter byte, so that a run crosses rows
    unbroken (the filter bytes it covers are part of it); a run next to a row start grows by that filter byte."""
    F = background(H, W, seed)
    for s, e in spans:
        F[s:e] = filter_byte(W)
    return F


def static_units():
    """Literals 0 .. 255 once each and one match of every length code 257 .. 285 (the longest length of each code, and
    258 besides 257), each match a run of its own byte: flat statistics that zlib sends with the fixed codes."""
    lengths = [pm.base_length[c] + 3 + (1 << pm.extra_lbits[c]) - 1 for c in range(28)] + [258, 257, 3]
    units = [np.array([v], np.uint8) for v in range(256) if v != 1]
    units += [np.full(L + 1, 2 + k, np.uint8) for k, L in enumerate(lengths)]
    return units


def corpus():
    """(family, name, W, F) of every designed stream."""
    out = []

    def add(family, name, F, W):
        assert W < 32767 and len(F) // (1 + 3 * W) < 32767      # the encoder's size limit
        out.append((family, name, W, np.asarray(F, np.uint8).reshape(-1)))

    # literal / length tree deeper than 15 bits: Fibonacci chains, with match-length symbols among the deep leaves
    for n in (16, 17, 18):
        add("lit_overflow", f"chain{n}", *chain_row(n, n))
        add("lit_overflow", f"chain{n}_lengths", *chain_row(n, n, (258, 3, 130, 227)))
        add("lit_overflow", f"chain{n}_all_lengths", *chain_row(n, n, (258, 257, 227, 131, 67, 35, 17, 11, 10, 4, 3)))
    # bit-length tree deeper than 7 bits: blocky content (8 x 8 blocks of random colours) whose code-length profile has it
    rng = np.random.default_rng(0)
    h, w = 265, 283
    img = np.repeat(np.repeat(rng.integers(0, 256, ((h + 7) // 8, (w + 7) // 8, 3), dtype=np.uint8), 8, 0), 8, 1)[:h, :w]
    add("bl_overflow", "blocky", np.frombuffer(pm.sub_filter(np.ascontiguousarray(img)), np.uint8), w)
    # fixed codes: the flat block alone, as a short last block behind a dynamic one, and tiny images
    rng = np.random.default_rng(1)
    flat = _arrange(static_units(), rng)
    flat = flat[: len(flat) - len(flat) % 3]
    add("static", "flat", *fill_row(flat))
    chain, _ = chain_row(18, 7)
    skew = np.concatenate([chain[1:], chain[1:]])[: 3 * ((len(chain) * 2 - 2) // 3)]     # > 16383 literals, dynamic
    tail = np.concatenate([skew, flat])
    tail = tail[: len(tail) - len(tail) % 3]
    add("static", "dynamic_then_flat", *fill_row(tail))
    for W, H in ((1, 1), (2, 1), (5, 3), (20, 2)):
        add("static", f"tiny{W}x{H}", background(H, W, W + H), W)
    # the largest tree description: literal and length frequencies spread over 2^0 .. 2^9.5, so the code lengths spread
    # over most of 1 .. 15 and vary between neighbouring symbols (few repeat codes)
    rng = np.random.default_rng(6)
    units = []
    for v, f in zip(range(2, 256), np.maximum(1, np.round(2.0 ** rng.uniform(0, 9.5, 254))).astype(int)):
        units += [np.array([v], np.uint8)] * int(f)
    lengths = [pm.base_length[c] + 3 for c in range(28)] + [258]
    for k, (L, f) in enumerate(zip(lengths, np.maximum(1, np.round(2.0 ** rng.uniform(0, 6, 29))).astype(int))):
        units += [np.full(L + 1, 2 + (k * 7) % 250, np.uint8)] * int(f)
    big = _arrange(units, rng)
    add("big_header", "spread_lengths", *fill_row(big[: len(big) - len(big) % 3]))
    # stored blocks: behind Huffman blocks ending at every bit residue, behind stored blocks, as the last block
    for k in range(16):
        rng = np.random.default_rng(100 + k)
        head = np.concatenate([chain[1 + 31 * k:], chain[1:]])[: 16383 + 3 + k]   # a dynamic block of 16383 literals ...
        noise = rng.integers(0, 256, 5000 + 3 * k, dtype=np.uint8)        # ... then white noise: a stored last block
        body = np.concatenate([head, noise])
        add("stored", f"after_huffman{k}", *fill_row(body[: len(body) - len(body) % 3]))
    for W, H in ((381, 14), (1000, 40), (7, 5)):
        add("stored", f"noise{W}x{H}", np.frombuffer(pm.sub_filter(np.random.default_rng(W).integers(0, 256, (H, W, 3), dtype=np.uint8)), np.uint8), W)
    # exact block fills: N = 16383 and 32766 run-free bytes (one token each, the last block empty), and N +- 1
    for W, H in ((14, 381), (42, 258), (2730, 2), (5, 1024), (1, 4096), (14, 382)):
        add("fill", f"runfree{W}x{H}", background(H, W, W * H), W)
    # ... and a block whose 16383rd token is a 258-byte match
    W = 10000
    add("fill", "match258_last", with_runs(2, W, 3, [(16381, 16381 + 259)]), W)
    # runs at the tokeniser's edges
    for r in range(4):                         # the whole image one run: (N - 1) mod 258 = r
        W, H = next((W, H) for W in range(2, 400) for H in range(1, 40) if (H * (1 + 3 * W) - 1) % 258 == r and H * (1 + 3 * W) > 300)
        add("runs", f"ramp{r}", np.full(H * (1 + 3 * W), 1, np.uint8), W)
    W, H = 3000, 120                           # runs over every residue of (j - 1) mod 258 at a tile boundary
    n_bound = (H * (1 + 3 * W)) // TILE - 1
    spans = []
    for k in range(1, min(n_bound, 259)):
        B, rho = k * TILE, (k - 1) % 258
        s = B - 1 - rho
        spans.append((s, B + 40 + (k * 13) % 600))
    add("runs", "tile_residues", with_runs(H, W, 5, spans), W)
    W, H = 3000, 19                            # run ends 0 .. 290 bytes behind a tile boundary, and long runs
    spans = []
    ends = [0, 1, 2, 255, 256, 257, 258, 259, 287, 288, 289, 290]
    for k, d in enumerate(ends, start=1):
        B = k * 2 * TILE
        spans.append((B - 600, B + d))
    # a chunk of the run starts at the tile's last byte (B - 1) and the run ends 250 .. 258 bytes behind the tile: that match's
    # length comes from the look-ahead's last bytes
    spans += [(B - 260, B + d) for B, d in zip(range(30 * TILE, 40 * TILE, TILE), (250, 254, 255, 256, 257, 258))]
    spans += [(26 * TILE - 3, 26 * TILE + 4096 + 400), (28 * TILE + 5, 28 * TILE + 9000)]
    spans += [(60000 + 50 * k, 60000 + 50 * k + L) for k, L in enumerate((2, 3, 4, 5, 6, 259, 260, 261, 516, 517))]
    F = with_runs(H, W, 6, spans)
    F[-300:] = 0                               # a run that ends at N
    add("runs", "tile_ends", F, W)
    W, H = 1, 3000                             # width 1: filter type 0, runs across rows
    add("runs", "width1", with_runs(H, W, 7, [(100, 2000), (4090, 4100), (8000, 8258 + 3)]), W)
    return out
