"""Seeded random Vorbis streams, an independent packet reader and a model of `after_residue` (test helper, not a conftest).

Generator: seeded tools/vorbis_writer.StreamSetup objects and PacketChoice lists over the whole legal space this build
decodes: 1 to 8 channels, every power-of-two block-size pair from 64 to 8192 (equal pairs included), up to 64 modes,
1 to 4 mappings with up to one submap per channel and coupling chains that share channels, floor1 with 2 to 250 posts,
multipliers 1 to 4, rangebits up to 15, classes of dimension 1 to 8 with 0 to 3 subclass bits and "no book" subclasses,
codebooks in the ordered, sparse and dense length forms with codewords of 1 to 32 bits (and books made of 9- and 10-bit
codewords only, the edge of the device's first-level lookup table), lookup types 1 and 2 with sequence_p, 1 to 16 value
bits and negative minima, a book of more than 65536 entries (32-bit entry numbers), residues of types 0, 1 and 2 whose
`begin` and `end` lie inside, at and past the decode length, partition sizes 1 to 256, classbooks of dimension 1 to 4,
2 to 64 classifications and 1 to 8 cascade passes with gaps. Packets have unused floors, all channels unused, and are
cut short at a random byte.

Reader: a plain-Python packet reader that follows Vorbis I §3.2.1 (Huffman codewords, built here with its own tree),
§4.3 (audio packet header), §7.2.3 (floor1 packet decode) and §8.6.2 (residue decode) straight from the packet bits.
Bits past the end of a packet read as zero, as in the reference decoder (Utils.hpp:389-392). It uses nothing of the
library under test or of the oracle.

Model: the expected `after_residue` of every channel from what the reader read: VQ tables expanded as the reference does
(double arithmetic rounded to float, `last` re-reading the rounded value), each bin summing its addends in float32 from
0 in pass order, type 0 placing vector element l of entry k at k + l*nvec, types 1 and 2 at k*dim + l, type 2
de-interleaved, the nonzero propagate applied first.

Two conventions are the reference decoder's rather than libvorbis': a type-2 submap is decoded even when all of its
channels are unused (hpp:688; libvorbis skips it), and the writer encodes the packets that way. Where several channels
share one type-0/1 submap the reader follows the specification and libvorbis (one partition counter for all channels),
not the reference (hpp:755), like the synth_shared_submap golden.
"""
from __future__ import annotations

import ctypes as C
import functools
import math
import os
import sys
from dataclasses import dataclass, field
from typing import Dict, List, Optional, Tuple

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if os.path.join(ROOT, "tools") not in sys.path:
    sys.path.insert(0, os.path.join(ROOT, "tools"))
import vorbis_writer as vw  # noqa: E402
from parseoggvorbis_b200 import abi, workloads  # noqa: E402

FLOOR_RANGE = {1: 256, 2: 128, 3: 86, 4: 64}
SEEDS = list(range(40))
# bins times channels coded per packet that a random stream aims at: keeps the pure-Python writer and reader fast
BIN_BUDGET = 60000


# =====================================================================================================================
# generator
# =====================================================================================================================
def _lengths(rng, n, form):
    """Codeword lengths of n entries: 'dense' / 'sparse' (some entries unused) / 'ordered' (non-decreasing, all used) /
    'deep' (skewed towards long codewords, up to 32 bits) / 'nine_ten' (9- and 10-bit codewords only)."""
    if form == "nine_ten":
        assert 512 < n <= 1024
        k = n - 512                         # split k of the 512 depth-9 leaves
        out = [9] * (512 - k) + [10] * (2 * k)
        rng.shuffle(out)
        return [int(x) for x in out]
    if form == "deep":
        return vw.full_tree_lengths(n, rng, skew=0.97, max_len=32)
    if form == "ordered":
        return sorted(vw.full_tree_lengths(n, rng, skew=float(rng.random()), max_len=32))
    if form == "sparse":
        used = rng.random(n) < 0.7
        used[:2] = True
        if used.sum() < 2:
            used[:] = True
        lens = iter(vw.full_tree_lengths(int(used.sum()), rng, skew=float(rng.random()) * 0.6, max_len=32))
        return [next(lens) if u else 0 for u in used]
    return vw.full_tree_lengths(n, rng, skew=float(rng.random()) * 0.6, max_len=32)


def scalar_book(rng, n, form="dense"):
    return vw.Book(1, _lengths(rng, n, form))


def vq_book(rng, dim, n=None, form=None, lookup_type=None, value_bits=None, sequence_p=None):
    """A VQ book of `dim` dimensions whose values stay small (|v| <= ~8): value_bits 1..16, a power-of-two delta, a
    negative minimum or a running sum (sequence_p)."""
    if n is None:
        n = int(rng.integers(2, 1 + min(64, 4 ** dim)))
    if form is None:
        form = str(rng.choice(["dense", "dense", "sparse", "ordered", "deep"]))
    if lookup_type is None:
        lookup_type = int(rng.integers(1, 3))
    if value_bits is None:
        value_bits = int(rng.integers(1, 17))
    if sequence_p is None:
        sequence_p = bool(rng.random() < 0.25)
    lengths = _lengths(rng, n, form)
    book = vw.Book(dim, lengths, lookup_type, value_bits=value_bits, sequence_p=sequence_p, ordered=(form == "ordered"))
    top = (1 << value_bits) - 1
    nv = book.lookup1_values() if lookup_type == 1 else n * dim
    book.multiplicands = [int(x) for x in rng.integers(0, top + 1, size=nv)]
    span = 1.0 / max(1, dim) if sequence_p else 2.0
    book.delta = 2.0 ** math.floor(math.log2(span / max(1, top)))     # top * delta <= span
    book.minimum = 0.0 if sequence_p else -float(int(rng.integers(0, 9))) * 0.125
    if sequence_p:
        book.minimum = -book.delta * float(int(rng.integers(0, max(1, top // 2) + 1)))
    return book


def make_floor(rng, books, n_posts, multiplier, rangebits, form_of_book=None):
    """A floor1 of n_posts posts: classes of dimension 1..8 with 0..3 subclass bits (a "no book" subclass in most of
    them); its Y books and masterbooks are appended to `books`."""
    R = FLOOR_RANGE[multiplier]
    left = n_posts - 2
    k = int(rng.integers(-(-left // 8), min(31, left) + 1)) if left else 0     # at most 31 partitions (5 bits)
    dims = [1] * k
    extra = left - k
    while extra:
        i = int(rng.integers(0, k))
        if dims[i] < 8:
            dims[i] += 1
            extra -= 1
    assert len(dims) <= 31 and all(1 <= d <= 8 for d in dims), dims
    n_ybooks = int(rng.integers(1, 3))
    ybooks = []
    for _ in range(n_ybooks):
        ybooks.append(len(books))
        books.append(scalar_book(rng, R, form_of_book or str(rng.choice(["dense", "ordered", "deep"]))))
    classes, class_of_dim = [], {}
    for d in sorted(set(dims)):
        sb = int(rng.integers(0, 4))
        while sb and (1 << (sb * d)) > 256:  # masterbook of (2^sb)^d entries
            sb -= 1
        if sb == 0:
            fc = vw.FloorClass(d, 0, 0, [int(rng.choice(ybooks))])
        else:
            master = len(books)
            books.append(scalar_book(rng, 1 << (sb * d), form_of_book or "dense"))
            sub = [int(rng.choice(ybooks)) for _ in range(1 << sb)]
            if rng.random() < 0.7:
                sub[int(rng.integers(0, len(sub)))] = -1
            if all(b < 0 for b in sub):
                sub[0] = ybooks[0]
            fc = vw.FloorClass(d, sb, master, sub)
        class_of_dim[d] = len(classes)
        classes.append(fc)
    # distinct X values: 0, 1 << rangebits, then n_posts - 2 others below 1 << rangebits
    top = 1 << rangebits
    tail = [int(x) for x in rng.choice(np.arange(1, top), size=n_posts - 2, replace=False)]
    return vw.Floor1([class_of_dim[d] for d in dims], classes, multiplier, rangebits, tail)


def make_residue(rng, books, vq_pool, rtype, begin, end, psize, n_class, cw, passes=None, full_class=False):
    """Residue with a classbook of n_class^cw entries; every class but 0 codes 1..8 passes (gaps allowed) with VQ books
    whose dimension divides the partition size (class 0 codes nothing). `passes`: force these passes on class 1.
    full_class: class 1 codes all 8 passes."""
    classbook = len(books)
    books.append(vw.Book(cw, _lengths(rng, n_class ** cw, str(rng.choice(["dense", "ordered", "deep"])))))
    cand = [b for b in vq_pool if psize % books[b].dim == 0]
    assert cand, "no VQ book divides the partition size"
    rows = [[-1] * 8]
    for c in range(1, n_class):
        row = [-1] * 8
        if full_class and c == 1:
            chosen = list(range(8))
        else:
            chosen = sorted(int(p) for p in rng.choice(8, size=int(rng.integers(1, 9)), replace=False))
        for p in chosen:
            row[p] = int(rng.choice(cand))
        rows.append(row)
    return vw.Residue(rtype, begin, end, psize, classbook, rows)


def choose_packet(rng, s, mode, prev_flag, next_flag, p_unused=0.15, dense=0.5, all_unused=False):
    """One packet's symbols: Y lists from workloads.gen_ys (audio-like curves), random classifications (class 0 with
    probability 1 - dense) and random used VQ entries. A type-2 submap with a channel that has neither a floor nor a
    coupling partner that has one codes class 0 throughout: such a channel takes its residue unscaled into the PCM
    (hpp:1247), so an encoder codes nothing for it, and the PCM stays audio-like."""
    mp = s.mappings[s.modes[mode].mapping]
    n = s.blocksize[s.modes[mode].blockflag]
    draw = rng.random(s.channels) >= p_unused
    if all_unused:
        draw[:] = False
    elif not workloads.closed_under_propagation(draw[None, :], mp.couplings)[0]:
        draw[:] = True
    ys = []
    for c in range(s.channels):
        fl = s.floors[mp.submap_floor[mp.mux[c]]]
        ys.append([int(v) for v in workloads.gen_ys(rng, 1, fl.xs, fl.multiplier)[0]] if draw[c] else None)
    prop = vw.propagate([y is not None for y in ys], mp.couplings)
    residue = []
    for sm in range(len(mp.submap_floor)):
        chs = [c for c in range(s.channels) if mp.mux[c] == sm]
        r = s.residues[mp.submap_residue[sm]]
        nch, dl = (1, len(chs) * (n // 2)) if r.type == 2 else (len(chs), n // 2)
        _, _, parts = vw.residue_geometry(r, dl)
        cls = np.where(rng.random((nch, parts)) < dense, rng.integers(1, r.n_class, size=(nch, parts)), 0)
        if r.type == 2 and not all(prop[c] for c in chs):
            cls[:] = 0
        entries = {}
        for pass_ in range(8):
            for p in range(parts):
                for j in range(nch):
                    b = r.books[int(cls[j][p])][pass_]
                    if b >= 0:
                        bk = s.books[b]
                        used = _used_entries(bk)
                        entries[(pass_, p, j)] = [int(used[k]) for k in rng.integers(0, len(used), size=r.partition_size // bk.dim)]
        residue.append((cls, entries))
    return vw.PacketChoice(mode, prev_flag, next_flag, ys, residue)


def _used_entries(book):
    u = getattr(book, "_used", None)
    if u is None:
        u = np.flatnonzero(np.asarray(book.lengths) > 0)
        book._used = u
    return u


def _block_flags(rng, P, modes):
    have = {m.blockflag for m in modes}
    if have == {0}:
        return [0] * P
    if have == {1}:
        return [1] * P
    pat = [0, 0, 1, 1, 0, 1, 0, 0, 0, 1, 1, 1]
    while len(pat) < P:
        pat.append(int(rng.random() < 0.6))
    return pat[:P]


def packets_for(rng, s, P, dense, p_unused=0.15, all_unused_every=0):
    modes_of = {f: [i for i, m in enumerate(s.modes) if m.blockflag == f] for f in (0, 1)}
    flags = _block_flags(rng, P, s.modes)
    out = []
    for i, f in enumerate(flags):
        prev_f = flags[i - 1] if i else 1
        next_f = flags[i + 1] if i + 1 < len(flags) else 1
        au = bool(all_unused_every) and i % all_unused_every == all_unused_every - 1
        out.append(choose_packet(rng, s, int(rng.choice(modes_of[f])), prev_f, next_f, p_unused, dense, au))
    return out


def _coded_bins(s, mode):
    """Bins times channels the residues of a mode can code: what a packet of it costs the Python writer and reader."""
    mp = s.mappings[s.modes[mode].mapping]
    half = s.blocksize[s.modes[mode].blockflag] // 2
    tot = 0
    for sm in range(len(mp.submap_floor)):
        nch = sum(1 for c in range(s.channels) if mp.mux[c] == sm)
        r = s.residues[mp.submap_residue[sm]]
        dl = nch * half if r.type == 2 else half
        lb, le, parts = vw.residue_geometry(r, dl)
        tot += parts * r.partition_size * (1 if r.type == 2 else nch)
    return tot


@dataclass
class Stream:
    name: str
    setup: vw.StreamSetup
    packets: List[vw.PacketChoice]
    data: bytes
    trim: int = 0
    expect_kernel: Optional[str] = None


def cut_some_packets(rng, s, packets, frac=0.1):
    """Cut about `frac` of the packets at a random byte after their floors (the floors stay whole, so the floor checks
    of hpp:536/587 cannot fire on zero-filled Ys; the residue reads zeros from the cut on)."""
    for pc in packets:
        if rng.random() >= frac:
            continue
        full = vw.write_audio_packet(s, pc)
        rp = read_packet(s, full)
        lo = (rp.floor_end_bit + 7) // 8
        if lo >= len(full):
            continue
        pc.truncate_bytes = int(rng.integers(max(1, lo), len(full)))


def random_stream(seed: int) -> Stream:
    rng = np.random.default_rng(1000 + seed)
    channels = int(rng.integers(1, 9))
    e0 = int(rng.integers(6, 14))
    e1 = int(rng.integers(e0, 14))
    if rng.random() < 0.35:                  # the common encoder pairs (and the warp kernel's)
        e0, e1 = [(8, 11), (8, 9), (8, 10), (9, 10), (9, 11), (10, 11)][int(rng.integers(0, 6))]
    bs = (1 << e0, 1 << e1)
    books: List[vw.Book] = []
    # VQ pool: dims 1..8 (1 and 2 always present so that every partition size has a book)
    vq_pool = []
    for dim in [1, 2] + [int(d) for d in rng.integers(1, 9, size=int(rng.integers(1, 5)))]:
        vq_pool.append(len(books))
        books.append(vq_book(rng, dim))
    if rng.random() < 0.2:                   # one book of 9- and 10-bit codewords only
        vq_pool.append(len(books))
        books.append(vq_book(rng, 1, n=int(rng.integers(513, 700)), form="nine_ten", lookup_type=1))
    # floors: small ones mostly (the warp kernel takes up to 64 posts), sometimes wide
    n_floors = int(rng.integers(1, 4))
    floors = []
    for _ in range(n_floors):
        wide = rng.random() < 0.2
        posts = int(rng.integers(65, 251)) if wide else int(rng.integers(2, 40))
        rb = int(rng.integers(max(vw.ilog(posts), e0 - 1), 16))
        floors.append(make_floor(rng, books, posts, int(rng.integers(1, 5)), rb))
    # residues
    n_res = int(rng.integers(1, 4))
    residues = []
    for _ in range(n_res):
        rtype = int(rng.integers(0, 3))
        dl = bs[1] // 2 * (channels if rtype == 2 else 1)
        psize = int(rng.choice([1, 2, 4, 8, 8, 16, 16, 32, 32, 64, 128, 256]))
        if rng.random() < 0.15:
            psize = int(rng.choice([3, 6, 12, 24, 48, 96]))
        u = rng.random()
        begin = 0 if u < 0.6 else int(rng.integers(0, dl + 64))
        v = rng.random()
        end = begin + int(rng.integers(0, dl + 1)) if v < 0.5 else (dl if v < 0.7 else dl + int(rng.integers(1, 5000)))
        end = max(begin, min(end, (1 << 24) - 1))           # begin <= end (hpp:638)
        cw = int(rng.integers(1, 5))
        n_class = int(rng.integers(2, 65))
        while n_class ** cw > 300:
            n_class = max(2, n_class // 2) if cw > 1 and n_class > 2 else n_class
            if n_class ** cw > 300:
                cw -= 1
        cand = [b for b in vq_pool if psize % books[b].dim == 0]
        if not cand:
            psize = 8
        residues.append(make_residue(rng, books, vq_pool, rtype, begin, end, psize, n_class, cw))
    # mappings: submaps up to one per channel, couplings sharing channels
    n_maps = int(rng.integers(1, 5))
    maps = []
    for _ in range(n_maps):
        ns = int(rng.integers(1, channels + 1)) if rng.random() < 0.5 else 1
        order = rng.permutation(channels)
        mux = [0] * channels
        for i, c in enumerate(order):
            mux[int(c)] = i if i < ns else int(rng.integers(0, ns))
        cp = []
        if channels > 1:
            for _ in range(int(rng.integers(0, min(8, 2 * channels)))):
                m, a = (int(x) for x in rng.choice(channels, size=2, replace=False))
                cp.append((m, a))
        maps.append(vw.Mapping(mux, [int(rng.integers(0, n_floors)) for _ in range(ns)],
                               [int(rng.integers(0, n_res)) for _ in range(ns)], cp))
    n_modes = int(rng.choice([1, 2, 2, 3, 4, 7, 16, 33, 64]))
    modes = [vw.Mode(int(rng.integers(0, 2)), int(rng.integers(0, n_maps))) for _ in range(n_modes)]
    modes[0].blockflag = 0
    if n_modes > 1:
        modes[1].blockflag = 1
    s = vw.StreamSetup(channels, int(rng.choice([8000, 22050, 44100, 48000])), bs, books, floors, residues, maps, modes)
    cost = max(1, max(_coded_bins(s, m) for m in range(n_modes)))
    P = int(np.clip(BIN_BUDGET // cost, 4, 60))
    pk = packets_for(rng, s, P, dense=float(rng.uniform(0.2, 0.9)), p_unused=float(rng.uniform(0, 0.4)),
                     all_unused_every=int(rng.choice([0, 0, 7])))
    cut_some_packets(rng, s, pk)
    trim = int(rng.integers(0, bs[0] // 4))
    return Stream("seed%d" % seed, s, pk, vw.write_stream(s, pk, serial=0x6000 + seed, packets_per_page=6, trim_last=trim), trim)


# ---- named edge streams ------------------------------------------------------------------------------------------------
def _simple(rng, name, channels, bs, books, floors, residues, maps, modes, P, dense=0.6, p_unused=0.1, cut=0.1,
            expect_kernel=None, seed=0):
    s = vw.StreamSetup(channels, 44100, bs, books, floors, residues, maps, modes)
    pk = packets_for(rng, s, P, dense, p_unused)
    if cut:
        cut_some_packets(rng, s, pk, cut)
    return Stream(name, s, pk, vw.write_stream(s, pk, serial=0x7700 + seed, packets_per_page=6, trim_last=0), 0, expect_kernel)


def _mono_floor_pair(rng, books, bs, posts=(9, 17), mult=(2, 3)):
    e = [vw.ilog(b) - 1 for b in bs]
    return [make_floor(rng, books, posts[0], mult[0], max(vw.ilog(posts[0]), e[0] - 1)),
            make_floor(rng, books, posts[1], mult[1], max(vw.ilog(posts[1]), e[1] - 1))]


def edge_cw9_10(rng):
    """Every codebook (floor Y books, masterbooks, classbook, VQ books) made of 9- and 10-bit codewords only."""
    books = []
    vq = [len(books), len(books) + 1]
    books += [vq_book(rng, 1, n=600, form="nine_ten", lookup_type=1, value_bits=10),
              vq_book(rng, 2, n=700, form="nine_ten", lookup_type=2, value_bits=4)]
    floors = []
    for posts, mult, rb in ((8, 4, 7), (20, 1, 10)):
        R = FLOOR_RANGE[mult]
        yb = len(books)
        books.append(vw.Book(1, _lengths(rng, 520, "nine_ten")))       # Ys < R use the first entries
        dims = [3, 3] if posts == 8 else [6, 6, 6]
        tail = [int(x) for x in rng.choice(np.arange(1, 1 << rb), size=posts - 2, replace=False)]
        floors.append(vw.Floor1([0] * len(dims), [vw.FloorClass(dims[0], 0, 0, [yb])], mult, rb, tail))
        assert R <= 520
    r = make_residue(rng, books, vq, 1, 0, 1 << 20, 4, 8, 3)
    books[r.classbook] = vw.Book(3, _lengths(rng, 600, "nine_ten"))    # 8^3 = 512 class words + 88 unused ones
    maps = [vw.Mapping([0, 0], [0], [0], [(0, 1)]), vw.Mapping([0, 0], [1], [0], [(0, 1)])]
    return _simple(rng, "cw9_10", 2, (256, 2048), books, floors, [r], maps, [vw.Mode(0, 0), vw.Mode(1, 1)], 30, seed=1)


def edge_cut32(rng):
    """A VQ book with 32-bit codewords; the last packet's final codeword is one of them, and the packet is cut inside it
    (10 to 17 bits in): the zero fill makes the lookup key equal a codeword exactly."""
    books = []
    floors = _mono_floor_pair(rng, books, (256, 2048))
    deep = len(books)
    books.append(vq_book(rng, 1, n=40, form="deep", lookup_type=1, value_bits=6))
    assert max(books[deep].lengths) == 32
    other = len(books)
    books.append(vq_book(rng, 2, n=25))
    r = make_residue(rng, books, [deep, other], 1, 0, 512, 8, 3, 2)
    r.books = [[-1] * 8, [deep] + [-1] * 7, [other] + [-1] * 7]     # pass 0 only: nothing is coded after pass 0
    maps = [vw.Mapping([0], [0], [0]), vw.Mapping([0], [1], [0])]
    s = vw.StreamSetup(1, 44100, (256, 2048), books, floors, [r], maps, [vw.Mode(0, 0), vw.Mode(1, 1)])
    pk = packets_for(rng, s, 24, 0.7, 0.0)
    long32 = [e for e, L in enumerate(books[deep].lengths) if L == 32]
    used = _used_entries(books[deep])
    cuts = 0
    for pc in pk[4::5]:                                # every fifth packet: the last partition codes the deep book, last entry 32 bits
        cls, entries = pc.residue[0]
        last = cls.shape[1] - 1
        cls[0][last] = 1
        es = [int(used[k]) for k in rng.integers(0, len(used), size=8)]
        es[-1] = long32[0]
        entries[(0, last, 0)] = es
        full = vw.write_audio_packet(s, pc)
        rp = read_packet(s, full)
        self_check(s, pc, rp)
        start = rp.last_code_start
        assert rp.last_code_len == 32 and rp.nbits - 8 < start + 32 <= rp.nbits     # the packet's last codeword
        pc.truncate_bytes = (start + 10 + 7) // 8
        assert start + 10 <= pc.truncate_bytes * 8 < start + 32
        cuts += 1
    assert cuts >= 2, cuts
    return Stream("cut32", s, pk, vw.write_stream(s, pk, serial=0x7702, packets_per_page=6))


def edge_wide_floors(rng):
    """Floors of 65, 128 and 250 posts (250 = 2 + 31 * 8: the most a floor1 can have), one per mapping."""
    books = []
    vq = [len(books), len(books) + 1]
    books += [vq_book(rng, 2, n=25), vq_book(rng, 4, n=81)]
    floors = [make_floor(rng, books, 65, 2, 9), make_floor(rng, books, 128, 1, 10), make_floor(rng, books, 250, 4, 12)]
    assert len(floors[2].partition_class) == 31
    r = make_residue(rng, books, vq, 2, 0, 3000, 16, 5, 2)
    maps = [vw.Mapping([0, 0], [0], [0], [(0, 1)]), vw.Mapping([0, 0], [1], [0], [(1, 0)]), vw.Mapping([0, 0], [2], [0], [(0, 1)])]
    modes = [vw.Mode(0, 0), vw.Mode(1, 1), vw.Mode(1, 2)]
    return _simple(rng, "wide_floors", 2, (256, 2048), books, floors, [r], maps, modes, 30, seed=3)


def edge_submaps(rng):
    """8 channels in 8 submaps (one submap per channel: the most a stream of up to 8 channels can fill; a submap without
    channels fails every packet of its mapping, hpp:680), with all three residue types across the submaps."""
    books = []
    vq = [len(books), len(books) + 1, len(books) + 2]
    books += [vq_book(rng, 1), vq_book(rng, 2, n=16), vq_book(rng, 4, n=81)]
    floors = _mono_floor_pair(rng, books, (256, 1024), posts=(6, 12))
    residues = [make_residue(rng, books, vq, t, 0, 400, 8, 4, 2) for t in (0, 1, 2)]
    perm = [int(x) for x in rng.permutation(8)]
    maps = [vw.Mapping(perm, [i % 2 for i in range(8)], [i % 3 for i in range(8)], [(0, 1), (1, 2), (5, 4)]),
            vw.Mapping([i // 2 for i in range(8)], [1, 0, 1, 1], [2, 1, 0, 2], [(6, 7), (7, 3)])]
    return _simple(rng, "submaps8", 8, (256, 1024), books, floors, residues, maps, [vw.Mode(0, 0), vw.Mode(1, 1)], 16, seed=4)


def edge_modes64(rng):
    """64 modes (6 mode bits) over 4 mappings."""
    books = []
    vq = [len(books), len(books) + 1]
    books += [vq_book(rng, 2, n=25), vq_book(rng, 1, n=9)]
    floors = _mono_floor_pair(rng, books, (128, 512))
    residues = [make_residue(rng, books, vq, 1, 0, 200, 4, 4, 2), make_residue(rng, books, vq, 0, 8, 100, 8, 3, 1)]
    maps = [vw.Mapping([0], [i % 2], [i // 2]) for i in range(4)]
    modes = [vw.Mode(i % 2, int(rng.integers(0, 4))) for i in range(64)]
    return _simple(rng, "modes64", 1, (128, 512), books, floors, residues, maps, modes, 40, seed=5)


def edge_begin_past_end(rng):
    """Residue `begin` at and beyond the decode length (nothing to read, hpp:704-705), next to `end` beyond it."""
    books = []
    vq = [len(books)]
    books += [vq_book(rng, 2, n=25)]
    floors = _mono_floor_pair(rng, books, (256, 2048))
    residues = [make_residue(rng, books, vq, 1, 128, 900, 8, 3, 2),     # begin == n/2 of the short block
                make_residue(rng, books, vq, 2, 5000, 9000, 8, 3, 2),   # begin > 2 * 1024 on long blocks
                make_residue(rng, books, vq, 0, 1000, 100000, 8, 3, 2)]  # end > n/2 on every block
    maps = [vw.Mapping([0, 1], [0, 0], [0, 2], [(0, 1)]), vw.Mapping([0, 0], [1], [1], [(0, 1)]),
            vw.Mapping([0, 1], [1, 1], [2, 0], [])]
    modes = [vw.Mode(0, 0), vw.Mode(1, 1), vw.Mode(1, 2)]
    return _simple(rng, "begin_past_end", 2, (256, 2048), books, floors, residues, maps, modes, 24, seed=6)


def edge_psize1(rng):
    """Partition size 1 (one dim-1 vector per partition), types 1 and 2."""
    books = []
    vq = [len(books), len(books) + 1]
    books += [vq_book(rng, 1, n=17), vq_book(rng, 1, n=5, lookup_type=2)]
    floors = _mono_floor_pair(rng, books, (256, 512))
    residues = [make_residue(rng, books, vq, 1, 3, 200, 1, 4, 2), make_residue(rng, books, vq, 2, 0, 301, 1, 5, 3)]
    maps = [vw.Mapping([0, 0], [0], [0], [(0, 1)]), vw.Mapping([0, 0], [1], [1], [(1, 0)])]
    return _simple(rng, "psize1", 2, (256, 512), books, floors, residues, maps, [vw.Mode(0, 0), vw.Mode(1, 1)], 30, seed=7)


def edge_classdim3(rng):
    """A classbook of dimension 3 with 7 partitions (the last class word codes 2 partitions that do not exist), on two
    channels of one type-1 submap and on a type-0 one."""
    books = []
    vq = [len(books), len(books) + 1]
    books += [vq_book(rng, 2, n=25), vq_book(rng, 4, n=81)]
    floors = _mono_floor_pair(rng, books, (256, 2048))
    residues = [make_residue(rng, books, vq, 1, 16, 16 + 7 * 16, 16, 5, 3),
                make_residue(rng, books, vq, 0, 0, 7 * 32 + 5, 32, 4, 3)]
    maps = [vw.Mapping([0, 0], [0], [0]), vw.Mapping([0, 0], [1], [1])]
    return _simple(rng, "classdim3_parts7", 2, (256, 2048), books, floors, residues, maps, [vw.Mode(0, 0), vw.Mode(1, 1)], 30,
                   dense=0.9, seed=8)


def edge_nclass64(rng):
    """64 classifications, class 1 coding all 8 passes."""
    books = []
    vq = [len(books), len(books) + 1, len(books) + 2]
    books += [vq_book(rng, 2, n=16, sequence_p=True), vq_book(rng, 4, n=81), vq_book(rng, 8, n=64, lookup_type=2)]
    floors = _mono_floor_pair(rng, books, (256, 2048))
    r = make_residue(rng, books, vq, 2, 0, 2600, 16, 64, 1, full_class=True)
    maps = [vw.Mapping([0, 0], [0], [0], [(0, 1)]), vw.Mapping([0, 0], [1], [0], [(0, 1)])]
    return _simple(rng, "nclass64_passes8", 2, (256, 2048), books, floors, [r], maps, [vw.Mode(0, 0), vw.Mode(1, 1)], 20, seed=9)


def edge_book65537(rng):
    """A VQ book of 65537 entries: entry numbers need 32 bits in the residue payload."""
    books = []
    big = len(books)
    lengths = [16] * 65535 + [17] * 2
    books.append(vw.Book(2, lengths, 1, minimum=-1.0, delta=1.0 / 128, value_bits=8,
                         multiplicands=[int(x) for x in rng.integers(0, 256, size=256)], ordered=True))
    small = len(books)
    books.append(vq_book(rng, 2, n=25))
    floors = _mono_floor_pair(rng, books, (256, 2048))
    r = make_residue(rng, books, [big, small], 1, 0, 800, 16, 4, 2)
    maps = [vw.Mapping([0], [0], [0]), vw.Mapping([0], [1], [0])]
    return _simple(rng, "book65537", 1, (256, 2048), books, floors, [r], maps, [vw.Mode(0, 0), vw.Mode(1, 1)], 16, seed=10)


def _edge_blocks(rng, bs, channels=2, P=24, name=None, expect_kernel=None, rtype=2, psize=16, end=None, seed=11, dims=(2, 4, 8)):
    books = []
    vq = list(range(len(dims)))
    books += [vq_book(rng, d, n=min(100, 5 ** d)) for d in dims]
    floors = _mono_floor_pair(rng, books, bs, posts=(8, 24))
    dl = bs[1] // 2 * (channels if rtype == 2 else 1)
    r = make_residue(rng, books, vq, rtype, 0, end if end is not None else dl, psize, 4, 2)
    cp = [(c, c + 1) for c in range(0, channels - 1, 2)]
    maps = [vw.Mapping([0] * channels, [0], [0], cp), vw.Mapping([0] * channels, [1], [0], cp)]
    modes = [vw.Mode(0, 0), vw.Mode(1, 1)] if bs[0] != bs[1] else [vw.Mode(0, 0), vw.Mode(1, 1)]
    return _simple(rng, name or "bs_%d_%d" % bs, channels, bs, books, floors, [r], maps, modes, P, dense=0.4, p_unused=0.02,
                   expect_kernel=expect_kernel, seed=seed)


EDGE = {
    "cw9_10": edge_cw9_10,
    "cut32": edge_cut32,
    "wide_floors": edge_wide_floors,
    "submaps8": edge_submaps,
    "modes64": edge_modes64,
    "begin_past_end": edge_begin_past_end,
    "psize1": edge_psize1,
    "classdim3_parts7": edge_classdim3,
    "nclass64_passes8": edge_nclass64,
    "book65537": edge_book65537,
    "bs_64_64": lambda rng: _edge_blocks(rng, (64, 64), P=40, seed=12),
    "bs_64_8192": lambda rng: _edge_blocks(rng, (64, 8192), P=24, end=6000, seed=13),
    "bs_128_4096": lambda rng: _edge_blocks(rng, (128, 4096), P=24, end=5000, seed=14),
    "bs_8192_8192": lambda rng: _edge_blocks(rng, (8192, 8192), P=6, end=6000, seed=15),
    # 8 channels, long blocks of 8192: beyond what one SM holds for the warp and fused kernels
    "ch8_256_8192": lambda rng: _edge_blocks(rng, (256, 8192), channels=8, P=10, end=9000, expect_kernel="staged", seed=16),
    # 8 channels, 4096-sample long blocks, type 2, partition size 16: the residue stage's largest shared-memory need
    "ch8_4096_type2_p16": lambda rng: _edge_blocks(rng, (256, 4096), channels=8, P=8, rtype=2, psize=16, end=2000, seed=17),
    # 8 channels, 8192-sample blocks, partition size 1: 160000 read cursors per packet, more than shared memory holds
    "ch8_8192_type2_p1": lambda rng: _edge_blocks(rng, (256, 8192), channels=8, P=4, rtype=2, psize=1, end=20000, seed=18,
                                                  dims=(1, 1)),
}


@functools.lru_cache(maxsize=None)
def stream(name: str) -> Stream:
    """The named stream: "seed<k>" or an EDGE key. Deterministic; cached for the session."""
    if name.startswith("seed"):
        return random_stream(int(name[4:]))
    rng = np.random.default_rng(sum(map(ord, name)))
    return EDGE[name](rng)


ALL_NAMES = ["seed%d" % k for k in SEEDS] + list(EDGE)


# =====================================================================================================================
# reader
# =====================================================================================================================
def float32_unpack(x: int) -> float:
    """Vorbis I §9.2.2."""
    mantissa = x & 0x1FFFFF
    sign = x & 0x80000000
    exponent = (x & 0x7FE00000) >> 21
    v = float(mantissa) * 2.0 ** (exponent - 788)
    return -v if sign else v


class Huffman:
    """Codeword tree of §3.2.1 built entry by entry: each used entry takes the lowest-valued free codeword of its length,
    i.e. the leftmost free node at that depth. Nodes are [child0, child1, full]; a leaf is the entry number."""

    def __init__(self, lengths):
        self.root = [None, None, False]
        for e, L in enumerate(lengths):
            if L:
                if not self._insert(self.root, 0, int(L), e):
                    raise ValueError("overspecified codebook")
        self.len_of = {e: int(L) for e, L in enumerate(lengths) if L}

    @staticmethod
    def _done(x):
        return x is not None and (x.__class__ is int or x[2])

    def _insert(self, node, depth, L, e):
        for b in (0, 1):
            ch = node[b]
            if depth + 1 == L:
                if ch is None:
                    node[b] = e
                    node[2] = self._done(node[0]) and self._done(node[1])
                    return True
                continue
            if ch is None:
                ch = node[b] = [None, None, False]
            elif ch.__class__ is int or ch[2]:
                continue
            if self._insert(ch, depth + 1, L, e):
                node[2] = self._done(node[0]) and self._done(node[1])
                return True
        return False


@functools.lru_cache(maxsize=None)
def _huffman_cached(lengths: tuple) -> Huffman:
    return Huffman(lengths)


def huffman_of(book) -> Huffman:
    h = getattr(book, "_reader_tree", None)
    if h is None:
        h = _huffman_cached(tuple(book.lengths))
        book._reader_tree = h
    return h


class BitReader:
    """LSb-first bit reader (§2.1.4); bits past the end read as zero."""

    def __init__(self, data: bytes):
        self.bits = np.unpackbits(np.frombuffer(data, np.uint8), bitorder="little").tolist() if data else []
        self.n = len(self.bits)
        self.pos = 0
        self.last_code_start = -1
        self.last_code_len = 0

    def read(self, nbits: int) -> int:
        v = 0
        bits, n, p = self.bits, self.n, self.pos
        for i in range(nbits):
            if p < n and bits[p]:
                v |= 1 << i
            p += 1
        self.pos = p
        return v

    def code(self, tree: Huffman) -> int:
        bits, n, p = self.bits, self.n, self.pos
        self.last_code_start = p
        node = tree.root
        while True:
            node = node[bits[p] if p < n else 0]
            p += 1
            if node.__class__ is int:
                break
            if node is None:
                raise ValueError("undecodable codeword")
        self.last_code_len = p - self.pos
        self.pos = p
        return node


@dataclass
class ReadPacket:
    mode: int
    prev_flag: int
    next_flag: int
    ys: List[Optional[List[int]]]
    # per submap: cls [vch][parts] (rows of channels that are not decoded stay 0), entries {(pass, part, ch): [entry...]},
    # the entry numbers in decode order, and what the geometry was
    residue: List[Tuple[np.ndarray, Dict[Tuple[int, int, int], List[int]], List[int]]] = field(default_factory=list)
    floor_end_bit: int = 0
    last_code_start: int = -1
    last_code_len: int = 0
    nbits: int = 0


def read_packet(s: vw.StreamSetup, data: bytes) -> ReadPacket:
    br = BitReader(data)
    assert br.read(1) == 0, "not an audio packet"
    mode = br.read(vw.ilog(len(s.modes) - 1))
    m = s.modes[mode]
    prev_flag = next_flag = 0
    if m.blockflag:
        prev_flag = br.read(1)
        next_flag = br.read(1)
    mp = s.mappings[m.mapping]
    n = s.blocksize[m.blockflag]
    # §7.2.3 floor1 packet decode
    ys: List[Optional[List[int]]] = []
    for c in range(s.channels):
        fl = s.floors[mp.submap_floor[mp.mux[c]]]
        if br.read(1) == 0:
            ys.append(None)
            continue
        rng_ = FLOOR_RANGE[fl.multiplier]
        y = [br.read(vw.ilog(rng_ - 1)), br.read(vw.ilog(rng_ - 1))]
        for cls_no in fl.partition_class:
            cl = fl.classes[cls_no]
            cbits = cl.subclass_bits
            csub = (1 << cbits) - 1
            cval = br.code(huffman_of(s.books[cl.masterbook])) if cbits else 0
            for _ in range(cl.dim):
                book = cl.books[cval & csub]
                cval >>= cbits
                y.append(br.code(huffman_of(s.books[book])) if book >= 0 else 0)
        ys.append(y)
    floor_end = br.pos
    # §4.3.3 nonzero vector propagate
    used = [v is not None for v in ys]
    for mg, an in mp.couplings:
        if used[mg] or used[an]:
            used[mg] = used[an] = True
    # §8.6.2 residue decode, one submap after the other
    out = []
    for sm in range(len(mp.submap_floor)):
        chs = [c for c in range(s.channels) if mp.mux[c] == sm]
        r = s.residues[mp.submap_residue[sm]]
        if r.type == 2:
            vch, decode, dl = 1, [True], len(chs) * (n // 2)
        else:
            vch, decode, dl = len(chs), [used[c] for c in chs], n // 2
        lb, le = min(r.begin, dl), min(r.end, dl)
        parts = (le - lb) // r.partition_size
        cb = s.books[r.classbook]
        cw = cb.dim
        cls = np.zeros((vch, parts + cw), np.int64)          # room for the class-word digits past the last partition
        entries: Dict[Tuple[int, int, int], List[int]] = {}
        flat: List[int] = []
        if le > lb:
            for pass_ in range(8):
                pc = 0
                while pc < parts:
                    if pass_ == 0:
                        for j in range(vch):
                            if not decode[j]:
                                continue
                            t = br.code(huffman_of(cb))
                            for i in range(cw - 1, -1, -1):
                                cls[j][pc + i] = t % r.n_class
                                t //= r.n_class
                    for _ in range(cw):
                        if pc >= parts:
                            break
                        for j in range(vch):
                            if not decode[j]:
                                continue
                            book = r.books[int(cls[j][pc])][pass_]
                            if book < 0:
                                continue
                            bk = s.books[book]
                            tree = huffman_of(bk)
                            es = [br.code(tree) for _ in range(r.partition_size // bk.dim)]
                            entries[(pass_, pc, j)] = es
                            flat += es
                        pc += 1
        out.append((cls[:, :parts].copy(), entries, flat))
    return ReadPacket(mode, prev_flag, next_flag, ys, out, floor_end, br.last_code_start, br.last_code_len, br.n)


def self_check(s: vw.StreamSetup, pc: vw.PacketChoice, rp: ReadPacket):
    """The reader read what the writer encoded (untruncated packets)."""
    assert rp.mode == pc.mode
    if s.modes[pc.mode].blockflag:
        assert (rp.prev_flag, rp.next_flag) == (pc.prev_flag, pc.next_flag)
    assert rp.ys == [None if y is None else list(y) for y in pc.ys]
    mp = s.mappings[s.modes[pc.mode].mapping]
    used = vw.propagate([y is not None for y in pc.ys], mp.couplings)
    for sm, ((wcls, wents), (rcls, rents, _)) in enumerate(zip(pc.residue, rp.residue)):
        r = s.residues[mp.submap_residue[sm]]
        chs = [c for c in range(s.channels) if mp.mux[c] == sm]
        dec = [True] if r.type == 2 else [used[c] for c in chs]
        wcls = np.asarray(wcls).reshape(rcls.shape) if np.asarray(wcls).size else np.zeros(rcls.shape, np.int64)
        for j, d in enumerate(dec):
            if d:
                assert np.array_equal(rcls[j], wcls[j]), (sm, j)
        want = {k: list(v) for k, v in wents.items() if dec[k[2]]}
        if rcls.shape[1] == 0:
            want = {}
        assert rents == want, sm


# =====================================================================================================================
# model
# =====================================================================================================================
@functools.lru_cache(maxsize=None)
def _vq_cached(dim, n, lookup_type, minimum_packed, delta_packed, sequence_p, mult: tuple) -> np.ndarray:
    minimum, delta = float32_unpack(minimum_packed), float32_unpack(delta_packed)
    mult = np.asarray(mult, np.float64)
    out = np.zeros((n, dim), np.float32)
    last = np.zeros(n, np.float64)
    e = np.arange(n, dtype=np.int64)
    nv = len(mult)
    for d in range(dim):
        if lookup_type == 1:
            off = (e // (nv ** d)) % nv
        else:
            off = e * dim + d
        v = (mult[off] * delta + minimum + last).astype(np.float32)      # double arithmetic, rounded to float
        out[:, d] = v
        if sequence_p:
            last = v.astype(np.float64)
    return out


def vq_table(book) -> np.ndarray:
    """[n_entries, dim] float32 VQ values of a lookup type 1/2 book, from its header fields as coded."""
    return _vq_cached(book.dim, book.n_entries, book.lookup_type, vw.float32_pack(book.minimum), vw.float32_pack(book.delta),
                      bool(book.sequence_p), tuple(book.multiplicands))


def model_after_residue(s: vw.StreamSetup, rp: ReadPacket) -> np.ndarray:
    """[channels, n/2] float32: the residue vectors after §8.6.2 (+ type-2 de-interleave), before inverse coupling."""
    m = s.modes[rp.mode]
    mp = s.mappings[m.mapping]
    half = s.blocksize[m.blockflag] // 2
    out = np.zeros((s.channels, half), np.float32)
    for sm, (cls, entries, _) in enumerate(rp.residue):
        chs = [c for c in range(s.channels) if mp.mux[c] == sm]
        r = s.residues[mp.submap_residue[sm]]
        nch = len(chs)
        vch, dl = (1, nch * half) if r.type == 2 else (nch, half)
        lb = min(r.begin, dl)
        v = np.zeros((vch, dl), np.float32)
        for pass_ in range(8):                       # every bin gets at most one addend per pass: add pass by pass
            for (ps, p, j), es in entries.items():
                if ps != pass_:
                    continue
                bk = s.books[r.books[int(cls[j][p])][pass_]]
                dim, nvec = bk.dim, r.partition_size // bk.dim
                vals = vq_table(bk)[np.asarray(es, np.int64)]          # [nvec, dim]
                k = np.arange(nvec)[:, None]
                l = np.arange(dim)[None, :]
                idx = lb + p * r.partition_size + ((k + l * nvec) if r.type == 0 else (k * dim + l))
                v[j, idx.ravel()] += vals.ravel()
        if r.type == 2:
            for j, c in enumerate(chs):
                out[c] = v[0, j::nch]
        else:
            for j, c in enumerate(chs):
                out[c] = v[j]
    return out


# =====================================================================================================================
# what the library's host parse produced (ctypes views)
# =====================================================================================================================
def packets_array(b) -> np.ndarray:
    raw = np.ctypeslib.as_array(C.cast(b.packets, C.POINTER(C.c_uint8)), shape=(b.n_packets * C.sizeof(abi.pov_packet),))
    return raw.view(abi.PACKET_DTYPE).copy()


def streams_array(b) -> np.ndarray:
    raw = np.ctypeslib.as_array(C.cast(b.streams, C.POINTER(C.c_uint8)), shape=(b.n_streams * C.sizeof(abi.pov_stream),))
    return raw.view(abi.STREAM_DTYPE).copy()


def entry_bits(s: vw.StreamSetup) -> int:
    return 32 if max(bk.n_entries for bk in s.books) > 65536 else 16


def split_entries_payload(s: vw.StreamSetup, b, pk, mode) -> List[Tuple[np.ndarray, np.ndarray]]:
    """One POV_INPUT_ENTRIES packet payload (include/pov_synth.h) -> per submap (cls [vch, parts], entries in order)."""
    payload = np.ctypeslib.as_array(C.cast(b.payload, C.POINTER(C.c_uint8)), shape=(int(b.payload_bytes),))
    m = s.modes[mode]
    mp = s.mappings[m.mapping]
    half = s.blocksize[m.blockflag] // 2
    eb = entry_bits(s) // 8
    off = int(pk["spec_off"])
    out = []
    for sm in range(len(mp.submap_floor)):
        nch = sum(1 for c in range(s.channels) if mp.mux[c] == sm)
        r = s.residues[mp.submap_residue[sm]]
        vch, dl = (1, nch * half) if r.type == 2 else (nch, half)
        parts = (min(r.end, dl) - min(r.begin, dl)) // r.partition_size
        ne = int(payload[off:off + 4].view(np.uint32)[0])
        cls = payload[off + 4:off + 4 + vch * parts].reshape(vch, parts).astype(np.int64)
        cb = (vch * parts + 3) & ~3
        e0 = off + 4 + cb
        ents = payload[e0:e0 + ne * eb].view(np.uint16 if eb == 2 else np.uint32).astype(np.int64)
        out.append((cls, ents))
        off = e0 + ((ne * eb + 3) & ~3)
    return out
