"""Cut mode of the corpus decode on the GPU (pov_ctx_set_cut_damage, k_cut_damaged). One corpus mixes clean files, every kind
of geometry damage (truncation, CRC, capture pattern, a bad packet header at a page start, the second link of a chained file,
random bytes, an empty file) and content damage (the bit-flip helper of test_gpu_decode.py on random multichannel streams, one
of them 200 packets long and cut past packet 100 and frame 32 768, and synth_bad_vq_book.ogg), whose strict decode fails
with a status word.

The reference is the strict decode of the "repaired" corpus: every geometry-damaged file replaced by its pages before the
damage (random bytes by an empty file), every content-damaged file by itself with the packets from the first damaged one on
restored from the undamaged original. It has the same stream table,
the same setups per chunk and, in the same layout, the same alignment, so in every output mode:
- clean streams and geometry-damaged streams are bit-identical to it,
- a content-damaged stream is bit-identical over [0, valid) and exactly 0 over [valid, frames),
- padding keeps its sentinel, and the report says what the CPU side predicts."""
import contextlib
import ctypes as C
import os
import re
import sys

import numpy as np
import pytest

from parseoggvorbis_b200 import abi, lib
from tests import random_vorbis as rv
from tests.test_corpus_damage_cpu import audio_packets, bad_header_bits, load, page_starts, parse_packets, with_page_crc, vw
from tests.test_gpu_corpus_device import SENTINEL_I16, _env, _layout, _sentinel_tensor

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@contextlib.contextmanager
def _cut(ctx, on):
    ctx.set_cut_damage(on)
    try:
        yield
    finally:
        ctx.set_cut_damage(False)


@pytest.fixture(scope="module")
def ctx():
    c = lib.SynthContext(0)
    yield c
    c.close()


def content_damage(ctx):
    """(damaged file, undamaged original, p, reason): synth_bad_vq_book.ogg, whose residue class points at a scalar codebook so
    that the first packet using the class fails with a VQ-entry status word, and the same packets under a setup in which that
    book has a VQ table. Packets < p are the same in both, so is every packet's geometry."""
    import copy
    sys.path.insert(0, os.path.join(ROOT, "tests", "golden"))
    import make_synthetic_golden as msg
    s, packets, bad = msg.build("bad_vq_book")
    assert bad == load("synth_bad_vq_book")
    fixed = copy.deepcopy(s)
    k = 1 + next(i for i, b in enumerate(s.books) if b.lookup_type)          # the scalar book after the good VQ book
    b = fixed.books[k]
    fixed.books[k] = vw.Book(b.dim, b.lengths, lookup_type=2, multiplicands=[(3 * i) % 16 for i in range(b.n_entries * b.dim)])
    original = vw.write_stream(fixed, packets, serial=0x5000 + 17, packets_per_page=6)
    with pytest.raises(lib.PovError) as ei:
        ctx.decode_ogg(bad)
    m = re.fullmatch(r"audio packet (\d+): check failed: (.*)", ei.value.msg)
    assert m, ei.value.msg
    ctx.decode_ogg(original)
    return bad, original, int(m.group(1)), m.group(2)


def _statuses(ctx, data):
    """Per audio packet, the status word of the single-stream batch decode (POV_INPUT_PACKETS) of `data`."""
    po = lib.ParsedOgg(data, raw_packets=True)
    h = C.c_void_p(None)
    try:
        s, b = po.get(0)
        sid = C.c_uint32(0)
        ctx._check(ctx.L.pov_setup_register(ctx.ctx, C.byref(s), C.byref(sid)))
        abi.pov_stream.from_address(C.addressof(b.streams.contents)).setup_id = sid.value
        ctx._check(ctx.L.pov_batch_upload(ctx.ctx, C.byref(b), C.byref(h)))
        ctx._check(ctx.L.pov_batch_run(ctx.ctx, h))
        out = np.zeros(b.n_packets, np.uint32)
        ctx.L.pov_batch_status(ctx.ctx, h, out.ctypes.data_as(C.POINTER(C.c_uint32)), len(out))
        return out
    finally:
        if h:
            ctx.L.pov_batch_free(ctx.ctx, h)
        po.close()


def flip_damage(ctx, base, flips, keep=0, want=lambda p, bad, pcm_off: True, seeds=range(400)):
    """(damaged file, repaired file, p, reason) from the bit-flip helper of test_gpu_decode.py: the first seed whose damage
    leaves every packet's geometry as it was (so it is content damage), makes the strict whole-file decode fail with a status
    word at packet p, and satisfies want(p, damaged packets, pcm_off). Audio pages before the one holding packet `keep` stay
    pristine. The repaired file is the damaged one with packets >= p restored from `base`: its packets < p are the damaged
    file's, so a strict decode of it is what the cut decode must equal before the cut."""
    from tests.test_gpu_decode import _flip_bits_in_audio_packets
    (_, pcm_off, emit, _, _), = parse_packets(base, raw_packets=True)
    pk = audio_packets(base)
    for seed in seeds:
        bad = bytearray(_flip_bits_in_audio_packets(base, np.random.default_rng(seed), flips=flips))
        bad[:pk[keep][0]] = base[:pk[keep][0]]
        bad = bytes(bad)
        try:
            lib.corpus_streams([bad])
        except lib.PovError:
            continue                                      # geometry damage
        if parse_packets(bad, raw_packets=True)[0][1:3] != (pcm_off, emit):
            continue
        try:
            ctx.decode_ogg(bad)
            continue                                      # not damaged at all
        except lib.PovError as e:
            m = re.fullmatch(r"audio packet (\d+): check failed: (.*)", e.msg)
        if not m:
            continue
        p = int(m.group(1))
        damaged = np.flatnonzero(_statuses(ctx, bad))
        if damaged[0] != p or not want(p, damaged, pcm_off):
            continue
        fixed = bytearray(bad)
        for _, off, n in pk[p:]:
            fixed[off:off + n] = base[off:off + n]
        for at in page_starts(base)[3:]:
            with_page_crc(fixed, at)
        fixed = bytes(fixed)
        ctx.decode_ogg(fixed)
        return bad, fixed, p, m.group(2)
    raise AssertionError("no seed gives content damage")


def long_stream():
    """A 5-channel random stream of 200 packets (about 75 000 frames): seed6's setup, whose floors bit flips can push out of range."""
    st = rv.stream("seed6")
    return vw.write_stream(st.setup, rv.packets_for(np.random.default_rng(606), st.setup, 200, 0.5), serial=0x7606, packets_per_page=8)


def _geometry_error(f, k):
    try:
        lib.corpus_streams([f])
    except lib.PovError as e:
        return e.msg.replace("file 0:", "file %d:" % k, 1)
    raise AssertionError("file %d is not damaged at the page level" % k)


def _build(ctx):
    """(damaged corpus, repaired corpus, {file: ("geometry", message) | ("content", packet, reason)})."""
    stereo, mono, sub = load("stereo44khz"), load("mono44khz"), load("synth_two_submaps")
    seeds = [rv.stream("seed%d" % k).data for k in (0, 9, 7, 3)]
    D, R, what = [], [], {}

    def add(bad, ref, kind=None):
        k = len(D)
        D.append(bad); R.append(ref)
        if kind == "geometry":
            what[k] = ("geometry", _geometry_error(bad, k))
        elif kind is not None:
            what[k] = kind
    add(stereo, stereo)
    st = page_starts(stereo)
    cut = int(len(stereo) * 0.7)
    add(stereo[:cut], stereo[:max(s for s in st if s <= cut)], "geometry")         # truncated inside a page
    add(mono, mono)
    s3 = seeds[3]; p3 = page_starts(s3); buf = bytearray(s3); buf[p3[4] + 33] ^= 4
    add(bytes(buf), s3[:p3[4]], "geometry")                                         # CRC
    add(seeds[0], seeds[0])
    s51 = load("synth_surround51"); p51 = page_starts(s51); buf = bytearray(s51); buf[p51[3]] = ord("x")
    add(bytes(buf), s51[:p51[3]], "geometry")                                       # capture pattern
    s1 = seeds[1]; ap = audio_packets(s1); pages = sorted({a for a, _, _ in ap}); pg = pages[len(pages) // 2]
    p = next(i for i, (a, _, _) in enumerate(ap) if a == pg)                        # first packet of a middle audio page
    add(bad_header_bits(s1, p), s1[:pg], "geometry")
    bad, original, p, reason = content_damage(ctx)
    add(bad, original, ("content", p, reason))
    for src in ("seed6", "seed5"):                       # the bit-flip helper on random multichannel streams
        bad, fixed, p, reason = flip_damage(ctx, rv.stream(src).data, 12)
        add(bad, fixed, ("content", p, reason))
    # a long 5-channel stream cut past packet 100 and frame 32 768, with damaged packets in more than one 32-packet group
    bad, fixed, p, reason = flip_damage(ctx, long_stream(), 60, keep=100,
                                        want=lambda p, bad, pcm_off: pcm_off[p] > 32768 and len({int(q) // 32 for q in bad}) >= 2)
    add(bad, fixed, ("content", p, reason))
    add(sub, sub)
    chained = vw.chain_files([mono, seeds[2]]); at = len(mono) + page_starts(seeds[2])[4]
    buf = bytearray(chained); buf[at + 40] ^= 1
    add(bytes(buf), chained[:at], "geometry")                                       # second link
    add(bytes(np.random.default_rng(3).integers(0, 256, 3000, dtype=np.uint8)), b"", "geometry")
    add(b"", b"")
    add(seeds[2], seeds[2])
    return D, R, what


@pytest.fixture(scope="module")
def corpus(ctx):
    return _build(ctx)


def _expected_report(D, R, what):
    """Per file: (status, message) and per record the valid frames, from the CPU side."""
    table = lib.corpus_streams(R)
    valid = table.frames.copy()
    msgs = {}
    for k, w in what.items():
        if w[0] == "geometry":
            msgs[k] = w[1]
        else:
            i = int(np.flatnonzero(table.file == k)[0])
            (_, pcm_off, _, _, _), = parse_packets(R[k], raw_packets=True)
            valid[i] = pcm_off[w[1]]
            msgs[k] = "file %d: stream 0: check failed: audio packet %d: %s" % (k, w[1], w[2])
    return table, valid, msgs


def _check_report(rep, table, valid, msgs, n_files):
    assert rep.damaged == msgs
    assert np.array_equal(rep.stream_valid_frames, valid)
    for k in range(n_files):
        sel = table.file == k
        assert rep.n_streams[k] == sel.sum() and rep.frames[k] == table.frames[sel].sum() and rep.valid_frames[k] == valid[sel].sum()
        assert rep.status[k] == (abi.POV_ERR_STREAM if k in msgs else abi.POV_OK)


def _streams(pcm_img, table, base, stride, frames=None):
    frames = table.frames if frames is None else frames
    return [np.stack([pcm_img[int(b) + c * int(s):int(b) + c * int(s) + int(f)] for c in range(int(ch))])
            for b, s, ch, f in zip(base, stride, table.channels, frames)]


def _compare(got, ref, valid, frames):
    for i, (g, r) in enumerate(zip(got, ref)):
        v = int(valid[i])
        assert g.shape == r.shape, i
        gb = g.view(np.uint32) if g.dtype == np.float32 else g
        rb = r.view(np.uint32) if r.dtype == np.float32 else r
        assert np.array_equal(gb[:, :v], rb[:, :v]), i
        assert not np.any(gb[:, v:]), i                 # exact (+0) zeros


def _device(ctx, files, cut, s16=False, chunk=None, sample_rate=None, mono=False):
    """decode_corpus_into a packed sentinel tensor; -> (table, per-stream arrays, frames per file, report or None)."""
    env = {} if chunk is None else {"POV_CORPUS_CHUNK": str(chunk)}
    table = lib.corpus_streams(files, cut_damage=cut)
    if sample_rate or mono:
        ofr = lib.resampled_frames(table, int(sample_rate or 0))
        och = np.ones(len(table), np.uint32) if mono else table.channels.astype(np.uint32)
    else:
        ofr, och = table.frames, table.channels
    view = lib.StreamTable(table.file, och, table.sample_rate, ofr)
    base, stride, n = _layout(view, "packed")
    t = _sentinel_tensor(n, s16)
    with _env(env), _cut(ctx, cut):
        frames, _ = ctx.decode_corpus_into(files, t, table, base, stride, s16=s16, host_threads=4, sample_rate=sample_rate, mono=mono)
    img = t.cpu().numpy()
    mask = np.ones(n, bool)
    for b, s, c, f in zip(base, stride, och, ofr):
        for k in range(int(c)):
            mask[int(b) + k * int(s):int(b) + k * int(s) + int(f)] = False
    pad = img[mask]
    assert np.all(pad == SENTINEL_I16) if s16 else np.all(np.isnan(pad))
    return table, _streams(img, view, base, stride), frames, ctx.corpus_report() if cut else None


@pytest.mark.parametrize("s16", [False, True])
@pytest.mark.parametrize("chunk", [None, 1, 7])
def test_device_output_is_the_repaired_corpus_cut(ctx, corpus, s16, chunk):
    D, R, what = corpus
    table, valid, msgs = _expected_report(D, R, what)
    with _env({} if chunk is None else {"POV_CORPUS_CHUNK": str(chunk)}):
        with pytest.raises(lib.PovError) as ei:
            ctx.decode_corpus(D, host_threads=4)
    assert ei.value.code == abi.POV_ERR_STREAM and ei.value.msg == msgs[min(msgs)]     # strict mode: today's first error
    t_cut, got, frames, rep = _device(ctx, D, True, s16=s16, chunk=chunk)
    t_ref, ref, frames_ref, _ = _device(ctx, R, False, s16=s16, chunk=chunk)
    assert [tuple(map(int, x)) for x in zip(*t_cut)] == [tuple(map(int, x)) for x in zip(*t_ref)]
    assert np.array_equal(frames, frames_ref)
    _check_report(rep, table, valid, msgs, len(D))
    _compare(got, ref, valid, table.frames)


def test_padded_layout_and_device_corpus_fields(ctx, corpus):
    D, R, what = corpus
    table, valid, msgs = _expected_report(D, R, what)
    out = ctx.decode_corpus_device(D, layout="padded", cut_damage=True, host_threads=4)
    ref = ctx.decode_corpus_device(R, layout="padded", host_threads=4)
    assert out.damaged == msgs and np.array_equal(out.valid_frames, valid)
    assert ref.damaged == {} and np.array_equal(ref.valid_frames, ref.table.frames)
    a, b = out.pcm.cpu().numpy(), ref.pcm.cpu().numpy()
    _compare([a[i, :int(c), :int(f)] for i, (c, f) in enumerate(zip(table.channels, table.frames))],
             [b[i, :int(c), :int(f)] for i, (c, f) in enumerate(zip(table.channels, table.frames))], valid, table.frames)
    for i, (c, f) in enumerate(zip(table.channels, table.frames)):      # zero padding stays zero
        assert not a[i, int(c):].any() and not a[i, :, int(f):].any()


def test_host_entropy_walk_gives_the_same_report_and_pcm(ctx, corpus):
    """The host walk (a packet it cannot walk enters the batch as silence) reports what the device walk reports, and its PCM
    is the repaired corpus' strict decode with the same walk cut the same way. (The two walks' chunks can run different
    synthesis kernels, whose float32 results may differ in the last bit, so each walk is held to its own strict decode.)"""
    D, R, what = corpus
    table, valid, msgs = _expected_report(D, R, what)
    _, _, _, rep_dev = _device(ctx, D, True)
    ctx.set_device_entropy(False)
    try:
        _, host, _, rep_host = _device(ctx, D, True)
        _, ref, _, _ = _device(ctx, R, False)
    finally:
        ctx.set_device_entropy(True)
    assert rep_host.damaged == rep_dev.damaged == msgs
    assert np.array_equal(rep_host.stream_valid_frames, rep_dev.stream_valid_frames)
    _compare(host, ref, valid, table.frames)


def test_resampled_output_is_the_resample_of_the_zero_tailed_stream(ctx, corpus):
    D, R, what = corpus
    table, valid, _ = _expected_report(D, R, what)
    _, got, _, _ = _device(ctx, D, True, sample_rate=16000, mono=True)
    _, ref, _, _ = _device(ctx, R, False, sample_rate=16000, mono=True)
    for i, (g, r) in enumerate(zip(got, ref)):
        assert g.shape == r.shape
        if valid[i] == table.frames[i]:
            assert np.array_equal(g.view(np.uint32), r.view(np.uint32)), i
            continue
        L, M, hl, _ = lib.resample_filter(int(table.sample_rate[i]), 16000)
        v = int(valid[i])
        same = max(0, (v * L - hl + M - 1) // M)          # outputs that read inputs < valid only
        zero = (v * L + hl + M - 1) // M                  # outputs that read inputs >= valid only
        assert np.array_equal(g[:, :same].view(np.uint32), r[:, :same].view(np.uint32)), i
        assert not np.any(g[:, zero:].view(np.uint32)), i


def test_sink_and_checksum_see_the_zero_tailed_pcm(ctx, corpus):
    D, R, what = corpus
    table, valid, msgs = _expected_report(D, R, what)

    def run(files, cut):
        got = []

        def sink(i, pcm):
            got.append((i, pcm.copy()))
            return False
        with _cut(ctx, cut):
            frames, total, chk = ctx.decode_corpus_pcm(files, sink, host_threads=4)
        return got, frames, total, chk
    got, frames, total, chk = run(D, True)
    assert ctx.corpus_report().damaged == msgs
    ref, frames_r, total_r, _ = run(R, False)
    assert [i for i, _ in got] == [i for i, _ in ref] and np.array_equal(frames, frames_r) and total == total_r
    nz = table.frames > 0                               # streams without frames are not delivered
    _compare([p for _, p in got], [p for _, p in ref], valid[nz], table.frames[nz])
    expect = sum(float(p.astype(np.float64).sum()) for _, p in got)
    with _cut(ctx, True):
        _, _, chk2 = ctx.decode_corpus(D, host_threads=4)
    assert abs(chk - expect) <= 1e-6 * max(1.0, abs(expect)) and abs(chk2 - expect) <= 1e-6 * max(1.0, abs(expect))
    with _cut(ctx, True):
        _, _, s16 = ctx.decode_corpus(D, host_threads=4, s16=True)
    _, got16, _, _ = _device(ctx, D, True, s16=True)
    assert s16 == sum(int(p.astype(np.int64).sum()) for p in got16)


def test_every_file_damaged_and_damage_at_the_first_packet(ctx, corpus):
    D, R, what = corpus
    bad = [D[k] for k in sorted(what)]
    t_cut, got, _, rep = _device(ctx, bad, True)
    assert set(rep.damaged) == set(range(len(bad)))
    stereo = load("stereo44khz")
    files = [stereo, bad_header_bits(stereo, 0)]
    t_cut, got, _, rep = _device(ctx, files, True)
    assert list(t_cut.frames) == [int(lib.corpus_streams([stereo]).frames[0]), 0]
    assert rep.damaged == {1: "file 1: check failed: audio packet 0: audio packet: packet type bit set (hpp:1142)"}
    assert list(rep.stream_valid_frames) == list(t_cut.frames) and got[1].shape == (2, 0)


def test_clean_cut_mode_costs_one_launch_per_chunk(ctx, corpus):
    D, R, what = corpus
    clean = [D[k] for k in range(len(D)) if k not in what and len(D[k])]
    with _env({"POV_CORPUS_CHUNK": "1"}):
        counts = []
        for cut in (False, True, False):
            before = ctx.launch_count
            with _cut(ctx, cut):
                ctx.decode_corpus(clean, host_threads=2)
            counts.append(ctx.launch_count - before)
            if cut:
                assert ctx.corpus_report().damaged == {}
    assert counts[0] == counts[2] and counts[1] == counts[0] + len(clean)


def test_report_refuses_the_wrong_sizes(ctx, corpus):
    D, _, _ = corpus
    with _cut(ctx, True):
        ctx.decode_corpus(D[:3], host_threads=2)
    files = (abi.pov_file_report * 4)()
    L = ctx.L
    assert L.pov_corpus_report(ctx.ctx, 4, files, 0, None) == abi.POV_ERR_ARG
    assert L.pov_corpus_report(ctx.ctx, 3, files, 0, None) == abi.POV_OK
    m = int(sum(files[i].n_streams for i in range(3)))
    valid = (C.c_uint64 * (m + 1))()
    assert L.pov_corpus_report(ctx.ctx, 3, files, m + 1, valid) == abi.POV_ERR_ARG
    assert L.pov_corpus_report(ctx.ctx, 3, files, m, valid) == abi.POV_OK
    # a corpus call that fails, even in its argument checks before any decode, leaves no report behind
    arr, lens = (C.c_char_p * 3)(*D[:3]), (C.c_size_t * 3)(*[len(f) for f in D[:3]])
    assert L.pov_decode_corpus_device(ctx.ctx, 3, arr, lens, 0, None, None, None) == abi.POV_ERR_ARG
    assert L.pov_corpus_report(ctx.ctx, 3, files, 0, None) == abi.POV_ERR_ARG
