"""Resampling and mono downmix of the device corpus decode (pov_decode_corpus_device_resampled, decode_corpus_device(
sample_rate=, mono=)). The reference is the native padded float32 decode of the same context variant, taken to float64, averaged
over the channels for mono and passed through scipy.signal.resample_poly. Same-rate output must be the native samples (or the
float32 downmix) bit for bit, int16 the POV_PCM_S16 rule applied to the float32 output, and float32 the same in every chunking,
entropy path and layout.

SNR is taken against the larger of the output's and the input's power. A float32 evaluation errs in proportion to its input,
and a stream whose energy lies mostly above the new Nyquist frequency loses most of its power to the lowpass:
synth_codebooks at 44.1 kHz -> 16 kHz keeps -35 dB of its power, and an exact numpy model of the kernel's float32
arithmetic reaches 114-121 dB against its output there. Streams that keep at least 1 % of their power are held to 120 dB
against their output as well."""
import copy
import ctypes as C
import os
import sys

import numpy as np
import pytest
import scipy.signal as ss

from parseoggvorbis_b200 import abi, lib
from tests import random_vorbis as rv
from tests.test_gpu_corpus_device import FIX, RANDOM, VARIANTS, _env, _layout, _load, _raw_device_pcm, _sentinel_tensor

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "tools"))
import vorbis_writer as vw  # noqa: E402

# (out_rate, mono)
TARGETS = [(16000, True), (16000, False), (48000, False), (22050, False), (8000, False)]


def _rewrite(name, rate, n_packets=None, serial=0x7900):
    """Stream `name` of the random set with its header saying `rate` Hz (and only its first n_packets audio packets)."""
    st = rv.stream(name)
    s = copy.copy(st.setup)
    s.sample_rate = rate
    pk = st.packets if n_packets is None else st.packets[:n_packets]
    return vw.write_stream(s, pk, serial=serial, packets_per_page=6)


@pytest.fixture(scope="module")
def files():
    out = [_load(n) for n in FIX] + [rv.stream(n).data for n in RANDOM]
    out.insert(5, vw.chain_files([_load("stereo44khz"), _load("synth_surround51"), _load("mono44khz")]))
    out.append(_rewrite("seed3", 16000, serial=0x7901))          # a 16 kHz stream
    out.append(_rewrite("seed5", 48000, n_packets=0, serial=0x7902))   # headers only
    out.append(_rewrite("bs_64_64", 48000, n_packets=2, serial=0x7903))   # 48 kHz, 32 frames: at 48k -> 8k every output
    return out                                                           # reaches the zero padding on both sides


@pytest.fixture(scope="module")
def contexts():
    made = {}

    def get(variant):
        if variant not in made:
            with _env({k: v for k, v in VARIANTS[variant].items() if k != "POV_CORPUS_CHUNK"}):
                made[variant] = lib.SynthContext(0)
        return made[variant]
    yield get
    for c in made.values():
        c.close()


def _chunk_env(variant):
    return _env({k: v for k, v in VARIANTS[variant].items() if k == "POV_CORPUS_CHUNK"})


_NATIVE = {}


def _native(ctx, variant, files):
    """Per stream the (channels, frames) float32 PCM of the native padded device decode."""
    key = (variant, len(files), sum(len(f) for f in files))
    if key not in _NATIVE:
        with _chunk_env(variant):
            out = ctx.decode_corpus_device(files, layout="padded", host_threads=4)
        pcm = out.pcm.cpu().numpy()
        _NATIVE[key] = (out.table, [pcm[i, :int(out.table.channels[i]), :int(out.table.frames[i])].copy() for i in range(len(out.table))])
    return _NATIVE[key]


def _downmix_f32(x):
    """The float32 downmix rule: s = x0; s = s + x1 (rounded); ...; m = s * (1.0f / C) (rounded)."""
    s = x[0].astype(np.float32)
    for c in range(1, x.shape[0]):
        s = (s + x[c]).astype(np.float32)
    return (s * (np.float32(1) / np.float32(x.shape[0]))).astype(np.float32)


def _s16(y):
    r = np.clip(np.rint(y.astype(np.float64) * 32768.0), -32768, 32767)
    r[np.isnan(y)] = 0
    return r.astype(np.int16)


def _resampled(ctx, variant, files, out_rate, mono, s16=False, layout="packed"):
    """Run the resampled decode into a sentinel tensor laid out by `layout`; -> (table, per-stream outputs, tensor image, base,
    stride, out_channels, out_frames)."""
    table = lib.corpus_streams(files)
    ofr = lib.resampled_frames(table, out_rate)
    och = np.ones(len(table), np.uint32) if mono else table.channels.astype(np.uint32)
    view = lib.StreamTable(table.file, och, table.sample_rate, ofr)
    base, stride, n = _layout(view, layout)
    t = _sentinel_tensor(n, s16)
    with _chunk_env(variant):
        frames, total = ctx.decode_corpus_into(files, t, table, base, stride, s16=s16, host_threads=4, sample_rate=out_rate, mono=mono)
    assert total == int((och.astype(np.uint64) * ofr).sum())
    assert list(frames) == [int(table.frames[table.file == i].sum()) for i in range(len(files))]
    img = t.cpu().numpy()
    outs = []
    for i in range(len(table)):
        b, s, c, f = int(base[i]), int(stride[i]), int(och[i]), int(ofr[i])
        outs.append(np.stack([img[b + k * s:b + k * s + f] for k in range(c)]) if c else np.zeros((0, f), img.dtype))
    # every sample outside the written rows keeps its sentinel
    mask = np.ones(n, bool)
    for i in range(len(table)):
        b, s = int(base[i]), int(stride[i])
        for k in range(int(och[i])):
            mask[b + k * s:b + k * s + int(ofr[i])] = False
    rest = img[mask]
    assert (rest == 0x7FFF).all() if s16 else np.isnan(rest).all(), "a sentinel was overwritten"
    return table, outs, och, ofr


def _check_against_scipy(table, native, outs, out_rate, mono):
    worst = 0.0
    for i, y in enumerate(outs):
        x = native[i].astype(np.float64)
        rate = int(table.sample_rate[i])
        if x.shape[1] == 0:
            assert y.shape[1] == 0
            continue
        if out_rate in (0, rate):                             # a copy: bit for bit
            exp = _downmix_f32(native[i])[None] if mono else native[i]
            assert np.array_equal(y.view(np.uint32), exp.view(np.uint32)), "stream %d: the copy differs" % i
            continue
        if mono:
            x = x.mean(axis=0, keepdims=True)
        ref = ss.resample_poly(x, out_rate, rate, axis=1)
        assert ref.shape == y.shape, (i, ref.shape, y.shape)
        peak = float(np.abs(x).max())
        err = float(np.abs(y - ref).max())
        worst = max(worst, err / max(1.0, peak))
        assert err <= 2e-6 * max(1.0, peak), (i, rate, out_rate, err, peak)
        p_out = float((ref ** 2).mean())
        p_in = float((x ** 2).mean())
        if p_out > 0:
            p_err = max(float(((y - ref) ** 2).mean()), 1e-300)
            snr = 10 * np.log10(max(p_out, p_in) / p_err)
            assert snr >= 120.0, (i, rate, out_rate, snr)
            if p_out >= 0.01 * p_in:
                assert 10 * np.log10(p_out / p_err) >= 120.0, (i, rate, out_rate, p_out, p_in, p_err)
    print("max-abs error / max(1, peak): %.3g" % worst)


@pytest.mark.parametrize("variant", ["default", "fused"])
@pytest.mark.parametrize("out_rate,mono", TARGETS)
def test_resampled_equals_resample_poly(files, contexts, variant, out_rate, mono):
    ctx = contexts(variant)
    table, native = _native(ctx, variant, files)
    t2, outs, och, ofr = _resampled(ctx, variant, files, out_rate, mono)
    assert np.array_equal(t2.frames, table.frames)
    _check_against_scipy(table, native, outs, out_rate, mono)


def test_short_stream_uses_the_padding_on_both_sides(files):
    table = lib.corpus_streams(files)
    i = len(table) - 1
    assert int(table.sample_rate[i]) == 48000 and 0 < int(table.frames[i]) < 60     # 10 R / L = 60 input frames at 48k -> 8k
    assert int(table.frames[len(table) - 2]) == 0                                    # the headers-only file
    assert 16000 in set(int(r) for r in table.sample_rate) and {8000, 22050, 44100, 48000} <= set(int(r) for r in table.sample_rate)


@pytest.mark.parametrize("mono", [False, True])
def test_keep_rate_is_a_copy_or_the_float32_downmix(files, contexts, mono):
    ctx = contexts("default")
    table, native = _native(ctx, "default", files)
    _, outs, _, _ = _resampled(ctx, "default", files, 0, mono)
    _check_against_scipy(table, native, outs, 0, mono)


def test_s16_is_the_rule_on_the_float32_output(files, contexts):
    ctx = contexts("default")
    over = 0
    for out_rate, mono in [(16000, True), (48000, False)]:
        _, f32, _, _ = _resampled(ctx, "default", files, out_rate, mono)
        _, i16, _, _ = _resampled(ctx, "default", files, out_rate, mono, s16=True)
        for a, b in zip(f32, i16):
            assert np.array_equal(_s16(a), b), (out_rate, mono)
            over += int((np.abs(a) > 1.0).sum())
    # synth_codebooks peaks at 6.3 and keeps that at 48 kHz
    assert over > 0, "no output sample past full scale: saturation is not exercised"


@pytest.mark.parametrize("variant", ["default", "one_file_per_chunk", "host_entropy"])
def test_float32_is_the_same_in_every_variant_and_layout(files, contexts, variant):
    """The resampled output depends on the decoded samples only. The decoded samples themselves can differ in the last bits
    between chunkings: a chunk of one file with one setup runs k_warp_synth, a chunk of many setups k_fused_synth. So the
    output must be bit-identical to the default variant's on every stream whose native decode is, bit-identical across
    layouts within the variant, and within the scipy bounds against the variant's own native decode everywhere."""
    ctx = contexts(variant)
    _, native = _native(ctx, variant, files)
    _, native0 = _native(contexts("default"), "default", files)
    same = [np.array_equal(a.view(np.uint32), b.view(np.uint32)) for a, b in zip(native, native0)]
    print("%s: %d of %d streams decode to the default variant's bits" % (variant, sum(same), len(same)))
    assert any(same)
    for out_rate, mono in [(16000, False), (22050, True)]:
        key = ("ref", out_rate, mono)
        if key not in _NATIVE:
            _NATIVE[key] = _resampled(contexts("default"), "default", files, out_rate, mono)[1]
        per_layout = {}
        for layout in ("padded", "packed", "odd"):
            table, per_layout[layout], _, _ = _resampled(ctx, variant, files, out_rate, mono, layout=layout)
        for i, a in enumerate(per_layout["packed"]):
            for layout in ("padded", "odd"):
                assert np.array_equal(a.view(np.uint32), per_layout[layout][i].view(np.uint32)), (variant, layout, out_rate, mono, i)
            if same[i]:
                assert np.array_equal(a.view(np.uint32), _NATIVE[key][i].view(np.uint32)), (variant, out_rate, mono, i)
        _check_against_scipy(table, native, per_layout["packed"], out_rate, mono)


def test_largest_table_2047_to_2048(contexts):
    ctx = contexts("default")
    one = [_rewrite("seed7", 2047, serial=0x7904)]
    table, native = _native(ctx, "default", one)
    assert int(table.sample_rate[0]) == 2047
    with pytest.raises(lib.PovError) as ei:                      # 2047 Hz to another target is past the cap
        ctx.decode_corpus_device(one, sample_rate=16000)
    assert ei.value.code == abi.POV_ERR_UNSUPPORTED
    _, outs, _, _ = _resampled(ctx, "default", one, 2048, False)
    _check_against_scipy(table, native, outs, 2048, False)


def test_decode_corpus_device_views(files, contexts):
    import torch
    ctx = contexts("default")
    for layout in ("padded", "packed"):
        out = ctx.decode_corpus_device(files, layout=layout, sample_rate=16000, mono=True, host_threads=4)
        assert out.sample_rate == 16000 and (out.out_channels == 1).all()
        assert np.array_equal(out.out_frames, lib.resampled_frames(out.table, 16000))
        if layout == "padded":
            assert out.pcm.shape == (len(out.table), 1, int(out.stride[0]))
        for i in range(len(out.table)):
            assert tuple(out.stream(i).shape) == (1, int(out.out_frames[i]))
    plain = ctx.decode_corpus_device(files, layout="packed")
    assert plain.sample_rate is None and plain.out_frames is None
    torch.cuda.synchronize()


def test_waits_for_the_callers_stream(files, contexts):
    import torch
    ctx = contexts("default")
    ref = _resampled(ctx, "default", files, 16000, True)[1]
    table = lib.corpus_streams(files)
    ofr = lib.resampled_frames(table, 16000)
    view = lib.StreamTable(table.file, np.ones(len(table), np.uint32), table.sample_rate, ofr)
    base, stride, n = _layout(view, "packed")
    t = torch.zeros(n, dtype=torch.float32, device="cuda:0")
    torch.cuda.synchronize()
    s = torch.cuda.Stream()
    with torch.cuda.stream(s):
        torch.cuda._sleep(2_000_000_000)
        t.fill_(float("nan"))
        ctx.decode_corpus_into(files, t, table, base, stride, host_threads=4, sample_rate=16000, mono=True)
        got = t.cpu().numpy()
    for i in range(len(table)):
        b, f = int(base[i]), int(ofr[i])
        assert np.array_equal(got[b:b + f].view(np.uint32), ref[i][0].view(np.uint32)), i


def test_device_to_host_bytes_are_the_status_words(files, contexts):
    ctx = contexts("default")
    packets = 0
    for data in files:
        po = lib.ParsedOgg(data, raw_packets=True)
        packets += sum(int(po.get(k)[1].n_packets) for k in range(po.n_streams) if po.get(k)[0].channels)
        po.close()
    for s16 in (False, True):
        h0, d0 = ctx.io_bytes()
        ctx.decode_corpus_device(files, layout="packed", s16=s16, sample_rate=16000, mono=True)
        h1, d1 = ctx.io_bytes()
        assert d1 - d0 == 4 * packets
        assert h1 > h0


def _raw_call(ctx, files, o, rs):
    arr = (C.c_char_p * len(files))(*files)
    lens = (C.c_size_t * len(files))(*[len(f) for f in files])
    return ctx.L.pov_decode_corpus_device_resampled(ctx.ctx, len(files), arr, lens, 2, C.byref(o) if o is not None else None,
                                                    C.byref(rs) if rs is not None else None, None, None)


@pytest.mark.parametrize("case", ["null_rs", "null_rates", "flags", "unsupported", "stride", "capacity", "overlap", "layout",
                                  "rate_mismatch"])
def test_refusals_launch_nothing(files, contexts, case):
    import torch
    ctx = contexts("default")
    table = lib.corpus_streams(files)
    out_rate = 16000
    ofr = lib.resampled_frames(table, out_rate)
    view = lib.StreamTable(table.file, table.channels, table.sample_rate, ofr)
    base, stride, n = _layout(view, "packed")
    k = int(np.argmax(ofr))
    rates = np.ascontiguousarray(table.sample_rate, np.uint32)
    layout = abi.POV_PCM_PLANAR
    rs = abi.pov_resample()
    rs.out_rate, rs.flags = out_rate, 0
    if case == "stride":
        stride = stride.copy(); stride[k] = ofr[k] - 1
    elif case == "capacity":
        n = int(base[-1] + table.channels[-1] * stride[-1]) - 1
    elif case == "overlap":
        base = base.copy(); base[k] = base[k - 1] + 1
    elif case == "layout":
        layout = abi.POV_PCM_INTERLEAVED
    elif case == "flags":
        rs.flags = 2
    elif case == "unsupported":
        rs.out_rate = 44057                                    # 44100 -> 44057: 44100 phases
    elif case == "rate_mismatch":
        rates = rates.copy(); rates[0] = 48000 if rates[0] != 48000 else 44100    # (fewer output frames: the regions still fit)
    t = _sentinel_tensor(n, False)
    if case != "null_rates":
        rs.sample_rate = rates.ctypes.data_as(C.POINTER(C.c_uint32))
    o, keep = _raw_device_pcm(table, t, base, stride, layout)
    launches = ctx.launch_count
    rc = _raw_call(ctx, files, o, None if case == "null_rs" else rs)
    msg = ctx.L.pov_last_error(ctx.ctx).decode()
    if case == "unsupported":
        assert rc == abi.POV_ERR_UNSUPPORTED, msg
        assert "stream 0" in msg and "44100 Hz -> 44057 Hz" in msg and "44100" in msg, msg
    else:
        assert rc == abi.POV_ERR_ARG, msg
    if case == "rate_mismatch":
        assert msg.startswith("file 0: ") and "sample rate" in msg, msg
    assert ctx.launch_count == launches
    assert bool(torch.isnan(t).all())


def test_errors_equal_the_host_decode_and_the_context_keeps_working(files, contexts):
    from tests.test_gpu_decode import _flip_bits_in_audio_packets
    ctx = contexts("default")
    good = [_load("stereo44khz"), _load("synth_two_submaps")] * 3
    with open(os.path.join(ROOT, "tests", "golden", "synth_bad_vq_book.ogg"), "rb") as f:
        candidates = [f.read()]
    rng = np.random.default_rng(2024)
    candidates += [_flip_bits_in_audio_packets(_load("stereo44khz"), rng, flips=40) for _ in range(16)]
    compared = 0
    for bad in candidates:
        corpus = good[:3] + [bad] + good[3:]
        try:
            ctx.decode_corpus_pcm(corpus, lambda i, pcm: False, host_threads=3)
            continue
        except lib.PovError as e:
            host = (e.code, e.msg)
        try:
            table = lib.corpus_streams(corpus)
        except lib.PovError as e:
            assert (e.code, e.msg) == host
            continue
        with pytest.raises(lib.PovError) as ei:
            ctx.decode_corpus_device(corpus, layout="packed", sample_rate=16000, mono=True, host_threads=3)
        assert (ei.value.code, ei.value.msg) == host
        compared += 1
    assert compared >= 1
    table, native = _native(ctx, "default", files)
    _, outs, _, _ = _resampled(ctx, "default", files, 16000, True)
    _check_against_scipy(table, native, outs, 16000, True)
