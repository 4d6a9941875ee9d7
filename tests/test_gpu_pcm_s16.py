"""Signed 16-bit PCM output (POV_PCM_S16): the kernels convert at their PCM store, so every path's int16 output must equal the
conversion rule applied to the float32 output of the same path on the same batch, bit for bit."""
import ctypes as C
import dataclasses
import os
import subprocess

import numpy as np
import pytest

from parseoggvorbis_b200 import abi, workloads
from tests.conftest import SYNTHETIC

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
FIX = {"stereo44khz": "test.stereo44khz.ogg", "mono44khz": "test.mono44khz.ogg"}
FIX.update({n: n + ".ogg" for n in SYNTHETIC})
WARP_PAIRS = [(256, 512), (256, 1024), (256, 2048), (512, 1024), (512, 2048), (1024, 2048)]
LAYOUTS = [abi.POV_PCM_PLANAR, abi.POV_PCM_INTERLEAVED]


def to_s16(x):
    """The conversion rule of include/pov_synth.h (np.rint rounds half to even)."""
    x = np.asarray(x)
    return np.where(np.isnan(x), 0, np.clip(np.rint(x.astype(np.float64) * 32768), -32768, 32767)).astype(np.int16)


def _load(name):
    with open(os.path.join(ROOT, "tests", "golden", FIX[name]), "rb") as f:
        return f.read()


def test_decoded_s16_struct_size_matches_c_compiler(tmp_path):
    src = tmp_path / "s.c"
    src.write_text('#include <stdio.h>\n#include "pov_synth.h"\nint main(){printf("%zu\\n", sizeof(pov_decoded_s16)); return 0;}\n')
    exe = tmp_path / "s.bin"
    subprocess.check_call(["gcc", "-I", os.path.join(ROOT, "include"), str(src), "-o", str(exe)])
    assert int(subprocess.check_output([str(exe)], text=True)) == C.sizeof(abi.pov_decoded_s16)


def test_to_s16_reference_rule():
    x = np.array([0.0, 0.5 / 32768, 1.5 / 32768, -0.5 / 32768, -1.5 / 32768, 1.0, -1.0, 2.0, -2.0, np.inf, -np.inf, np.nan],
                 np.float32)
    assert to_s16(x).tolist() == [0, 0, 2, 0, -2, 32767, -32768, 32767, -32768, 32767, -32768, 0]


# ---- GPU ----------------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def ctx():
    from parseoggvorbis_b200.lib import SynthContext
    c = SynthContext(0)
    yield c
    c.close()


def _run_both(ctx, setup, batch, kernel, staged=False):
    """Upload `batch` as float32 and as POV_PCM_S16, run both on the same path, return (float32 arena, int16 arena)."""
    sid = ctx.register_setup(setup)
    out = []
    for layout in (batch.pcm_layout, batch.pcm_layout | abi.POV_PCM_S16):
        b = dataclasses.replace(batch, streams=batch.streams.copy(), pcm_layout=layout)
        b.streams["setup_id"] = sid
        bh = ctx.upload(b)
        if staged:
            ctx.run_staged(bh)
        else:
            assert ctx.kernel_name(bh) == kernel
            ctx.run(bh)
        pcm = ctx.fetch_pcm(bh)
        assert pcm.dtype == (np.int16 if layout & abi.POV_PCM_S16 else np.float32)
        assert not ctx.status(bh).any()
        out.append(pcm.copy())
        bh.free()
    return out[0], out[1]


def _assert_same_path(ctx, setup, batch, kernel, staged=False):
    f32, s16 = _run_both(ctx, setup, batch, kernel, staged)
    assert np.array_equal(s16, to_s16(f32))
    assert np.abs(s16).max() >= 256          # real audio, not an all-zero arena
    return f32, s16


def _stereo_batch(bs, seed, packets=150):
    rng = np.random.default_rng(seed)
    setup = workloads.make_setup(2, bs, 22050, couplings=[(0, 1)])
    plans = [workloads.plan_stream(workloads.block_sequence(packets, rng, p_short=0.2), setup.blocksize, trim_last=int(rng.integers(0, 30)))
             for _ in range(3)]
    return setup, workloads.build_dense_batch(setup, plans, rng, p_unused=0.05)


@pytest.mark.gpu
@pytest.mark.parametrize("layout", LAYOUTS)
@pytest.mark.parametrize("bs", WARP_PAIRS)
def test_warp_kernel_s16_equals_rule_of_f32(ctx, bs, layout):
    setup, batch = _stereo_batch(bs, bs[0] + 5 * bs[1])
    _assert_same_path(ctx, setup, dataclasses.replace(batch, pcm_layout=layout), "k_warp_synth")


@pytest.mark.gpu
@pytest.mark.parametrize("layout", LAYOUTS)
def test_warp_kernel_s16_wide_floors(ctx, layout):
    """Floors of 33..64 posts: the kWide instantiations."""
    rng = np.random.default_rng(7003)
    for _ in range(50):
        setup = workloads.random_setup(rng, 2, max_posts=64, max_couplings=2, max_posts_short=32)
        if max(len(f.xs) for f in setup.floors) > 32 and len(setup.floors) <= 4 and len(setup.mappings) <= 4:
            break
    assert max(len(f.xs) for f in setup.floors) > 32
    batch = workloads.random_batch(setup, rng, streams=3, packets_per_stream=70)
    _assert_same_path(ctx, setup, dataclasses.replace(batch, pcm_layout=layout), "k_warp_synth")


@pytest.mark.gpu
@pytest.mark.parametrize("layout", LAYOUTS)
def test_warp_kernel_s16_config3_surround(ctx, layout):
    """5.1, two submaps, three coupling steps."""
    setup, batch = workloads.config3(P=200, streams=2, distinct=2, seed=1)
    _assert_same_path(ctx, setup, dataclasses.replace(batch, pcm_layout=layout), "k_warp_synth")


@pytest.mark.gpu
@pytest.mark.parametrize("layout", LAYOUTS)
@pytest.mark.parametrize("bs", [(64, 8192), (1024, 4096), (128, 128)])
def test_fused_kernel_s16_equals_rule_of_f32(ctx, bs, layout):
    """Block sizes outside the warp kernel: the vector (planar) and scalar (interleaved) stores of k_fused_synth."""
    setup, batch = _stereo_batch(bs, 3 * bs[0] + bs[1], packets=60)
    _assert_same_path(ctx, setup, dataclasses.replace(batch, pcm_layout=layout), "k_fused_synth")


@pytest.mark.gpu
@pytest.mark.parametrize("layout", LAYOUTS)
def test_fused_kernel_forced_s16(monkeypatch, layout):
    from parseoggvorbis_b200.lib import SynthContext
    monkeypatch.setenv("POV_KERNEL", "fused")
    c2 = SynthContext(0)
    try:
        setup, batch = workloads.config2(P=300, streams=3, distinct=3, seed=12)
        _assert_same_path(c2, setup, dataclasses.replace(batch, pcm_layout=layout), "k_fused_synth")
    finally:
        c2.close()


@pytest.mark.gpu
@pytest.mark.parametrize("layout", LAYOUTS)
def test_staged_path_s16_equals_rule_of_f32(ctx, layout):
    setup, batch = workloads.config2(P=120, streams=2, distinct=2, seed=13)
    _assert_same_path(ctx, setup, dataclasses.replace(batch, pcm_layout=layout), None, staged=True)


# ---- rounding, saturation, NaN --------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_saturation_and_round_half_even(ctx):
    """Spectra scaled by 128 put PCM far beyond ±1: both ends saturate, and the many samples whose x * 32768 lies exactly
    halfway between two integers round to the even one."""
    setup, batch = workloads.config2(P=600, streams=4, distinct=2, seed=31)
    batch = dataclasses.replace(batch, payload=batch.payload * np.float32(128))
    f32, s16 = _run_both(ctx, setup, batch, "k_warp_synth")
    assert np.array_equal(s16, to_s16(f32))
    assert np.mean(s16 == 32767) >= 0.01 and np.mean(s16 == -32768) >= 0.01
    y = f32.astype(np.float64) * 32768
    half = np.nonzero((y - np.floor(y) == 0.5) & (np.abs(y) < 32767))[0]      # (beyond the range the clip decides)
    assert len(half) >= 100, len(half)
    assert np.all(s16[half] % 2 == 0)
    assert np.all(np.abs(s16[half].astype(np.float64) - y[half]) == 0.5)


@pytest.mark.gpu
def test_nan_and_inf_spectra(ctx):
    """NaN / ±inf in one packet's spectrum (ordinary arithmetic: no status bit): NaN samples become 0, infinite and huge
    ones saturate, and every sample outside the two chunks that packet reaches is what the clean batch gives."""
    setup, batch = workloads.config2(P=200, streams=1, distinct=1, seed=14)
    clean_f32, clean_s16 = _run_both(ctx, setup, batch, "k_warp_synth")
    pk = batch.packets
    spec = batch.payload.copy()
    bad = {40: np.nan, 90: np.inf, 140: -np.inf}
    for p, v in bad.items():
        spec[int(pk["spec_off"][p]) + 3] = v
    spec[int(pk["spec_off"][170]) + 5] = 1e30          # finite, but far beyond the int16 range once transformed
    spec[int(pk["spec_off"][170]) + 9] = -1e30
    f32, s16 = _run_both(ctx, setup, dataclasses.replace(batch, payload=spec), "k_warp_synth")
    assert np.array_equal(s16, to_s16(f32))
    assert np.isnan(f32).any()
    assert np.all(s16[np.isnan(f32)] == 0)
    assert np.all(s16[f32 == np.inf] == 32767) and np.all(s16[f32 == -np.inf] == -32768)
    # the samples of packets p and p + 1 (a frame reaches two emitted chunks), both channels
    frames = int(batch.streams["pcm_frames"][0])
    touched = np.zeros(frames, bool)
    for p in list(bad) + [170]:
        for q in (p, p + 1):
            touched[int(pk["pcm_off"][q]):int(pk["pcm_off"][q]) + int(pk["emit_frames"][q])] = True
    touched = np.tile(touched, 2)
    assert np.array_equal(s16[~touched], clean_s16[~touched])
    assert (s16[touched] != clean_s16[touched]).any()
    chunk = np.zeros(frames, bool)
    for q in (170, 171):
        chunk[int(pk["pcm_off"][q]):int(pk["pcm_off"][q]) + int(pk["emit_frames"][q])] = True
    huge = s16[np.tile(chunk, 2)]
    assert (huge == 32767).any() and (huge == -32768).any()


# ---- whole files and the corpus ---------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("name", ["stereo44khz", "mono44khz"] + list(SYNTHETIC))
def test_decode_ogg_s16(ctx, golden, name):
    data = _load(name)
    f32, sr, npk = ctx.decode_ogg(data)
    s16, sr2, npk2 = ctx.decode_ogg(data, s16=True)
    assert (sr, npk) == (sr2, npk2) and s16.dtype == np.int16 and s16.shape == f32.shape
    assert np.array_equal(s16, to_s16(f32))
    ref = to_s16(golden[name]["pcm"])
    assert ref.shape == s16.shape
    assert np.abs(s16.astype(np.int32) - ref).max() <= 1


CORPUS = ["stereo44khz", "mono44khz", "synth_res0_mono", "synth_two_submaps", "synth_surround51"]


@pytest.mark.gpu
def test_corpus_s16_equals_rule_of_f32_corpus(ctx):
    files = [_load(CORPUS[i % len(CORPUS)]) for i in range(150)]
    got_f, got_s = [], []

    def sink_f(i, pcm):
        got_f.append((i, pcm.copy()))
        return False

    def sink_s(i, pcm):
        got_s.append((i, pcm.copy()))
        return False
    io0 = ctx.io_bytes()
    frames_f, total_f, _ = ctx.decode_corpus_pcm(files, sink_f, host_threads=4)
    io1 = ctx.io_bytes()
    frames_s, total_s, sum_s = ctx.decode_corpus_pcm(files, sink_s, host_threads=4, s16=True)
    io2 = ctx.io_bytes()
    assert [i for i, _ in got_s] == [i for i, _ in got_f] == list(range(150))
    for (_, a), (_, b) in zip(got_f, got_s):
        assert b.dtype == np.int16 and np.array_equal(b, to_s16(a))
    assert np.array_equal(frames_f, frames_s) and total_f == total_s
    assert sum_s == sum(int(b.astype(np.int64).sum()) for _, b in got_s)
    d2h_f, d2h_s = io1[1] - io0[1], io2[1] - io1[1]
    assert d2h_f - d2h_s == 2 * total_f
    assert io1[0] - io0[0] == io2[0] - io1[0]
    # without a sink: the same counts and sum
    frames_n, total_n, sum_n = ctx.decode_corpus(files, host_threads=4, s16=True)
    assert np.array_equal(frames_n, frames_s) and total_n == total_s and sum_n == sum_s


@pytest.mark.gpu
def test_corpus_s16_sink_stops_the_decode(ctx):
    from parseoggvorbis_b200.lib import PovError
    files = [_load("mono44khz")] * 200
    calls = []

    def sink(i, pcm):
        calls.append(i)
        return i == 70
    with pytest.raises(PovError) as ei:
        ctx.decode_corpus_pcm(files, sink, host_threads=3, s16=True)
    assert "gotPcmData" in str(ei.value) and calls == list(range(71))
    f, t, s = ctx.decode_corpus(files, host_threads=3, s16=True)          # the context keeps working
    assert len(f) == 200 and t > 0 and s != 0


# ---- validation -----------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_s16_arguments_are_validated(ctx):
    from parseoggvorbis_b200.lib import PovError
    setup, batch = workloads.config2(P=16)
    batch.streams["setup_id"] = ctx.register_setup(setup)
    b16 = dataclasses.replace(batch, pcm_layout=abi.POV_PCM_PLANAR | abi.POV_PCM_S16)
    bh = ctx.upload(b16)
    ctx.run(bh)
    f32 = np.empty(batch.pcm_floats, np.float32)
    rc = ctx.L.pov_batch_fetch_pcm(ctx.ctx, bh.h, f32.ctypes.data_as(C.POINTER(C.c_float)), batch.pcm_floats, 1)
    assert rc == abi.POV_ERR_ARG
    with pytest.raises(PovError):
        ctx._check(rc)
    assert ctx.fetch_pcm_s16(bh).dtype == np.int16
    bh.free()
    bh = ctx.upload(batch)
    ctx.run(bh)
    with pytest.raises(PovError):
        ctx.fetch_pcm_s16(bh)
    bh.free()
    for layout in (2, 0x200, 2 | abi.POV_PCM_S16):
        with pytest.raises(PovError):
            ctx.upload(dataclasses.replace(batch, pcm_layout=layout))
    with pytest.raises(ValueError):
        ctx.decode_ogg(_load("mono44khz"), debug_out="x.dump", s16=True)
