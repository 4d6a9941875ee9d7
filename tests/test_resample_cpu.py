"""The resampler's filter design and output sizes, without a GPU: pov_resample_filter against scipy's resample_poly design,
the polyphase indexing the kernel uses against resample_poly itself, and the pov_resample struct against the C compiler."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest
import scipy.signal as ss

from parseoggvorbis_b200 import abi, lib

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
RATIOS = [(44100, 16000), (48000, 16000), (22050, 16000), (8000, 16000), (11025, 48000), (44100, 48000), (16000, 44100),
          (2047, 2048)]


@pytest.mark.parametrize("in_rate,out_rate", RATIOS)
def test_taps_equal_scipys_design_within_one_ulp(in_rate, out_rate):
    L, M, hl, taps = lib.resample_filter(in_rate, out_rate)
    R = max(L, M)
    assert hl == 10 * R and taps.dtype == np.float32 and len(taps) == 2 * hl + 1
    ref = np.float32(ss.firwin(2 * hl + 1, 1.0 / R, window=("kaiser", 5.0)) * L)
    ulps = np.abs(taps.view(np.int32).astype(np.int64) - ref.view(np.int32).astype(np.int64))
    assert int(ulps.max()) <= 1


def test_ratio_is_reduced_by_the_gcd():
    assert lib.resample_filter(44100, 16000)[:3] == (160, 441, 4410)
    assert lib.resample_filter(48000, 16000)[:3] == (1, 3, 30)
    assert lib.resample_filter(8000, 16000)[:3] == (2, 1, 20)
    assert lib.resample_filter(44100, 48000)[:3] == (160, 147, 1600)
    assert lib.resample_filter(11025, 48000)[:3] == (640, 147, 6400)
    assert lib.resample_filter(2047, 2048)[:3] == (2048, 2047, 20480)


def test_equal_rates_are_a_copy():
    for rate in (8000, 44100, 2047):
        L, M, hl, taps = lib.resample_filter(rate, rate)
        assert (L, M, hl, len(taps)) == (1, 1, 0, 0)
    assert lib.resample_filter(44100, 0)[:3] == (1, 1, 0)        # out_rate 0: the stream keeps its rate


@pytest.mark.parametrize("in_rate,out_rate,phases", [(2048, 2049, 2049), (44056, 48000, 6000)])
def test_ratios_past_the_cap_are_unsupported(in_rate, out_rate, phases):
    up, down, hl = C.c_uint32(0), C.c_uint32(0), C.c_uint32(0)
    rc = lib.load().pov_resample_filter(in_rate, out_rate, C.byref(up), C.byref(down), C.byref(hl), None, 0)
    assert rc == abi.POV_ERR_UNSUPPORTED and max(up.value, down.value) == phases
    with pytest.raises(lib.PovError) as ei:
        lib.resample_filter(in_rate, out_rate)
    assert ei.value.code == abi.POV_ERR_UNSUPPORTED


def test_bad_arguments():
    L = lib.load()
    up, down, hl = C.c_uint32(0), C.c_uint32(0), C.c_uint32(0)
    assert L.pov_resample_filter(0, 16000, C.byref(up), C.byref(down), C.byref(hl), None, 0) == abi.POV_ERR_ARG
    small = np.zeros(60, np.float32)                                  # 48k -> 16k needs 61 taps
    assert L.pov_resample_filter(48000, 16000, C.byref(up), C.byref(down), C.byref(hl),
                                 small.ctypes.data_as(C.POINTER(C.c_float)), len(small)) == abi.POV_ERR_ARG


@pytest.mark.parametrize("out_rate", [16000, 48000, 22050, 8000, 0])
def test_resampled_frames_equal_resample_polys_length(out_rate):
    rates = np.array([8000, 16000, 22050, 44100, 48000, 44100, 48000, 11025], np.uint32)
    frames = np.array([0, 1, 2, 1000, 59, 4097, 1, 333], np.uint64)
    table = lib.StreamTable(np.arange(len(rates), dtype=np.uint32), np.ones(len(rates), np.uint32), rates, frames)
    got = lib.resampled_frames(table, out_rate)
    assert got.dtype == np.uint64
    for r, f, g in zip(rates, frames, got):
        want = int(f) if out_rate == 0 else len(ss.resample_poly(np.zeros(int(f)), out_rate, int(r)))
        assert int(g) == want, (r, f, out_rate)


def _polyphase(x, L, M, hl, taps):
    """The kernel's indexing in float64: y[j] = sum_k x[floor((j M + hl) / L) - k] h[(j M + hl) mod L + k L]."""
    N, n = len(taps), len(x)
    K = -(-N // L)
    out = np.zeros(-(-n * L // M))
    for j in range(len(out)):
        p = j * M + hl
        b, ph = p // L, p % L
        for k in range(K):
            i, t = b - k, ph + k * L
            if t < N and 0 <= i < n:
                out[j] += x[i] * float(taps[t])
    return out


@pytest.mark.parametrize("in_rate,out_rate,frames", [(48000, 8000, 40), (44100, 16000, 300), (8000, 48000, 50),
                                                     (44100, 48000, 200), (22050, 16000, 1)])
def test_polyphase_indexing_equals_resample_poly(in_rate, out_rate, frames):
    rng = np.random.default_rng(frames)
    x = rng.uniform(-0.9, 0.9, frames)
    L, M, hl, taps = lib.resample_filter(in_rate, out_rate)
    ref = ss.resample_poly(x, out_rate, in_rate, window=("kaiser", 5.0))
    got = _polyphase(x, L, M, hl, taps)
    assert got.shape == ref.shape
    # the taps are float32 here and float64 in scipy: agreement to float32 precision proves the indexing
    assert float(np.abs(got - ref).max()) <= 1e-6


def test_struct_size_matches_c_compiler(tmp_path):
    src = tmp_path / "s.c"
    src.write_text('#include <stdio.h>\n#include "pov_synth.h"\nint main(){printf("%zu %zu\\n", sizeof(pov_resample), '
                   'sizeof(pov_device_pcm)); return POV_RESAMPLE_MONO == 1 && POV_RESAMPLE_MAX_PHASES == 2048 ? 0 : 1;}\n')
    exe = tmp_path / "s.bin"
    subprocess.check_call(["gcc", "-I", os.path.join(ROOT, "include"), str(src), "-o", str(exe)])
    a, b = subprocess.check_output([str(exe)], text=True).split()
    assert int(a) == C.sizeof(abi.pov_resample) and int(b) == C.sizeof(abi.pov_device_pcm)
    assert abi.POV_RESAMPLE_MONO == 1 and abi.POV_RESAMPLE_MAX_PHASES == 2048
