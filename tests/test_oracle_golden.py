"""Pins the CPU oracle (oracle/synth_oracle.c) against the reference decoder's own output.

Goldens: tests/golden/*.npz = the reference's --debug_out dump of its two bundled fixtures (made by
tests/golden/make_golden.py from oracle/_ref/ours.bin). Tolerances are the reference harness' own
(tests/compare-debug-out.py:90-108: ints exact, floats abs < 1e-5) tightened per BASELINE.json: integer floor1
stages bit-exact; IMDCT/PCM max-abs <= 1e-5 and SNR >= 120 dB.
"""
import os

import numpy as np
import pytest

from parseoggvorbis_b200 import workloads
from tests import oracle_binding as ob

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
FIX = ["stereo44khz", "mono44khz"]


def _iter_channel_packets(g):
    """yield (packet, channel, n, offset into the per-(packet,channel) concatenations of length n/2 and n)."""
    off_half = off_full = 0
    C = int(g["channels"])
    for p, n in enumerate(g["blocksize"]):
        n = int(n)
        for c in range(C):
            yield p, c, n, off_half, off_full
            off_half += n // 2
            off_full += n


def test_inverse_db_table_matches_reference_header():
    gold = np.load(os.path.join(ROOT, "tests", "golden", "inverse_db_table.npy"))
    assert np.array_equal(ob.inverse_db_table().view(np.uint32), gold.view(np.uint32))


def test_neighbors_against_bruteforce_definition():
    # Utils.hpp:58-59, 89-90 definitions, checked on the fixtures' X lists
    for xs in (workloads.FIXTURE_XS_SHORT, workloads.FIXTURE_XS_LONG):
        lo, hi = ob.floor1_neighbors(xs)
        for i in range(2, len(xs)):
            below = [j for j in range(i) if xs[j] < xs[i]]
            above = [j for j in range(i) if xs[j] > xs[i]]
            assert lo[i] == max(below, key=lambda j: xs[j])
            assert hi[i] == min(above, key=lambda j: xs[j])


@pytest.mark.parametrize("name", FIX)
def test_floor1_bit_exact(golden, name):
    g = golden[name]
    table = ob.inverse_db_table()
    checked = 0
    for p, c, n, _, off_full in _iter_channel_packets(g):
        if not g["floor_used"][p, c]:
            continue
        fno = int(g["floor_number"][p, c])
        k = int(g["floor_nposts"][fno])
        xs = g["floor_xs"][fno, :k]
        st, fy, flag, fl, out = ob.floor1_curve(xs, int(g["floor_multipliers"][fno]), g["ys"][p, c, :k], n)
        assert st == 0
        assert np.array_equal(fy, g["final_ys"][p, c, :k]), (p, c)
        assert np.array_equal(flag, g["step2_flag"][p, c, :k]), (p, c)
        gold_floor = g["floor"][off_full:off_full + n]
        assert np.array_equal(fl, gold_floor), (p, c)
        assert np.array_equal(out.view(np.uint32), table[gold_floor].view(np.uint32))
        checked += 1
    assert checked >= 60


@pytest.mark.parametrize("name", FIX)
def test_imdct_against_reference_dump(golden, name):
    g = golden[name]
    worst_abs, worst_snr = 0.0, 1e9
    for p, c, n, off_half, off_full in _iter_channel_packets(g):
        if p % 3 and n == 2048:  # closed form is O(n^2): every third long packet is plenty
            continue
        x = g["after_envelope"][off_half:off_half + n // 2]
        ref = g["pcm_after_mdct"][off_full:off_full + n]
        if not np.any(x):
            assert not np.any(ref)
            continue
        for kind in ("closed", "fast"):
            y = ob.imdct(x, kind)
            worst_abs = max(worst_abs, float(np.abs(y - ref).max()))
            worst_snr = min(worst_snr, ob.snr_db(y, ref))
    assert worst_abs <= 1e-5, worst_abs
    assert worst_snr >= 120.0, worst_snr


def test_imdct_fast_vs_closed_all_sizes():
    rng = np.random.default_rng(5)
    for n in (64, 128, 256, 512, 1024, 2048, 4096, 8192):
        x = rng.standard_normal(n // 2).astype(np.float32)
        a, b = ob.imdct(x, "closed"), ob.imdct(x, "fast")
        assert ob.snr_db(b, a) >= 120.0, n
        # TDAC symmetries of the contract (SURVEY.md §8 a7)
        assert np.allclose(a[:n // 2], -a[:n // 2][::-1], atol=1e-4)
        assert np.allclose(a[n // 2:], a[n // 2:][::-1], atol=1e-4)


def test_vorbis_mdct_reproduces_the_reference_dumps(golden):
    """oracle/vorbis_mdct.c stands in for the reference's mdct_backward: it must give every transform the reference
    recorded in its dumps (after_envelope in, pcm_after_mdct out) bit for bit, at every block size they hold.
    (synth_shared_submap is the dump of libvorbis' own decoder, which differs from the reference here in the last bit.)"""
    from tests.conftest import SYNTHETIC
    names = ["stereo44khz", "mono44khz"] + [n for n in SYNTHETIC if n != "synth_shared_submap"]
    checked = {}
    for n, x, ref in ob.dump_mdct_pairs(*[golden[k] for k in names]):
        assert np.array_equal(ob.vorbis_imdct(x).view(np.uint32), ref.view(np.uint32)), n
        checked[n] = checked.get(n, 0) + 1
    assert sorted(checked) == [256, 512, 1024, 2048], checked


def test_imdct_closed_vs_reference_mdct_backward():
    rng = np.random.default_rng(6)
    for n in (64, 256, 2048, 8192):
        x = rng.standard_normal(n // 2).astype(np.float32)
        assert ob.snr_db(ob.imdct(x, "closed"), ob.vorbis_imdct(x)) >= 130.0, n


@pytest.mark.parametrize("name", FIX)
def test_whole_batch_against_reference_dump(golden, name):
    """floor -> coupling -> dot -> IMDCT -> window/OLA from the dump's ys + after_residue must reproduce the
    dump's after_envelope (bit-exact), pcm_after_mdct and final pcm (<=1e-5, >=120 dB)."""
    g = golden[name]
    setup, batch = workloads.golden_setup_and_batch(g)
    for kind in ("fast", "reference"):
        pcm, status, cap = ob.synth_batch([setup], batch, imdct=ob.golden_imdct(g) if kind == "reference" else kind, capture=True)
        assert not status.any()
        C = setup.channels
        for p, c, n, off_half, off_full in _iter_channel_packets(g):
            assert np.array_equal(cap["after_envelope"][p, c, :n // 2], g["after_envelope"][off_half:off_half + n // 2]), (p, c)
            d = np.abs(cap["pcm_after_mdct"][p, c, :n] - g["pcm_after_mdct"][off_full:off_full + n]).max()
            assert d <= 1e-5, (p, c, d)
        out = pcm.reshape(C, -1)
        gold = g["pcm"]
        assert out.shape == gold.shape
        assert np.abs(out - gold).max() <= 1e-5
        assert ob.snr_db(out, gold) >= 120.0
        if kind == "reference":
            # with the reference's own mdct_backward output (from its dump) plugged in, window + overlap-add must be bit-exact
            assert np.array_equal(out, gold)


def test_window_shapes():
    # hpp:837-862: zero outside the slopes, one between, power-complementary slopes
    w = ob.window(256, 2048, 1, 0, 1)
    assert np.all(w[:448] == 0) and w[448] > 0 and np.all(w[576:1024] == 1)
    s = ob.window(256, 2048, 0, 0, 0)
    assert np.allclose(s[:128] ** 2 + s[128:] ** 2, 1.0, atol=1e-6)
    l = ob.window(256, 2048, 1, 1, 1)
    assert np.allclose(l[:1024] ** 2 + l[1024:] ** 2, 1.0, atol=1e-6)
