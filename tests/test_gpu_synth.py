"""GPU parity tests: the CUDA path (through the C ABI) against the reference's golden dumps and the pinned oracle.

Tolerances (BASELINE.json north_star): floor1 integer stages, after_residue, after_envelope bit-exact;
pcm_after_mdct and PCM max-abs <= 1e-5 and SNR >= 120 dB.
"""
import numpy as np
import pytest

from parseoggvorbis_b200 import abi, workloads
from tests import oracle_binding as ob

pytestmark = pytest.mark.gpu

TOL_ABS = 1e-5
TOL_SNR = 120.0


@pytest.fixture(scope="module")
def ctx():
    from parseoggvorbis_b200.lib import SynthContext
    c = SynthContext(0)
    yield c
    c.close()


def _assert_float_parity(test, ref, what):
    test = np.asarray(test)
    ref = np.asarray(ref)
    assert test.shape == ref.shape, what
    d = float(np.abs(test - ref).max()) if test.size else 0.0
    # north_star's literal bound, the one the reference harness uses (compare-debug-out.py:90): the synthetic workloads
    # are audio-like (workloads.gen_ys), so their PCM sits inside [-1, 1] like the fixtures' and no scaling is needed.
    assert d <= TOL_ABS, (what, d, float(np.abs(ref).max()) if ref.size else 0.0)
    if np.any(ref):
        s = ob.snr_db(test, ref)
        assert s >= TOL_SNR, (what, s)


def _iter_cp(g):
    off_half = off_full = 0
    C = int(g["channels"])
    for p, n in enumerate(g["blocksize"]):
        n = int(n)
        for c in range(C):
            yield p, c, n, off_half, off_full
            off_half += n // 2
            off_full += n


@pytest.mark.parametrize("name", ["stereo44khz", "mono44khz"])
def test_golden_staged_every_stage(ctx, golden, name):
    """Config 1 (device part): every intermediate the reference dumps, from the same ys + after_residue."""
    g = golden[name]
    setup, batch = workloads.golden_setup_and_batch(g)
    sid = ctx.register_setup(setup)
    batch.streams["setup_id"] = sid
    bh = ctx.upload(batch)
    ctx.run_staged(bh)
    pcm = ctx.fetch_pcm(bh).reshape(setup.channels, -1)
    assert not ctx.status(bh).any()
    table = np.load(__import__("os").path.join(ob.ROOT, "tests", "golden", "inverse_db_table.npy"))
    for p, c, n, oh, of in _iter_cp(g):
        env = ctx.fetch_stage(bh, p, c, abi.POV_STAGE_AFTER_ENVELOPE, n // 2)
        assert np.array_equal(env, g["after_envelope"][oh:oh + n // 2]), (p, c)
        if p % 7 == 0 or n == 256:
            mdct = ctx.fetch_stage(bh, p, c, abi.POV_STAGE_PCM_AFTER_MDCT, n)
            _assert_float_parity(mdct, g["pcm_after_mdct"][of:of + n], ("pcm_after_mdct", p, c))
        if g["floor_used"][p, c]:
            k = int(g["floor_nposts"][g["floor_number"][p, c]])
            assert np.array_equal(ctx.fetch_stage(bh, p, c, abi.POV_STAGE_FINAL_YS, k), g["final_ys"][p, c, :k]), (p, c)
            assert np.array_equal(ctx.fetch_stage(bh, p, c, abi.POV_STAGE_STEP2_FLAG, k).astype(bool), g["step2_flag"][p, c, :k])
            fl = ctx.fetch_stage(bh, p, c, abi.POV_STAGE_FLOOR, n)
            assert np.array_equal(fl, g["floor"][of:of + n]), (p, c)
            fo = ctx.fetch_stage(bh, p, c, abi.POV_STAGE_FLOOR_OUTPUTS, n)
            assert np.array_equal(fo.view(np.uint32), table[g["floor"][of:of + n]].view(np.uint32))
    _assert_float_parity(pcm, g["pcm"], "pcm")
    bh.free()


@pytest.mark.parametrize("name", ["stereo44khz", "mono44khz"])
def test_golden_fused_pcm(ctx, golden, name):
    g = golden[name]
    setup, batch = workloads.golden_setup_and_batch(g)
    batch.streams["setup_id"] = ctx.register_setup(setup)
    bh = ctx.upload(batch)
    ctx.run(bh)
    fused = ctx.fetch_pcm(bh).reshape(setup.channels, -1)
    assert not ctx.status(bh).any()
    _assert_float_parity(fused, g["pcm"], "pcm")
    ctx.run_staged(bh)
    staged = ctx.fetch_pcm(bh).reshape(setup.channels, -1)
    # the staged path rounds its twiddles straight from float64 tables, the fused kernel derives part of them by
    # one extra float32 multiplication: same algorithm, last-ulp differences
    _assert_float_parity(fused, staged, "fused vs staged")
    bh.free()


def _check_against_oracle(ctx, setup, batch, stages=False):
    batch.streams["setup_id"] = ctx.register_setup(setup)
    bh = ctx.upload(batch)
    ctx.run(bh)
    fused = ctx.fetch_pcm(bh)
    st = ctx.status(bh)
    sid = batch.streams["setup_id"].copy()
    batch.streams["setup_id"] = 0
    if stages:
        ref, rst, cap = ob.synth_batch([setup], batch, imdct="fast", capture=True)
    else:
        ref, rst = ob.synth_batch([setup], batch, imdct="fast")
    batch.streams["setup_id"] = sid
    assert np.array_equal(st, rst)
    _assert_float_parity(fused, ref, "pcm vs oracle")
    if stages:
        ctx.run_staged(bh)
        staged = ctx.fetch_pcm(bh)
        _assert_float_parity(fused, staged, "fused vs staged")
        C = setup.channels
        flag_of_mode = np.asarray([m.blockflag for m in setup.modes])
        n_of = np.asarray(setup.blocksize)[flag_of_mode[batch.packets["mode"].astype(int)]]
        for p in range(0, len(batch.packets), max(1, len(batch.packets) // 40)):
            n = int(n_of[p])
            for c in range(C):
                env = ctx.fetch_stage(bh, p, c, abi.POV_STAGE_AFTER_ENVELOPE, n // 2)
                assert np.array_equal(env, cap["after_envelope"][p, c, :n // 2]), (p, c)
                mdct = ctx.fetch_stage(bh, p, c, abi.POV_STAGE_PCM_AFTER_MDCT, n)
                _assert_float_parity(mdct, cap["pcm_after_mdct"][p, c, :n], ("mdct", p, c))
    bh.free()
    return fused


def test_config2_stereo_mixed_blocks(ctx):
    setup, batch = workloads.config2(P=600, streams=3, distinct=3, seed=0)
    _check_against_oracle(ctx, setup, batch, stages=True)


def test_config3_5_1_coupling_order(ctx):
    setup, batch = workloads.config3(P=200, streams=2, distinct=2, seed=1)
    _check_against_oracle(ctx, setup, batch, stages=True)


@pytest.mark.parametrize("bs", [(256, 2048), (512, 1024), (64, 8192), (128, 128), (1024, 4096), (256, 512), (1024, 2048)])
def test_config4_mono_clips_blocksizes(ctx, bs):
    setup, batch = workloads.config4(clips=12, packets_per_clip=40, blocksizes=bs)
    _check_against_oracle(ctx, setup, batch, stages=(bs == (512, 1024)))


def test_interleaved_layout(ctx):
    setup, planar = workloads.config2(P=120, seed=4)
    rng = np.random.default_rng(4)
    plans = [workloads.plan_stream(planar.packets["mode"].copy(), setup.blocksize)]
    inter = workloads.build_dense_batch(setup, plans, rng, pcm_layout=abi.POV_PCM_INTERLEAVED)
    sid = ctx.register_setup(setup)
    inter.streams["setup_id"] = sid
    bh = ctx.upload(inter)
    ctx.run(bh)
    a = ctx.fetch_pcm(bh).reshape(-1, setup.channels)
    inter.pcm_layout = abi.POV_PCM_PLANAR
    bh2 = ctx.upload(inter)
    ctx.run(bh2)
    b = ctx.fetch_pcm(bh2).reshape(setup.channels, -1)
    assert np.array_equal(a.T, b)
    bh.free(); bh2.free()


def test_run_length_independence(ctx, monkeypatch):
    """Halo re-computation: PCM must not depend on how a stream is cut into runs (trimmed last packet included)."""
    setup, _ = workloads.config2(P=8)
    rng = np.random.default_rng(11)
    plan = workloads.plan_stream(workloads.block_sequence(300, rng), setup.blocksize, trim_last=100)
    batch = workloads.build_dense_batch(setup, [plan], rng)
    out = _check_against_oracle(ctx, setup, batch)
    from parseoggvorbis_b200.lib import SynthContext
    for rl in ("2", "5", "64"):
        monkeypatch.setenv("POV_RUN_LEN", rl)
        c2 = SynthContext(0)
        batch.streams["setup_id"] = c2.register_setup(setup)
        bh = c2.upload(batch)
        c2.run(bh)
        assert np.array_equal(c2.fetch_pcm(bh), out), rl
        bh.free(); c2.close()


def test_mdct_backward_dropin_all_sizes(ctx, golden):
    rng = np.random.default_rng(9)
    for n in (64, 128, 256, 512, 1024, 2048, 4096, 8192):
        x = rng.standard_normal((5, n // 2)).astype(np.float32)
        y = ctx.mdct_backward(x)
        for i in range(5):
            ref = ob.imdct(x[i], "closed")
            assert ob.snr_db(y[i], ref) >= TOL_SNR, n
            assert np.abs(y[i] - ref).max() <= 1e-5 * max(1.0, np.abs(ref).max()), n
            assert ob.snr_db(y[i], ob.vorbis_imdct(x[i])) >= TOL_SNR, n        # the reference's transform
    # the reference's own mdct_backward, as its dump of the bundled stereo fixture records it
    for n, x, ref in ob.dump_mdct_pairs(golden["stereo44khz"]):
        if np.any(x):
            assert ob.snr_db(ctx.mdct_backward(x[None])[0], ref) >= TOL_SNR, n


def test_error_status_matches_reference_checks(ctx):
    """Packets that trip the reference's fatal CHECKs (hpp:536, hpp:587) are reported per packet, not decoded."""
    setup, batch = workloads.config2(P=40, seed=3)
    ys = batch.ys.copy()
    pk = batch.packets
    # packet 5: huge coded value on a late post -> final Y far above range -> floor >= 256
    p = 5
    posts = 29 if pk["mode"][p] else 9
    ys[int(pk["ys_off"][p]) + posts - 1] = 5000
    # packet 9: first two posts maximal, third pushes predicted range check through a wrapped value
    p2 = 9
    ys[int(pk["ys_off"][p2]) + 2] = 60000
    batch.ys = ys
    sid = ctx.register_setup(setup)
    batch.streams["setup_id"] = sid
    bh = ctx.upload(batch)
    ctx.run(bh)
    st = ctx.status(bh)
    batch.streams["setup_id"] = 0
    _, rst = ob.synth_batch([setup], batch, imdct="fast")
    assert st[p] != 0 and st[p2] != 0
    assert np.array_equal(st != 0, rst != 0)
    assert np.array_equal(st, rst)
    from parseoggvorbis_b200.lib import PovError
    with pytest.raises(PovError):
        ctx.status(bh, check=True)
    bh.free()


def test_descriptor_validation_errors(ctx):
    from parseoggvorbis_b200.lib import PovError
    setup, batch = workloads.config2(P=16)
    batch.streams["setup_id"] = ctx.register_setup(setup)
    bad = abi.Batch(batch.streams.copy(), batch.packets.copy(), batch.ys, batch.payload, batch.pcm_floats)
    bad.packets["mode"][3] = 7
    with pytest.raises(PovError):
        ctx.upload(bad)
    bad = abi.Batch(batch.streams.copy(), batch.packets.copy(), batch.ys, batch.payload, batch.pcm_floats)
    bad.packets["emit_frames"][1] = 5000
    with pytest.raises(PovError):
        ctx.upload(bad)
    s2 = workloads.make_setup(2)
    s2.floors[0] = abi.Floor1([0, 128, 14, 14], 4)       # duplicate X
    with pytest.raises(PovError):
        ctx.register_setup(s2)


@pytest.mark.gpu
@pytest.mark.parametrize("seed", range(12))
def test_random_setups_against_oracle(ctx, seed):
    """Random floors (2..32 posts, multipliers 1..4, random X lists), submaps with their own floors, several modes and
    mappings, coupling graphs with shared channels, unused channels: the persistent warp kernel (and, for seeds whose
    setup it does not take, the generic kernel) against the CPU oracle, status words included."""
    rng = np.random.default_rng(1000 + seed)
    C = int(rng.integers(1, 9))
    setup = workloads.random_setup(rng, C)
    batch = workloads.random_batch(setup, rng, streams=3, packets_per_stream=70)
    _check_against_oracle(ctx, setup, batch, stages=(seed % 4 == 0))


@pytest.mark.gpu
@pytest.mark.parametrize("seed", range(8))
def test_floors_of_up_to_64_posts_stay_on_the_warp_kernel(ctx, seed):
    """libvorbis' high-quality setups carry more than 32 floor posts (up to 65 by VIF_POSIT): floors of 33..64 posts take the
    warp kernel's wide path (64-bit step-2 masks, 72-byte Y records, runs of <= 16 packets) and must equal the oracle —
    PCM, status words and, on the staged kernels, after_envelope — like the narrow ones."""
    rng = np.random.default_rng(7000 + seed)
    C = int(rng.integers(1, 4))
    for _ in range(50):                      # draw until a floor really has more than 32 posts
        setup = workloads.random_setup(rng, C, max_posts=64, max_couplings=2, max_posts_short=32)
        if max(len(f.xs) for f in setup.floors) > 32 and len(setup.floors) <= 4 and len(setup.mappings) <= 4:
            break
    assert max(len(f.xs) for f in setup.floors) > 32
    batch = workloads.random_batch(setup, rng, streams=3, packets_per_stream=70)
    batch.streams["setup_id"] = ctx.register_setup(setup)
    bh = ctx.upload(batch)
    assert ctx.kernel_name(bh) == "k_warp_synth", [len(f.xs) for f in setup.floors]
    bh.free()
    _check_against_oracle(ctx, setup, batch, stages=(seed % 2 == 0))


@pytest.mark.gpu
def test_random_setups_take_the_warp_kernel(ctx):
    """Every setup the generator draws — 1..8 channels, up to 64 posts per floor (libvorbis' long-block floors have up to
    65 values, of which the fast path holds 64), up to 5 coupling steps, 2-4 mappings — stays on k_warp_synth."""
    fallen = []
    for seed in range(12):
        rng = np.random.default_rng(1000 + seed)
        C = int(rng.integers(1, 9))
        setup = workloads.random_setup(rng, C, max_posts=64 if seed % 2 else 32)
        batch = workloads.random_batch(setup, rng, streams=1, packets_per_stream=8)
        batch.streams["setup_id"] = ctx.register_setup(setup)
        bh = ctx.upload(batch)
        if ctx.kernel_name(bh) != "k_warp_synth":
            fallen.append((seed, C, [len(f.xs) for f in setup.floors], [len(m.couplings) for m in setup.mappings]))
        bh.free()
    assert not fallen, fallen


@pytest.mark.gpu
def test_full_size_properties_config2(ctx, monkeypatch):
    """BASELINE.json configs[1] at its full per-stream size (4096 packets, mixed blocks): properties that do not need
    the oracle at full size — replicated streams decode to bit-identical PCM wherever they sit in the arenas, the result
    does not depend on how streams are cut into runs, no packet reports a status — plus the oracle on one whole stream."""
    setup, batch = workloads.config2(P=4096, streams=8, distinct=4, seed=5)
    batch.streams["setup_id"] = ctx.register_setup(setup)
    bh = ctx.upload(batch)
    assert ctx.kernel_name(bh) == "k_warp_synth"
    ctx.run(bh)
    pcm = ctx.fetch_pcm(bh)
    assert not ctx.status(bh).any()
    per = int(batch.pcm_floats) // 2
    assert np.array_equal(pcm[:per], pcm[per:])                    # second replica of the 4 distinct streams
    st = batch.streams[:1].copy(); st["setup_id"] = 0
    sub = abi.Batch(st, batch.packets[:int(st["n_packets"][0])].copy(), batch.ys, batch.payload,
                    int(st["pcm_frames"][0]) * setup.channels)
    ref, _ = ob.synth_batch([setup], sub, imdct="fast")
    _assert_float_parity(pcm[:sub.pcm_floats], ref, "stream 0 vs oracle")
    from parseoggvorbis_b200.lib import SynthContext
    monkeypatch.setenv("POV_RUN_LEN", "13")
    c2 = SynthContext(0)
    batch.streams["setup_id"] = c2.register_setup(setup)
    bh2 = c2.upload(batch)
    c2.run(bh2)
    assert np.array_equal(c2.fetch_pcm(bh2), pcm)
    bh2.free(); c2.close(); bh.free()


@pytest.mark.gpu
def test_mixed_setups_in_one_batch(ctx):
    """Streams of different setups (stereo, 5.1, mono) in one batch: the warp kernel is launched once per setup;
    PCM and status against the oracle, and the edge cases of tiny streams (1 and 2 packets) ride along."""
    s2, b2 = workloads.config2(P=150, streams=2, distinct=2, seed=21)
    s3, b3 = workloads.config3(P=90, streams=1, distinct=1, seed=22)
    s4, b4 = workloads.config4(clips=5, packets_per_clip=33, seed=23)
    s5, b5 = workloads.config4(clips=2, packets_per_clip=1, seed=24)       # single-packet streams emit nothing (hpp:1021)
    s6, b6 = workloads.config2(P=2, streams=1, distinct=1, seed=25)
    ids = [ctx.register_setup(s) for s in (s2, s3, s4)]
    merged = b2
    merged.streams["setup_id"] = 0
    merged = workloads.concat_batches(merged, b3, 1)
    merged = workloads.concat_batches(merged, b4, 2)
    merged = workloads.concat_batches(merged, b5, 2)
    merged = workloads.concat_batches(merged, b6, 0)
    ref, rstatus = ob.synth_batch([s2, s3, s4], merged, imdct="fast")
    dev = merged
    dev.streams["setup_id"] = np.asarray(ids, np.uint32)[merged.streams["setup_id"]]
    bh = ctx.upload(dev)
    assert ctx.kernel_name(bh) == "k_warp_synth"
    n0 = ctx.launch_count
    ctx.run(bh)
    assert ctx.launch_count - n0 == 3                  # one persistent launch per setup
    pcm = ctx.fetch_pcm(bh)
    assert np.array_equal(ctx.status(bh), rstatus)
    _assert_float_parity(pcm, ref, "mixed setups vs oracle")
    bh.free()


@pytest.mark.gpu
def test_empty_batch_is_a_no_op(ctx):
    setup, batch = workloads.config2(P=4, seed=1)
    batch.streams["setup_id"] = ctx.register_setup(setup)
    empty = abi.Batch(batch.streams[:0].copy(), batch.packets[:0].copy(), batch.ys[:0], batch.payload[:0], 0)
    bh = ctx.upload(empty)
    ctx.run(bh)
    assert ctx.fetch_pcm(bh).size == 0
    bh.free()


@pytest.mark.gpu
@pytest.mark.parametrize("bs", [(256, 512), (256, 1024), (256, 2048), (512, 1024), (512, 2048), (1024, 2048)])
def test_warp_kernel_block_size_pairs_stereo(ctx, bs):
    """Every block-size pair the persistent warp kernel is instantiated for (radix-2 / radix-4 first passes for 512 and
    1024, several FFTs per warp for the smaller sizes): stereo with coupling, mixed blocks, trimmed last packet."""
    rng = np.random.default_rng(bs[0] * 7 + bs[1])
    setup = workloads.make_setup(2, bs, 22050, couplings=[(0, 1)])
    plans = [workloads.plan_stream(workloads.block_sequence(220, rng, p_short=0.15), setup.blocksize, trim_last=int(rng.integers(0, 30)))
             for _ in range(3)]
    batch = workloads.build_dense_batch(setup, plans, rng, p_unused=0.05)
    batch.streams["setup_id"] = ctx.register_setup(setup)
    bh = ctx.upload(batch)
    assert ctx.kernel_name(bh) == "k_warp_synth"
    bh.free()
    _check_against_oracle(ctx, setup, batch, stages=True)


@pytest.mark.gpu
@pytest.mark.parametrize("bs", [(256, 512), (512, 1024), (1024, 2048)])
def test_interleaved_layout_block_size_pairs(ctx, bs):
    """Interleaved PCM is a second instantiation of the warp kernel: it must equal the planar result bit for bit for the
    grouped small-block geometries too (several long FFTs per warp, strided stores)."""
    rng = np.random.default_rng(bs[0] + 3 * bs[1])
    setup = workloads.make_setup(2, bs, 22050, couplings=[(0, 1)])
    plans = [workloads.plan_stream(workloads.block_sequence(150, rng, p_short=0.2), setup.blocksize, trim_last=int(rng.integers(0, 30)))
             for _ in range(2)]
    out = {}
    for layout in (abi.POV_PCM_PLANAR, abi.POV_PCM_INTERLEAVED):
        batch = workloads.build_dense_batch(setup, plans, np.random.default_rng(11), pcm_layout=layout)
        batch.streams["setup_id"] = ctx.register_setup(setup)
        bh = ctx.upload(batch)
        assert ctx.kernel_name(bh) == "k_warp_synth"
        ctx.run(bh)
        out[layout] = (ctx.fetch_pcm(bh).copy(), batch.streams.copy())
        bh.free()
    planar, st = out[abi.POV_PCM_PLANAR]
    inter, _ = out[abi.POV_PCM_INTERLEAVED]
    for s in st:
        base, frames = int(s["pcm_base"]), int(s["pcm_frames"])
        a = planar[base:base + 2 * frames].reshape(2, frames)
        b = inter[base:base + 2 * frames].reshape(frames, 2)
        assert np.array_equal(a, b.T)
