"""Whole-file decode of seeded random Vorbis streams (tests/random_vorbis.py) on the GPU, against an independent packet
reader and the pinned CPU oracle: the device walk (k_packet_decode) and the residue stage (k_residue_apply) must give the
reader's model of `after_residue` bit for bit, the floor stage the oracle's floor1 of the reader's Ys, and the PCM of
every synthesis route the oracle's PCM of a dense batch built from the reader, the model and the host's packet framing."""
import ctypes as C

import numpy as np
import pytest

from parseoggvorbis_b200 import abi, lib
from tests import oracle_binding as ob
from tests import random_vorbis as rv
from tests.test_gpu_pcm_s16 import to_s16

pytestmark = pytest.mark.gpu
ROUTES = {"k_warp_synth", "k_fused_synth", "staged"}


@pytest.fixture(scope="module")
def ctx():
    c = lib.SynthContext(0)
    yield c
    c.close()


def _upload(ctx, cs, b):
    sid = C.c_uint32(0)
    ctx._check(ctx.L.pov_setup_register(ctx.ctx, C.byref(cs), C.byref(sid)))
    abi.pov_stream.from_address(C.addressof(b.streams.contents)).setup_id = sid.value
    h = C.c_void_p(None)
    ctx._check(ctx.L.pov_batch_upload(ctx.ctx, C.byref(b), C.byref(h)))
    return h


def _pcm(ctx, h, b):
    out = np.empty(int(b.pcm_floats), np.float32)
    ctx._check(ctx.L.pov_batch_fetch_pcm(ctx.ctx, h, out.ctypes.data_as(C.POINTER(C.c_float)), out.size, 1))
    return out


def _stage(ctx, h, p, c, stage, count, dtype):
    out = np.zeros(count, dtype)
    ctx._check(ctx.L.pov_batch_fetch_stage(ctx.ctx, h, p, c, stage, out.ctypes.data_as(C.c_void_p), out.nbytes))
    return out


def _status(ctx, h, n):
    st = np.zeros(n, np.uint32)
    ctx.L.pov_batch_status(ctx.ctx, h, st.ctypes.data_as(C.POINTER(C.c_uint32)), n)     # (non-zero words: POV_ERR_STREAM)
    return st


def _dense_reference(s, b_host, reads):
    """POV_INPUT_DENSE batch: packet framing (mode, window flags, emit_frames, pcm_off, stream table) from the host parse,
    floor flags and Ys from the reader, spectra from the model."""
    streams = rv.streams_array(b_host)
    streams["setup_id"] = 0
    pk = rv.packets_array(b_host)
    ys, spectra = [], []
    yo = so = 0
    for p, rp in enumerate(reads):
        pk["floor_used"][p] = sum(1 << c for c, y in enumerate(rp.ys) if y is not None)
        pk["ys_off"][p] = yo
        pk["spec_off"][p] = so
        for y in rp.ys:
            if y is not None:
                ys += y
                yo += len(y)
        sp = rv.model_after_residue(s, rp).ravel()
        spectra.append(sp)
        so += sp.size
    return abi.Batch(streams, pk, np.asarray(ys, np.uint16), np.concatenate(spectra), int(b_host.pcm_floats),
                     input_kind=abi.POV_INPUT_DENSE, pcm_layout=int(b_host.pcm_layout))


@pytest.mark.parametrize("name", rv.ALL_NAMES)
def test_device_walk_residue_floor_and_pcm_match_the_reader(ctx, name):
    st = rv.stream(name)
    s = st.setup
    reads = [rv.read_packet(s, rv.vw.write_audio_packet(s, pc)) for pc in st.packets]
    P = len(reads)
    po_host, po_raw = lib.ParsedOgg(st.data), lib.ParsedOgg(st.data, raw_packets=True)
    handles = []
    try:
        cs_h, b_h = po_host.get(0)
        _, ostatus = ob.synth_batch_raw(cs_h, b_h)
        cs, b = po_raw.get(0)
        assert b.input_kind == abi.POV_INPUT_PACKETS and b.n_packets == P
        # 1. device walk + residue + floor stages
        h = _upload(ctx, cs, b)
        handles.append(h)
        ctx._check(ctx.L.pov_batch_run_staged(ctx.ctx, h))
        assert np.array_equal(_status(ctx, h, P), ostatus)
        for p, rp in enumerate(reads):
            m = s.modes[rp.mode]
            n = s.blocksize[m.blockflag]
            want = rv.model_after_residue(s, rp)
            mp = s.mappings[m.mapping]
            for c in range(s.channels):
                got = _stage(ctx, h, p, c, abi.POV_STAGE_AFTER_RESIDUE, n // 2, np.float32)
                assert np.array_equal(got.view(np.uint32), want[c].view(np.uint32)), (p, c, np.flatnonzero(got != want[c])[:4])
                if rp.ys[c] is None:
                    continue
                fl = s.floors[mp.submap_floor[mp.mux[c]]]
                _, fy, flag, _, _ = ob.floor1_curve(fl.xs, fl.multiplier, rp.ys[c], n)
                k = len(fl.xs)
                assert np.array_equal(_stage(ctx, h, p, c, abi.POV_STAGE_FINAL_YS, k, np.uint32), fy), (p, c)
                assert np.array_equal(_stage(ctx, h, p, c, abi.POV_STAGE_STEP2_FLAG, k, np.uint8).astype(bool), flag), (p, c)
        # 2. PCM of the production route: raw packets == host walk, bit for bit; both == the oracle on reader + model
        kernel = ctx.L.pov_batch_kernel_name(ctx.ctx, h).decode()
        if st.expect_kernel:
            assert kernel == st.expect_kernel
        ctx._check(ctx.L.pov_batch_run(ctx.ctx, h))
        pcm_raw = _pcm(ctx, h, b)
        h2 = _upload(ctx, cs_h, b_h)
        handles.append(h2)
        assert ctx.L.pov_batch_kernel_name(ctx.ctx, h2).decode() == kernel
        ctx._check(ctx.L.pov_batch_run(ctx.ctx, h2))
        pcm_host = _pcm(ctx, h2, b_h)
        assert np.array_equal(pcm_raw.view(np.uint32), pcm_host.view(np.uint32)), kernel
        dense = _dense_reference(s, b_h, reads)
        ref, rstatus = ob.synth_batch_raw(cs_h, dense.to_c())
        assert np.array_equal(rstatus, ostatus)
        err = float(np.abs(pcm_raw - ref).max()) if ref.size else 0.0
        assert err <= 1e-5 and ob.snr_db(pcm_raw, ref) >= 120.0, (kernel, err, ob.snr_db(pcm_raw, ref))
    finally:
        for hh in handles:
            ctx.L.pov_batch_free(ctx.ctx, hh)
        po_host.close()
        po_raw.close()


def test_all_three_synthesis_routes_are_reached(ctx):
    """The streams above must keep exercising every route pov_batch_run can take; a change of the selection logic that
    dropped one from them would otherwise go unnoticed."""
    seen = {}
    for name in rv.ALL_NAMES:
        po = lib.ParsedOgg(rv.stream(name).data, raw_packets=True)
        try:
            cs, b = po.get(0)
            h = _upload(ctx, cs, b)
            seen[name] = ctx.L.pov_batch_kernel_name(ctx.ctx, h).decode()
            ctx.L.pov_batch_free(ctx.ctx, h)
        finally:
            po.close()
    print("routes:", {k: sorted(n for n in seen if seen[n] == k) for k in ROUTES})
    assert set(seen.values()) == ROUTES, seen


def _corpus(ctx, files, s16=False):
    got, order = {}, []

    def sink(i, pcm):
        order.append(i)
        got[i] = pcm.copy()
        return False
    frames, total, _ = ctx.decode_corpus_pcm(files, sink, host_threads=4, s16=s16)
    return order, got, frames, total


def test_corpus_decode_matches_the_whole_file_decode(ctx, monkeypatch):
    """All streams through decode_corpus_pcm: delivered in file order. With one file per chunk every chunk is the batch
    decode_ogg makes, so the PCM is the same bit for bit; in the default chunks, which mix setups and hence may take another
    synthesis route than the file alone, it is the same within the decode's tolerance."""
    files = [rv.stream(n).data for n in rv.ALL_NAMES]
    single = [ctx.decode_ogg(f)[0] for f in files]
    monkeypatch.setenv("POV_CORPUS_CHUNK", "1")
    order, got, frames, total = _corpus(ctx, files)
    assert order == list(range(len(files)))
    assert list(frames) == [x.shape[1] for x in single] and total == sum(x.size for x in single)
    for i, x in enumerate(single):
        assert got[i].shape == x.shape and np.array_equal(got[i].view(np.uint32), x.view(np.uint32)), rv.ALL_NAMES[i]
    monkeypatch.delenv("POV_CORPUS_CHUNK")
    order, got, frames, _ = _corpus(ctx, files)
    assert order == list(range(len(files)))
    for i, x in enumerate(single):
        assert got[i].shape == x.shape, rv.ALL_NAMES[i]
        assert float(np.abs(got[i] - x).max(initial=0.0)) <= 1e-5 and ob.snr_db(got[i], x) >= 120.0, rv.ALL_NAMES[i]
    # int16 output of the same chunks: the conversion rule applied to the float32 output
    subset = files[::4]
    _, f32, _, _ = _corpus(ctx, subset)
    order, i16, _, _ = _corpus(ctx, subset, s16=True)
    assert order == list(range(len(subset)))
    for i in range(len(subset)):
        assert i16[i].dtype == np.int16 and np.array_equal(i16[i], to_s16(f32[i])), i
