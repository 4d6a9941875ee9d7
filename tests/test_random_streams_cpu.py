"""Whole-file parse of seeded random Vorbis streams (tests/random_vorbis.py) against an independent packet reader, on the
CPU: the host walk's floor flags, coded Ys, classifications and VQ entry numbers must be what the reader reads from the
packet bits, and the oracle applying the host's descriptors must give the model's `after_residue` bit for bit."""
import numpy as np
import pytest

from parseoggvorbis_b200 import lib
from tests import oracle_binding as ob
from tests import random_vorbis as rv


def _read_all(st):
    """Reader output of every packet of a stream, self-checked against the writer where the packet is whole."""
    out = []
    checked = 0
    for pc in st.packets:
        data = rv.vw.write_audio_packet(st.setup, pc)
        rp = rv.read_packet(st.setup, data)
        if pc.truncate_bytes is None:
            rv.self_check(st.setup, pc, rp)
            checked += 1
        out.append(rp)
    assert checked == sum(pc.truncate_bytes is None for pc in st.packets)
    return out


@pytest.mark.parametrize("name", rv.ALL_NAMES)
def test_host_walk_and_oracle_residue_match_the_reader(name):
    st = rv.stream(name)
    s = st.setup
    reads = _read_all(st)
    po = lib.ParsedOgg(st.data)
    try:
        assert po.n_streams == 1
        cs, b = po.get(0)
        assert int(cs.channels) == s.channels and tuple(cs.blocksize) == tuple(s.blocksize)
        assert b.n_packets == len(st.packets)
        pk = rv.packets_array(b)
        ys = np.ctypeslib.as_array(b.ys, shape=(int(b.n_ys),)) if b.n_ys else np.zeros(0, np.uint16)
        for p, rp in enumerate(reads):
            assert int(pk["mode"][p]) == rp.mode, p
            used = [y is not None for y in rp.ys]
            assert int(pk["floor_used"][p]) == sum(1 << c for c, u in enumerate(used) if u), p
            yo = int(pk["ys_off"][p])
            for c, y in enumerate(rp.ys):
                if y is not None:
                    assert ys[yo:yo + len(y)].tolist() == y, (p, c)
                    yo += len(y)
            for sm, ((cls, ents), (rcls, _, flat)) in enumerate(zip(rv.split_entries_payload(s, b, pk[p], rp.mode), rp.residue)):
                assert np.array_equal(cls, rcls), (p, sm)
                assert ents.tolist() == flat, (p, sm)
        _, status, cap = ob.synth_batch_raw(cs, b, capture=True)
        assert not status.any(), np.flatnonzero(status)
        for p, rp in enumerate(reads):
            want = rv.model_after_residue(s, rp)
            half = want.shape[1]
            got = cap["after_residue"][p, :, :half]
            assert np.array_equal(got.view(np.uint32), want.view(np.uint32)), (p, np.argwhere(got != want)[:4])
    finally:
        po.close()


def test_edge_streams_reach_their_edges():
    """The named streams hold what their names promise (guards the generator against a silent change)."""
    cw = rv.stream("cw9_10").setup
    assert all(set(bk.lengths) <= {9, 10} for bk in cw.books)
    cut = rv.stream("cut32")
    assert any(L == 32 for bk in cut.setup.books for L in bk.lengths)
    assert sum(pc.truncate_bytes is not None for pc in cut.packets) >= 2
    assert sorted(len(f.xs) for f in rv.stream("wide_floors").setup.floors) == [65, 128, 250]
    assert len(rv.stream("modes64").setup.modes) == 64
    assert max(len(m.submap_floor) for m in rv.stream("submaps8").setup.mappings) == 8
    assert max(bk.n_entries for bk in rv.stream("book65537").setup.books) == 65537
    assert rv.stream("nclass64_passes8").setup.residues[0].n_class == 64
    assert all(b >= 0 for b in rv.stream("nclass64_passes8").setup.residues[0].books[1])
    r = rv.stream("classdim3_parts7").setup
    assert r.books[r.residues[0].classbook].dim == 3 and (r.residues[0].end - r.residues[0].begin) // r.residues[0].partition_size == 7
    assert all(r.partition_size == 1 for r in rv.stream("psize1").setup.residues)
    seeds = [rv.stream("seed%d" % k) for k in rv.SEEDS]
    pairs = {st.setup.blocksize for st in seeds}
    assert any(a == b for a, b in pairs) and any(b == 8192 for _, b in pairs) and any(a == 64 for a, _ in pairs)
    assert {r.type for st in seeds for r in st.setup.residues} == {0, 1, 2}
    assert {st.setup.channels for st in seeds} == set(range(1, 9))
    assert sum(pc.truncate_bytes is not None for st in seeds for pc in st.packets) >= 40
