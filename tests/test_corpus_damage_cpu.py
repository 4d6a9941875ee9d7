"""Cut mode of the corpus parse without a GPU (POV_PARSE_CUT_DAMAGE: lib.corpus_streams(cut_damage=True), ParsedOgg(cut_damage=
True)). Damaged files are built from the bundled fixtures and from seeded random streams, chained files included. The strict
table must still fail with the text it always had; in cut mode a file damaged at the page level has the table of its pages
before the damage, a file whose packet p has a bad header keeps exactly packets < p (frames = pcm_off[p] of the undamaged file),
a failing host walk keeps the packet (as silence) and the geometry, and a clean corpus has the same table in both modes."""
import ctypes as C
import os
import struct
import sys

import numpy as np
import pytest

from parseoggvorbis_b200 import abi, lib
from tests import random_vorbis as rv

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "tools"))
import vorbis_writer as vw  # noqa: E402

FIX = {"stereo44khz": "test.stereo44khz.ogg", "mono44khz": "test.mono44khz.ogg", "synth_two_submaps": "synth_two_submaps.ogg",
       "synth_surround51": "synth_surround51.ogg", "synth_bad_vq_book": "synth_bad_vq_book.ogg"}


def load(name):
    with open(os.path.join(ROOT, "tests", "golden", FIX[name]), "rb") as f:
        return f.read()


def rows(t):
    return [(int(f), int(c), int(r), int(n)) for f, c, r, n in zip(t.file, t.channels, t.sample_rate, t.frames)]


def strict_error(files):
    try:
        lib.corpus_streams(files)
    except lib.PovError as e:
        return e.code, e.msg
    return None


def page_starts(data):
    out, at = [], 0
    for pg in vw.split_pages(data):
        out.append(at)
        at += len(pg)
    return out


def all_packets(data):
    """(page start, byte offset, length) of every packet of a single-stream file without spanning packets."""
    out = []
    for at in page_starts(data):
        nseg = data[at + 26]
        off, plen = at + 27 + nseg, 0
        for i in range(nseg):
            plen += data[at + 27 + i]
            if data[at + 27 + i] == 255:
                continue
            out.append((at, off, plen))
            off += plen
            plen = 0
    return out


def audio_packets(data):
    return all_packets(data)[3:]


def with_page_crc(buf, at):
    """Recompute the CRC of the page at `at` (after an edit that should reach the packet decoders, not the container check)."""
    nseg = buf[at + 26]
    size = 27 + nseg + sum(buf[at + 27:at + 27 + nseg])
    buf[at + 22:at + 26] = b"\0\0\0\0"
    buf[at + 22:at + 26] = struct.pack("<I", vw.ogg_crc(bytes(buf[at:at + size])))
    return buf


def bad_header_bits(data, p, mode_bits=None):
    """Audio packet p with its packet-type bit set, or (mode_bits = its mode field width) with an out-of-range mode number."""
    at, off, _ = audio_packets(data)[p]
    buf = bytearray(data)
    if mode_bits is None:
        buf[off] |= 1
    else:
        buf[off] = (buf[off] & ~(((1 << mode_bits) - 1) << 1)) | (((1 << mode_bits) - 1) << 1)
    return bytes(with_page_crc(buf, at))


def parse_packets(data, **kw):
    """Per stream with a setup: (n_modes, pcm_off[], emit_frames[], frames) of the single-file parse."""
    po = lib.ParsedOgg(data, **kw)
    try:
        out = []
        for k in range(po.n_streams):
            s, b = po.get(k)
            if s.channels == 0:
                continue
            pk = [b.packets[i] for i in range(b.n_packets)]
            out.append((int(s.n_modes), [int(x.pcm_off) for x in pk], [int(x.emit_frames) for x in pk], int(b.streams[0].pcm_frames),
                        [int(x.floor_used) for x in pk]))
        return out
    finally:
        po.close()


def prefix_before(data, offset):
    """The file truncated to its whole pages before byte `offset`."""
    pages, at, out = vw.split_pages(data), 0, []
    for pg in pages:
        if at + len(pg) > offset:
            break
        out.append(pg)
        at += len(pg)
    return b"".join(out)


def page_damage(data, seed):
    """(kind, damaged file, offset of the first damaged byte) for each page-level damage of `data`."""
    rng = np.random.default_rng(seed)
    starts = page_starts(data)
    out = []
    for frac in (0.3, 0.7):                                    # truncation inside a page body
        out.append(("truncated", data[:int(len(data) * frac)], int(len(data) * frac)))
    k = int(rng.integers(3, len(starts))) if len(starts) > 3 else len(starts) - 1
    out.append(("page_edge", data[:starts[k] + 28], starts[k]))            # one byte into a page's segment table
    out.append(("in_headers", data[:starts[1] + 40], starts[1]))           # inside the comment header page
    at = starts[k]
    buf = bytearray(data); buf[at + 30] ^= 0x40
    out.append(("crc", bytes(buf), at))
    buf = bytearray(data); buf[at] = ord("X")
    out.append(("capture", bytes(buf), at))
    return out


def damaged_corpus():
    """(name, damaged file, undamaged counterpart to compare with) for every page-level damage of the fixtures, a random
    stream and the second link of a chained file."""
    sources = {"stereo44khz": load("stereo44khz"), "synth_surround51": load("synth_surround51"), "seed3": rv.stream("seed3").data}
    out = []
    for i, (name, data) in enumerate(sources.items()):
        for kind, bad, offset in page_damage(data, i):
            out.append(("%s/%s" % (name, kind), bad, prefix_before(data, offset)))
    first, second = load("mono44khz"), rv.stream("seed5").data
    chained = vw.chain_files([first, second])
    at = len(first) + page_starts(second)[4]
    buf = bytearray(chained); buf[at + 40] ^= 1
    out.append(("chained/second_link_crc", bytes(buf), chained[:at]))
    out.append(("chained/second_link_truncated", chained[:at + 50], chained[:at]))
    return out


DAMAGED = damaged_corpus()


@pytest.mark.parametrize("case", range(len(DAMAGED)), ids=[d[0] for d in DAMAGED])
def test_page_damage_cuts_to_the_pages_before_it(case):
    name, bad, prefix = DAMAGED[case]
    clean = load("mono44khz")
    corpus = [clean, bad, clean]
    err = strict_error(corpus)
    assert err is not None and err[0] == abi.POV_ERR_STREAM and err[1].startswith("file 1: check failed: page"), (name, err)
    cut = rows(lib.corpus_streams(corpus, cut_damage=True))
    assert cut == rows(lib.corpus_streams([clean, prefix, clean])), name
    # the single-file parse agrees, packet by packet
    assert parse_packets(bad, raw_packets=True, cut_damage=True) == parse_packets(prefix, raw_packets=True)


def _mode_bits(n_modes):
    return (n_modes - 1).bit_length()


@pytest.mark.parametrize("name", ["stereo44khz", "synth_two_submaps"] + ["seed%d" % k for k in range(8)])
@pytest.mark.parametrize("kind", ["type_bit", "mode_number"])
def test_bad_packet_header_keeps_the_packets_before_it(name, kind):
    data = load(name) if name in FIX else rv.stream(name).data
    (n_modes, pcm_off, emit, frames, _), = parse_packets(data, raw_packets=True)
    bits = _mode_bits(n_modes)
    if kind == "mode_number" and (1 << bits) - 1 < n_modes:
        pytest.skip("every mode number the field can hold is valid (%d modes)" % n_modes)
    for p in sorted({0, 1, len(pcm_off) // 2, len(pcm_off) - 1}):
        bad = bad_header_bits(data, p, bits if kind == "mode_number" else None)
        err = strict_error([bad])
        want = "packet type bit set" if kind == "type_bit" else "mode %d out of range" % ((1 << bits) - 1)
        assert err == (abi.POV_ERR_STREAM, "file 0: check failed: audio packet %d: audio packet: %s (hpp:%s)"
                       % (p, want, "1142" if kind == "type_bit" else "1147")), err
        t = lib.corpus_streams([bad], cut_damage=True)
        assert list(t.frames) == [pcm_off[p]]
        got, = parse_packets(bad, raw_packets=True, cut_damage=True)
        assert got[1] == pcm_off[:p] and got[2] == emit[:p] and got[3] == pcm_off[p]


def test_host_walk_failure_keeps_the_packet_as_silence():
    """A VQ entry the host walk refuses: strict parse fails there; the cut parse keeps every packet and the geometry the raw
    (device walk) parse has, with the failing packet and every later one as silence (no floor used)."""
    data = load("synth_bad_vq_book")
    with pytest.raises(lib.PovError) as ei:
        lib.ParsedOgg(data)
    assert "invalid VQ entry" in ei.value.msg
    p = int(ei.value.msg.split("audio packet ")[1].split(":")[0])
    (_, off_raw, emit_raw, frames_raw, _), = parse_packets(data, raw_packets=True)
    (_, off, emit, frames, used), = parse_packets(data, cut_damage=True)
    assert (off, emit, frames) == (off_raw, emit_raw, frames_raw)
    assert all(u == 0 for u in used[p:])
    assert rows(lib.corpus_streams([data], cut_damage=True)) == rows(lib.corpus_streams([data]))


def test_random_bytes_and_empty_files():
    rng = np.random.default_rng(5)
    junk = bytes(rng.integers(0, 256, 5000, dtype=np.uint8))
    clean = load("stereo44khz")
    err = strict_error([clean, junk])
    assert err == (abi.POV_ERR_STREAM, "file 1: check failed: page: capture pattern (hpp:77)")
    assert rows(lib.corpus_streams([clean, junk, b"", clean], cut_damage=True)) == rows(lib.corpus_streams([clean, b"", b"", clean]))
    assert len(lib.corpus_streams([junk, b""], cut_damage=True)) == 0


def test_damage_in_the_headers_leaves_no_record():
    data = load("stereo44khz")
    at, off, _ = all_packets(data)[2]
    buf = bytearray(data)
    buf[off] = 7                                                  # the setup header's packet type, CRC repaired
    bad = bytes(with_page_crc(buf, at))
    err = strict_error([bad])
    assert err is not None and err[1].startswith("file 0: check failed:")
    assert len(lib.corpus_streams([bad], cut_damage=True)) == 0


def test_clean_corpus_has_the_same_table_in_both_modes():
    files = [load(n) for n in FIX if n != "synth_bad_vq_book"] + [rv.stream("seed%d" % k).data for k in range(10)]
    files.append(vw.chain_files([load("stereo44khz"), load("mono44khz")]))
    assert rows(lib.corpus_streams(files, cut_damage=True)) == rows(lib.corpus_streams(files))
    for f in files[:4]:
        assert parse_packets(f, raw_packets=True, cut_damage=True) == parse_packets(f, raw_packets=True)


def test_report_struct_matches_the_c_compiler(tmp_path):
    import subprocess
    src = tmp_path / "s.c"
    src.write_text('#include <stdio.h>\n#include <stddef.h>\n#include "pov_synth.h"\nint main(){printf("%zu %zu", sizeof(pov_file_report), '
                   'offsetof(pov_file_report, message));return 0;}\n')
    exe = tmp_path / "s.bin"
    subprocess.check_call(["gcc", "-I", os.path.join(ROOT, "include"), str(src), "-o", str(exe)])
    size, off = map(int, subprocess.check_output([str(exe)], text=True).split())
    assert size == C.sizeof(abi.pov_file_report) and off == abi.pov_file_report.message.offset
