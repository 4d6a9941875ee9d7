"""The corpus stream table (pov_corpus_streams / lib.corpus_streams) without a GPU: one record per logical stream with a
complete setup, in file order, whose channels, rate and frames must equal what the single-file parse
(pov_ogg_parse_memory_ex) gives for the same stream; errors carry the corpus decode's "file k: check failed: ..." text."""
import ctypes as C
import os
import subprocess
import sys

import numpy as np
import pytest

from parseoggvorbis_b200 import abi, lib
from tests import random_vorbis as rv
from tests.conftest import SYNTHETIC

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "tools"))
import vorbis_writer as vw  # noqa: E402

FIX = {"stereo44khz": "test.stereo44khz.ogg", "mono44khz": "test.mono44khz.ogg"}
FIX.update({n: n + ".ogg" for n in SYNTHETIC})


def _load(name):
    with open(os.path.join(ROOT, "tests", "golden", FIX[name]), "rb") as f:
        return f.read()


def _expected(files, allow_spanning=False):
    """(file, channels, rate, frames) of every stream with a setup, from the single-file parse."""
    out = []
    for i, data in enumerate(files):
        po = lib.ParsedOgg(data, raw_packets=True, allow_spanning=allow_spanning)
        try:
            for k in range(po.n_streams):
                s, b = po.get(k)
                if s.channels == 0:                   # no complete setup: the decode skips the stream
                    continue
                frames = int(b.streams[0].pcm_frames)
                assert int(b.pcm_floats) == frames * int(s.channels)
                out.append((i, int(s.channels), int(s.sample_rate), frames))
        finally:
            po.close()
    return out


def _rows(t):
    return [(int(f), int(c), int(r), int(n)) for f, c, r, n in zip(t.file, t.channels, t.sample_rate, t.frames)]


def _headers_only(data):
    """The three header pages of a synthetic stream: a complete setup and no audio packet."""
    return b"".join(vw.split_pages(data)[:3])


def _corpus():
    chained = vw.chain_files([_load("stereo44khz"), _load("mono44khz")])
    files = [_load(n) for n in FIX] + [rv.stream("seed%d" % k).data for k in range(20)]
    files += [chained, _headers_only(_load("synth_two_submaps")), _load("mono44khz")]
    return files


def test_table_equals_the_single_file_parse():
    files = _corpus()
    t = lib.corpus_streams(files, host_threads=4)
    exp = _expected(files)
    assert _rows(t) == exp
    assert t.file.dtype == np.uint32 and t.frames.dtype == np.uint64 and len(t) == len(exp)
    # the chained file gives two records, the headers-only file one with no frames
    chained = len(FIX) + 20
    assert [r[1] for r in exp if r[0] == chained] == [2, 1]
    assert [r[3] for r in exp if r[0] == chained + 1] == [0]
    assert all(r[3] > 0 for r in exp if r[0] != chained + 1)
    # the thread count does not change the table
    assert _rows(lib.corpus_streams(files, host_threads=1)) == exp
    assert _rows(lib.corpus_streams(files)) == exp


def test_empty_corpus():
    t = lib.corpus_streams([])
    assert len(t) == 0 and t.frames.dtype == np.uint64


def test_spanning_pages_follow_the_flag():
    from tests.test_front_end_cpu import _spanning_twin
    files = [_load("mono44khz"), _spanning_twin("two_submaps")]
    with pytest.raises(lib.PovError) as ei:
        lib.corpus_streams(files)
    with pytest.raises(lib.PovError) as single:
        lib.ParsedOgg(files[1], raw_packets=True)
    assert ei.value.code == abi.POV_ERR_STREAM and "spanning pages" in ei.value.msg
    assert ei.value.msg == "file 1: " + single.value.msg
    t = lib.corpus_streams(files, allow_spanning=True)
    assert _rows(t) == _expected(files, allow_spanning=True)
    assert int(t.frames[1]) == int(lib.corpus_streams([_load("synth_two_submaps")]).frames[0])


def _broken_header(data):
    """The setup header's "vorbis" signature damaged, the page checksum repaired: a header error, not a framing error."""
    pages = vw.split_pages(data)
    p = bytearray(pages[2])
    body = 27 + p[26]
    assert p[body:body + 7] == b"\x05vorbis"
    p[body + 1] ^= 0x20
    pages[2] = vw.with_serial(bytes(p), int.from_bytes(p[14:18], "little"))
    return b"".join(pages)


@pytest.mark.parametrize("kind", ["header", "crc"])
def test_errors_name_the_first_failing_file(kind):
    good = _load("synth_two_submaps")
    if kind == "header":
        bad = _broken_header(good)
    else:
        b = bytearray(good); b[len(b) // 2] ^= 0x55
        bad = bytes(b)
    with pytest.raises(lib.PovError) as single:
        lib.ParsedOgg(bad, raw_packets=True)
    files = [good] * 5 + [bad] + [good] * 3 + [_broken_header(_load("synth_res0_mono"))]
    for threads in (1, 3, 8):
        with pytest.raises(lib.PovError) as ei:
            lib.corpus_streams(files, host_threads=threads)
        assert ei.value.code == abi.POV_ERR_STREAM
        assert ei.value.msg == "file 5: " + single.value.msg
        assert ei.value.msg.startswith("file 5: check failed: ")


def test_new_struct_sizes_match_c_compiler(tmp_path):
    names = ["pov_stream_info", "pov_device_pcm"]
    src = tmp_path / "s.c"
    src.write_text('#include <stdio.h>\n#include "pov_synth.h"\nint main(){' +
                   "".join('printf("%s %%zu\\n", sizeof(%s));' % (n, n) for n in names) + "return 0;}\n")
    exe = tmp_path / "s.bin"
    subprocess.check_call(["gcc", "-I", os.path.join(ROOT, "include"), str(src), "-o", str(exe)])
    out = dict(line.split() for line in subprocess.check_output([str(exe)], text=True).splitlines())
    for n in names:
        assert int(out[n]) == C.sizeof(getattr(abi, n)), n
