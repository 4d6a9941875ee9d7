"""Corpus and batch decode into caller-owned device memory (pov_decode_corpus_device, pov_batch_upload_into): every stream's
samples must equal what the host-memory decode of the same chunks delivers, and every sample outside the written rows must
keep the sentinel the test put there first.

k_warp_synth and k_fused_synth choose between a 16-byte vector store path and a scalar one by the alignment of each
destination, and for float32 the two paths do not always agree in the last bit. So the comparison is bit for bit wherever
each channel's destination has the alignment (sample index mod 4) it has in the host decode's chunk arena ("mirror"
layouts), and for int16 everywhere; float32 in other layouts must agree within 1e-6."""
import contextlib
import ctypes as C
import dataclasses
import os
import sys

import numpy as np
import pytest

from parseoggvorbis_b200 import abi, lib, workloads
from tests import random_vorbis as rv
from tests.conftest import SYNTHETIC

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "tools"))
import vorbis_writer as vw  # noqa: E402

FIX = {"stereo44khz": "test.stereo44khz.ogg", "mono44khz": "test.mono44khz.ogg"}
FIX.update({n: n + ".ogg" for n in SYNTHETIC})
# random streams: 1-8 channels, block sizes 64..8192 (the 8-channel 8192 ones need the staged kernels)
RANDOM = ["seed%d" % k for k in range(12)] + ["bs_64_64", "bs_64_8192", "bs_128_4096", "bs_8192_8192", "ch8_256_8192",
                                              "ch8_4096_type2_p16", "wide_floors", "submaps8"]
VARIANTS = {"default": {}, "one_file_per_chunk": {"POV_CORPUS_CHUNK": "1"}, "fused": {"POV_KERNEL": "fused"},
            "host_entropy": {"POV_DEVICE_ENTROPY": "0"}}
SENTINEL_I16 = 0x7FFF


def _load(name):
    with open(os.path.join(ROOT, "tests", "golden", FIX[name]), "rb") as f:
        return f.read()


@contextlib.contextmanager
def _env(env):
    old = {k: os.environ.get(k) for k in env}
    os.environ.update(env)
    try:
        yield
    finally:
        for k, v in old.items():
            if v is None:
                os.environ.pop(k, None)
            else:
                os.environ[k] = v


@pytest.fixture(scope="module")
def files():
    out = [_load(n) for n in FIX] + [rv.stream(n).data for n in RANDOM]
    out.insert(5, vw.chain_files([_load("stereo44khz"), _load("synth_surround51"), _load("mono44khz")]))
    return out


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


_REF = {}


def _reference(ctx, variant, files, s16):
    """Per logical stream, in order: the (channels, frames) PCM decode_corpus_pcm delivers (streams without frames are not
    delivered: None)."""
    key = (variant, s16, len(files))
    if key not in _REF:
        got = []

        def sink(i, pcm):
            got.append((i, pcm.copy()))
            return False
        with _env({k: v for k, v in VARIANTS[variant].items() if k == "POV_CORPUS_CHUNK"}):
            ctx.decode_corpus_pcm(files, sink, host_threads=4, s16=s16)
        table = lib.corpus_streams(files)
        out, k = [], 0
        for f, c, n in zip(table.file, table.channels, table.frames):
            if n == 0:
                out.append(None)
                continue
            assert got[k][0] == f and got[k][1].shape == (c, n)
            out.append(got[k][1])
            k += 1
        assert k == len(got)
        _REF[key] = out
    return _REF[key]


def _host_arena_bases(table, n_files, files_per_chunk):
    """Each stream's sample index in the PCM arena of its chunk in the host decode (front_end.cpp: the first chunk holds
    files_per_chunk / 8 files and every next one half as many more, up to files_per_chunk; streams are packed in order)."""
    owner = np.zeros(n_files, np.int64)
    at, size, k = 0, max(1, files_per_chunk // 8), 0
    while at < n_files:
        owner[at:at + size] = k
        at += size
        size = min(files_per_chunk, size + (size + 1) // 2)
        k += 1
    out = np.zeros(len(table), np.uint64)
    used, last = 0, -1
    for i in range(len(table)):
        c = owner[int(table.file[i])]
        if c != last:
            used, last = 0, c
        out[i] = used
        used += int(table.channels[i]) * int(table.frames[i])
    return out


def _layout(table, kind, host_bases=None):
    ch = table.channels.astype(np.uint64)
    fr = table.frames.astype(np.uint64)
    if kind == "mirror":                   # padded, with every destination aligned as in the host arena (mod 4)
        stride = fr + np.uint64(4)
        base, at = np.zeros(len(fr), np.uint64), 0
        for i in range(len(fr)):
            at = (at + 8) // 4 * 4 + int(host_bases[i]) % 4
            base[i] = at
            at += int(ch[i]) * int(stride[i])
        return base, stride, at + 5
    if kind == "padded":
        T = int((fr.max() + 3) // 4 * 4)
        stride = np.full(len(fr), T, np.uint64)
        base = np.arange(len(fr), dtype=np.uint64) * np.uint64(int(ch.max()) * T)
        return base, stride, int(len(fr) * int(ch.max()) * T)
    if kind == "packed":
        stride = (fr + 3) // 4 * 4
    else:                                  # "odd": stride = frames, every base one sample past the previous region
        stride = fr.copy()
    sizes = ch * stride + (1 if kind == "odd" else 0)
    base = np.cumsum(sizes) - sizes + (1 if kind == "odd" else 0)
    return base.astype(np.uint64), stride, int(sizes.sum()) + 3


def _sentinel_tensor(n, s16):
    import torch
    if s16:
        return torch.full((n,), SENTINEL_I16, dtype=torch.int16, device="cuda:0")
    return torch.full((n,), float("nan"), dtype=torch.float32, device="cuda:0")


def _expected(n, s16, table, base, stride, ref):
    """Host image of the whole tensor: the sentinel everywhere but the streams' rows."""
    out = np.full(n, SENTINEL_I16, np.int16) if s16 else np.full(n, np.nan, np.float32)
    for i, pcm in enumerate(ref):
        if pcm is None:
            continue
        b, s, f = int(base[i]), int(stride[i]), int(table.frames[i])
        for c in range(pcm.shape[0]):
            out[b + c * s:b + c * s + f] = pcm[c]
    return out


def _same_bits(got, exp):
    if got.dtype == np.float32:
        return np.array_equal(got.view(np.uint32), exp.view(np.uint32))
    return np.array_equal(got, exp)


def _assert_matches(got, exp, exact):
    """Sentinels and every int16 sample bit for bit; float32 samples bit for bit if `exact`, else within 1e-6."""
    if exact or got.dtype != np.float32:
        diff = np.nonzero(got.view(np.uint32) != exp.view(np.uint32) if got.dtype == np.float32 else got != exp)[0]
        assert diff.size == 0, "%d samples differ, first at %d" % (diff.size, diff[0])
        return
    sentinel = np.isnan(exp)
    assert np.array_equal(got[sentinel].view(np.uint32), exp[sentinel].view(np.uint32)), "a sentinel was overwritten"
    err = float(np.abs(got[~sentinel] - exp[~sentinel]).max(initial=0.0))
    print("float32, alignment differing from the host arena: %d of %d samples differ in bits, max-abs %.3g"
          % (int((got[~sentinel].view(np.uint32) != exp[~sentinel].view(np.uint32)).sum()), int((~sentinel).sum()), err))
    assert err <= 1e-6, err


def _files_per_chunk(variant):
    v = VARIANTS[variant]
    return int(v.get("POV_CORPUS_CHUNK", 64 if v.get("POV_DEVICE_ENTROPY") == "0" else 256))


@pytest.mark.parametrize("layout", ["mirror", "padded", "packed", "odd"])
@pytest.mark.parametrize("s16", [False, True])
@pytest.mark.parametrize("variant", list(VARIANTS))
def test_corpus_into_caller_memory_equals_the_host_decode(files, contexts, variant, s16, layout):
    ctx = contexts(variant)
    ref = _reference(ctx, variant, files, s16)
    table = lib.corpus_streams(files)
    base, stride, n = _layout(table, layout, _host_arena_bases(table, len(files), _files_per_chunk(variant)))
    t = _sentinel_tensor(n, s16)
    with _env({k: v for k, v in VARIANTS[variant].items() if k == "POV_CORPUS_CHUNK"}):
        frames, total = ctx.decode_corpus_into(files, t, table, base, stride, s16=s16, host_threads=4)
    assert total == int((table.channels.astype(np.uint64) * table.frames).sum())
    assert list(frames) == [int(table.frames[table.file == i].sum()) for i in range(len(files))]
    _assert_matches(t.cpu().numpy(), _expected(n, s16, table, base, stride, ref), exact=layout == "mirror")


@pytest.mark.parametrize("s16", [False, True])
@pytest.mark.parametrize("layout", ["padded", "packed"])
def test_decode_corpus_device_tensor_and_views(files, contexts, layout, s16):
    import torch
    ctx = contexts("default")
    ref = _reference(ctx, "default", files, s16)
    out = ctx.decode_corpus_device(files, layout=layout, s16=s16, host_threads=4)
    assert out.pcm.dtype == (torch.int16 if s16 else torch.float32) and out.pcm.device == torch.device("cuda", 0)
    assert np.all(out.base % 4 == 0) and np.all(out.stride % 4 == 0) and np.all(out.stride >= out.table.frames)
    if layout == "padded":
        assert out.pcm.shape == (len(out.table), int(out.table.channels.max()), int(out.stride[0]))
    for i, pcm in enumerate(ref):
        v = out.stream(i).cpu().numpy()
        assert v.shape == (int(out.table.channels[i]), int(out.table.frames[i]))
        if pcm is not None:
            _assert_matches(np.ascontiguousarray(v).ravel(), pcm.ravel(), exact=False)
    # nothing outside the streams is written: the padding is still zero
    mask = torch.ones_like(out.pcm, dtype=torch.bool)
    for i in range(len(out.table)):
        if layout == "padded":
            mask[i, :int(out.table.channels[i]), :int(out.table.frames[i])] = False
        else:
            b, s = int(out.base[i]), int(out.stride[i])
            mask[b:b + int(out.table.channels[i]) * s].view(int(out.table.channels[i]), s)[:, :int(out.table.frames[i])] = False
    assert int(out.pcm[mask].count_nonzero()) == 0


@pytest.mark.parametrize("side_stream", [False, True])
def test_corpus_waits_for_the_callers_stream(files, contexts, side_stream):
    """A long sleep and then a sentinel fill of the tensor queued on torch's current stream: if the library's writes did not
    wait for them, the fill would land on top of the PCM."""
    import torch
    ctx = contexts("default")
    ref = _reference(ctx, "default", files, False)
    table = lib.corpus_streams(files)
    base, stride, n = _layout(table, "packed")
    t = torch.zeros(n, dtype=torch.float32, device="cuda:0")
    torch.cuda.synchronize()
    s = torch.cuda.Stream() if side_stream else torch.cuda.current_stream()
    with torch.cuda.stream(s):
        torch.cuda._sleep(2_000_000_000)
        t.fill_(float("nan"))
        ctx.decode_corpus_into(files, t, table, base, stride, host_threads=4)
        got = t.cpu().numpy()
    _assert_matches(got, _expected(n, False, table, base, stride, ref), exact=False)


def test_errors_equal_the_host_decode_and_the_context_keeps_working(files, contexts):
    """A file refused in mid-corpus (a scalar book used as a VQ book; audio packets with bytes flipped and page checksums
    repaired): the device decode fails with decode_corpus_pcm's error text."""
    from tests.test_gpu_decode import _flip_bits_in_audio_packets
    import torch
    ctx = contexts("default")
    good = [_load("stereo44khz"), _load("synth_two_submaps")] * 3
    with open(os.path.join(ROOT, "tests", "golden", "synth_bad_vq_book.ogg"), "rb") as f:
        candidates = [f.read()]                               # a VQ entry the status words flag (hpp:739,748)
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
        except lib.PovError as e:                             # a framing / header error: the table says the same
            assert (e.code, e.msg) == host
            continue
        base, stride, n = _layout(table, "packed")
        t = _sentinel_tensor(n, False)
        with pytest.raises(lib.PovError) as ei:
            ctx.decode_corpus_into(corpus, t, table, base, stride, host_threads=3)
        assert (ei.value.code, ei.value.msg) == host
        assert "file 3" in host[1] or "chunk at file" in host[1]
        compared += 1
    assert compared >= 1
    # the context keeps working
    ref = _reference(ctx, "default", files, False)
    out = ctx.decode_corpus_device(files, layout="packed")
    for i, pcm in enumerate(ref):
        if pcm is not None:
            _assert_matches(np.ascontiguousarray(out.stream(i).cpu().numpy()).ravel(), pcm.ravel(), exact=False)
    torch.cuda.synchronize()


def test_device_to_host_bytes_are_the_status_words(files, contexts):
    ctx = contexts("default")
    packets = 0
    for data in files:
        po = lib.ParsedOgg(data, raw_packets=True)
        packets += sum(int(po.get(k)[1].n_packets) for k in range(po.n_streams) if po.get(k)[0].channels)
        po.close()
    for s16 in (False, True):
        h0, d0 = ctx.io_bytes()
        ctx.decode_corpus_device(files, layout="packed", s16=s16)
        h1, d1 = ctx.io_bytes()
        assert d1 - d0 == 4 * packets
        assert h1 > h0


def _raw_device_pcm(table, t, base, stride, layout):
    o = abi.pov_device_pcm()
    keep = [np.ascontiguousarray(x, dt) for x, dt in ((base, np.uint64), (stride, np.uint64), (table.file, np.uint32),
                                                        (table.channels, np.uint32), (table.frames, np.uint64))]
    o.pcm_layout, o.n_streams, o.pcm_dev, o.capacity = layout, len(table), t.data_ptr(), t.numel()
    o.stream_base, o.channel_stride = (k.ctypes.data_as(C.POINTER(C.c_uint64)) for k in keep[:2])
    o.file, o.channels = (k.ctypes.data_as(C.POINTER(C.c_uint32)) for k in keep[2:4])
    o.frames = keep[4].ctypes.data_as(C.POINTER(C.c_uint64))
    return o, keep


@pytest.mark.parametrize("case", ["capacity", "overlap", "stride", "interleaved", "dtype", "other_files", "device"])
def test_refusals_launch_nothing(files, contexts, case):
    import torch
    ctx = contexts("default")
    table = lib.corpus_streams(files)
    base, stride, n = _layout(table, "packed")
    t = _sentinel_tensor(n, False)
    launches = ctx.launch_count
    s16, tab = False, table
    k = int(np.argmax(table.frames))
    if case == "capacity":
        t = t[:int(base[-1] + table.channels[-1] * stride[-1]) - 1]
    elif case == "overlap":
        base = base.copy(); base[k] = base[k - 1] + 1
    elif case == "stride":
        stride = stride.copy(); stride[k] = table.frames[k] - 1
    elif case == "dtype":
        s16 = True
    elif case == "other_files":
        tab = lib.corpus_streams(files[1:] + files[:1])
        base, stride, n = _layout(tab, "packed")
        t = _sentinel_tensor(n, False)
    elif case == "device":
        t = torch.full((n,), float("nan"))                     # host memory
    with pytest.raises(lib.PovError) as ei:
        if case == "interleaved":
            o, keep = _raw_device_pcm(table, t, base, stride, abi.POV_PCM_INTERLEAVED)
            arr = (C.c_char_p * len(files))(*files)
            lens = (C.c_size_t * len(files))(*[len(f) for f in files])
            ctx._check(ctx.L.pov_decode_corpus_device(ctx.ctx, len(files), arr, lens, 2, C.byref(o), None, None))
        else:
            ctx.decode_corpus_into(files, t, tab, base, stride, s16=s16, host_threads=2)
    assert ei.value.code == abi.POV_ERR_ARG, ei.value.msg
    if case == "device":
        o, keep = _raw_device_pcm(table, t, base, stride, abi.POV_PCM_PLANAR)    # the C check behind the Python one
        arr = (C.c_char_p * len(files))(*files)
        lens = (C.c_size_t * len(files))(*[len(f) for f in files])
        assert ctx.L.pov_decode_corpus_device(ctx.ctx, len(files), arr, lens, 2, C.byref(o), None, None) == abi.POV_ERR_ARG
        assert "device memory" in ctx.L.pov_last_error(ctx.ctx).decode()
    if case == "other_files":
        assert ei.value.msg.startswith("file 0: ")
    assert ctx.launch_count == launches
    assert bool(torch.isnan(t).all())


def test_table_shorter_or_longer_than_the_corpus(files, contexts):
    ctx = contexts("default")
    table = lib.corpus_streams(files)
    short = lib.StreamTable(*(x[:-1] for x in table))
    base, stride, n = _layout(short, "packed")
    with pytest.raises(lib.PovError) as ei:
        ctx.decode_corpus_into(files, _sentinel_tensor(n, False), short, base, stride)
    assert ei.value.code == abi.POV_ERR_ARG and "more logical streams" in ei.value.msg
    assert ei.value.msg.startswith("file %d: " % (len(files) - 1))
    longer = lib.StreamTable(*(np.concatenate([x, x[-1:]]) for x in table))
    base, stride, n = _layout(longer, "packed")
    with pytest.raises(lib.PovError) as ei:
        ctx.decode_corpus_into(files, _sentinel_tensor(n, False), longer, base, stride)
    assert ei.value.code == abi.POV_ERR_ARG and "stream table" in ei.value.msg
    frames, total = ctx.decode_corpus_into([], _sentinel_tensor(0, False), lib.corpus_streams([]), [], [])
    assert len(frames) == 0 and total == 0


# ---- batch level ----------------------------------------------------------------------------------------------------
def _wide_floor_workload():
    rng = np.random.default_rng(7003)
    for _ in range(50):
        setup = workloads.random_setup(rng, 2, max_posts=64, max_couplings=2, max_posts_short=32)
        if max(len(f.xs) for f in setup.floors) > 32 and len(setup.floors) <= 4 and len(setup.mappings) <= 4:
            break
    return setup, workloads.random_batch(setup, rng, streams=3, packets_per_stream=70)


def _fused_only_workload():
    rng = np.random.default_rng(3 * 64 + 8192)
    setup = workloads.make_setup(2, (64, 8192), 22050, couplings=[(0, 1)])
    plans = [workloads.plan_stream(workloads.block_sequence(60, rng, p_short=0.2), setup.blocksize, trim_last=int(rng.integers(0, 30)))
             for _ in range(3)]
    return setup, workloads.build_dense_batch(setup, plans, rng, p_unused=0.05)


WORKLOADS = {
    "config2": (lambda: workloads.config2(P=300, streams=3, distinct=3, seed=21), "k_warp_synth"),
    "surround51": (lambda: workloads.config3(P=200, streams=2, distinct=2, seed=1), "k_warp_synth"),
    "wide_floors": (_wide_floor_workload, "k_warp_synth"),
    "fused_only": (_fused_only_workload, "k_fused_synth"),
}


def _padded(batch, channels, pad):
    """The same batch with every stream's channels `frames + pad` apart (pad a multiple of 4) and a gap of 4 to 7 samples
    before every stream, which keeps each destination's alignment (mod 4 samples) and hence the kernels' store paths."""
    st = batch.streams.copy()
    at = 0
    for i in range(len(st)):
        at = (at + 7) // 4 * 4 + int(batch.streams["pcm_base"][i]) % 4
        st["pcm_base"][i] = at
        st["pcm_frames"][i] = int(batch.streams["pcm_frames"][i]) + pad
        at += channels * int(st["pcm_frames"][i])
    return dataclasses.replace(batch, streams=st, pcm_floats=at + 3)


@pytest.mark.parametrize("staged", [False, True])
@pytest.mark.parametrize("pad", [4, 12])
@pytest.mark.parametrize("s16", [False, True])
@pytest.mark.parametrize("name", list(WORKLOADS))
def test_batch_upload_into_equals_fetch_pcm(contexts, name, s16, pad, staged):
    import torch
    ctx = contexts("default")
    make, kernel = WORKLOADS[name]
    setup, batch = make()
    sid = ctx.register_setup(setup)
    layout = abi.POV_PCM_PLANAR | (abi.POV_PCM_S16 if s16 else 0)
    plain = dataclasses.replace(batch, streams=batch.streams.copy(), pcm_layout=layout)
    plain.streams["setup_id"] = sid
    bh = ctx.upload(plain)
    assert ctx.kernel_name(bh) == kernel
    ctx.run_staged(bh) if staged else ctx.run(bh)
    ref = ctx.fetch_pcm(bh).copy()
    assert not ctx.status(bh).any()
    bh.free()
    padded = _padded(plain, setup.channels, pad)
    t = _sentinel_tensor(int(padded.pcm_floats), s16)
    launches = ctx.launch_count
    bh = ctx.upload(padded, pcm_out=t)
    assert ctx.pcm_dev_ptr(bh) == t.data_ptr()
    ctx.run_staged(bh) if staged else ctx.run(bh)
    assert ctx.launch_count > launches
    got = t.cpu().numpy()                                   # torch's stream waits for the run
    exp = np.full(int(padded.pcm_floats), SENTINEL_I16, np.int16) if s16 else np.full(int(padded.pcm_floats), np.nan, np.float32)
    for i in range(len(plain.streams)):
        f, b0, b1, s1 = (int(plain.streams["pcm_frames"][i]), int(plain.streams["pcm_base"][i]), int(padded.streams["pcm_base"][i]),
                         int(padded.streams["pcm_frames"][i]))
        for c in range(setup.channels):
            exp[b1 + c * s1:b1 + c * s1 + f] = ref[b0 + c * f:b0 + (c + 1) * f]
    assert _same_bits(got, exp)
    # the fetch call copies from the caller's memory; a plain upload through the same handle gets an arena again
    assert _same_bits(ctx.fetch_pcm(bh), exp)
    ctx.upload(plain, reuse=bh)
    assert ctx.pcm_dev_ptr(bh) not in (0, t.data_ptr())
    ctx.run_staged(bh) if staged else ctx.run(bh)
    assert _same_bits(ctx.fetch_pcm(bh), ref)
    bh.free()
    torch.cuda.synchronize()


def test_batch_upload_into_orders_both_ways(contexts):
    """Sleep + sentinel fill queued before the upload must land before the kernels' writes; a torch read queued after run()
    must see them."""
    import torch
    ctx = contexts("default")
    setup, batch = workloads.config2(P=400, streams=4, distinct=2, seed=5)
    batch.streams["setup_id"] = ctx.register_setup(setup)
    bh = ctx.upload(batch)
    ctx.run(bh)
    ref = ctx.fetch_pcm(bh).copy()
    bh.free()
    t = torch.zeros(int(batch.pcm_floats), dtype=torch.float32, device="cuda:0")
    torch.cuda.synchronize()
    s = torch.cuda.Stream()
    with torch.cuda.stream(s):
        torch.cuda._sleep(2_000_000_000)
        t.fill_(float("nan"))
        bh = ctx.upload(batch, pcm_out=t)
        ctx.run(bh)
        copy = t.clone()                                    # queued on torch's stream right after run()
    s.synchronize()
    assert _same_bits(copy.cpu().numpy(), ref)
    bh.free()


def test_batch_upload_into_refusals(contexts):
    import torch
    ctx = contexts("default")
    setup, batch = workloads.config2(P=64, streams=2, distinct=2, seed=9)
    batch.streams["setup_id"] = ctx.register_setup(setup)
    n = int(batch.pcm_floats)
    for bad in (torch.zeros(n, dtype=torch.int16, device="cuda:0"), torch.zeros(n - 1, device="cuda:0"),
                torch.zeros(n), torch.zeros(2 * n, device="cuda:0")[::2]):
        with pytest.raises(lib.PovError) as ei:
            ctx.upload(batch, pcm_out=bad)
        assert ei.value.code == abi.POV_ERR_ARG
    # the C call checks the pointer itself: host memory, misaligned device memory
    h = C.c_void_p(None)
    cb = batch.to_c()
    host = np.zeros(n, np.float32)
    assert ctx.L.pov_batch_upload_into(ctx.ctx, C.byref(cb), host.ctypes.data, C.byref(h)) == abi.POV_ERR_ARG
    t = torch.zeros(n + 1, device="cuda:0")
    assert ctx.L.pov_batch_upload_into(ctx.ctx, C.byref(cb), t.data_ptr() + 2, C.byref(h)) == abi.POV_ERR_ARG
    assert not h.value
