"""ctypes loader for libpov_synth.so (the C ABI of include/pov_synth.h) and a thin object wrapper.

There is no fallback of any kind: if the shared library is missing, or no sm_100 GPU is usable, every entry
point raises. All arithmetic of the decode path happens inside the CUDA kernels behind the C ABI.
"""
from __future__ import annotations

import ctypes as C
import os
from typing import NamedTuple, Optional

import numpy as np

from . import abi

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("POV_LIB_PATH") or os.path.join(_HERE, "libpov_synth.so")   # override: A/B builds while tuning
_LIB: Optional[C.CDLL] = None

# every symbol include/pov_synth.h declares (tests/test_abi.py checks the header against this list and the .so)
SYMBOLS = [
    "pov_abi_version", "pov_inverse_db_table", "pov_window", "pov_ctx_create", "pov_ctx_destroy", "pov_last_error", "pov_ctx_stream",
    "pov_ctx_launch_count", "pov_ctx_io_bytes", "pov_ctx_set_device_entropy", "pov_ctx_set_page_spanning", "pov_ogg_parse_memory_ex", "pov_setup_register", "pov_setup_entry_bits", "pov_setup_get_window",
    "pov_batch_upload", "pov_batch_run", "pov_batch_kernel_name", "pov_batch_run_staged", "pov_batch_fetch_pcm", "pov_batch_fetch_pcm_s16", "pov_batch_pcm_dev",
    "pov_batch_fetch_stage", "pov_batch_status", "pov_batch_sync", "pov_batch_free", "pov_batch_features", "pov_batch_fetch_fast_floor", "pov_mdct_backward_batch",
    "pov_ogg_vorbis_decode_memory", "pov_decoded_free", "pov_decode_corpus", "pov_decode_corpus_pcm", "pov_ogg_vorbis_full_read_from_memory",
    "pov_ogg_vorbis_decode_memory_s16", "pov_decoded_s16_free", "pov_decode_corpus_s16",
    "pov_ogg_parse_memory", "pov_parsed_stream_count", "pov_parsed_get", "pov_parsed_free",
    "pov_batch_upload_into", "pov_corpus_streams", "pov_corpus_streams_free", "pov_decode_corpus_device",
    "pov_resample_filter", "pov_decode_corpus_device_resampled", "pov_ctx_set_cut_damage", "pov_corpus_report",
]


SINK_FN = C.CFUNCTYPE(C.c_int, C.c_uint32, C.c_uint32, C.c_uint64, C.POINTER(C.c_float), C.c_void_p)
SINK_S16_FN = C.CFUNCTYPE(C.c_int, C.c_uint32, C.c_uint32, C.c_uint64, C.POINTER(C.c_int16), C.c_void_p)


def _sink_fn(sink, fn_type):
    """`sink(file_index, pcm)` as a C sink of fn_type (SINK_FN / SINK_S16_FN), pcm a (channels, frames) view that is only
    valid during the call; a true return value asks the decode to stop. None: a null sink. Keep the result alive during the call."""
    if sink is None:
        return C.cast(None, fn_type)

    @fn_type
    def _sink(file_index, channels, nframes, planar, user):
        pcm = np.ctypeslib.as_array(planar, shape=(int(channels), int(nframes)))
        return 1 if sink(int(file_index), pcm) else 0
    return _sink


def _file_arrays(files):
    """The ctypes file-pointer and length arrays of a corpus call."""
    return (C.c_char_p * len(files))(*files), (C.c_size_t * len(files))(*[len(f) for f in files])


class PovError(RuntimeError):
    def __init__(self, code: int, msg: str):
        super().__init__("pov error %d: %s" % (code, msg))
        self.code = code
        self.msg = msg


def load() -> C.CDLL:
    """Load libpov_synth.so from the package directory (built in-tree by __graft_entry__.build())."""
    global _LIB
    if _LIB is not None:
        return _LIB
    if not os.path.exists(LIB_PATH):
        raise FileNotFoundError(
            "%s is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
            "(there is no CPU fallback)" % LIB_PATH)
    L = C.CDLL(LIB_PATH)
    vp, u32, u64, i32 = C.c_void_p, C.c_uint32, C.c_uint64, C.c_int
    L.pov_abi_version.restype = u32
    L.pov_inverse_db_table.argtypes = [C.POINTER(C.c_float)]
    L.pov_inverse_db_table.restype = None
    L.pov_ctx_create.argtypes = [i32, C.POINTER(vp), C.POINTER(C.c_char_p)]
    L.pov_ctx_destroy.argtypes = [vp]
    L.pov_ctx_destroy.restype = None
    L.pov_last_error.argtypes = [vp]
    L.pov_last_error.restype = C.c_char_p
    L.pov_ctx_stream.argtypes = [vp]
    L.pov_ctx_stream.restype = vp
    L.pov_ctx_launch_count.argtypes = [vp]
    L.pov_ctx_launch_count.restype = u64
    L.pov_ctx_io_bytes.argtypes = [vp, C.POINTER(u64), C.POINTER(u64)]
    L.pov_ctx_io_bytes.restype = None
    L.pov_setup_register.argtypes = [vp, C.POINTER(abi.pov_setup), C.POINTER(u32)]
    L.pov_setup_entry_bits.argtypes = [vp, u32]
    L.pov_window.argtypes = [u32, u32, i32, i32, i32, C.POINTER(C.c_float), u32]
    L.pov_window.restype = i32
    L.pov_setup_get_window.argtypes = [vp, u32, i32, i32, i32, C.POINTER(C.c_float), u32]
    L.pov_batch_upload.argtypes = [vp, C.POINTER(abi.pov_batch), C.POINTER(vp)]
    L.pov_batch_run.argtypes = [vp, vp]
    L.pov_batch_run_staged.argtypes = [vp, vp]
    L.pov_batch_kernel_name.argtypes = [vp, vp]
    L.pov_batch_kernel_name.restype = C.c_char_p
    L.pov_batch_fetch_pcm.argtypes = [vp, vp, C.POINTER(C.c_float), u64, i32]
    L.pov_batch_fetch_pcm_s16.argtypes = [vp, vp, C.POINTER(C.c_int16), u64, i32]
    L.pov_batch_pcm_dev.argtypes = [vp]
    L.pov_batch_pcm_dev.restype = vp
    L.pov_batch_fetch_stage.argtypes = [vp, vp, u32, u32, i32, vp, u64]
    L.pov_batch_status.argtypes = [vp, vp, C.POINTER(u32), u32]
    L.pov_batch_sync.argtypes = [vp, vp]
    L.pov_batch_free.argtypes = [vp, vp]
    L.pov_batch_free.restype = None
    L.pov_batch_fetch_fast_floor.argtypes = [vp, vp, C.POINTER(C.c_uint8), u64]
    L.pov_batch_features.argtypes = [vp, vp, u32, i32, u32, C.POINTER(C.c_float), u64, C.POINTER(u64)]
    L.pov_mdct_backward_batch.argtypes = [vp, u32, u64, C.POINTER(C.c_float), C.POINTER(C.c_float)]
    L.pov_ogg_vorbis_decode_memory.argtypes = [vp, C.c_char_p, C.c_size_t, C.c_char_p, C.POINTER(abi.pov_decoded)]
    L.pov_decoded_free.argtypes = [C.POINTER(abi.pov_decoded)]
    L.pov_decoded_free.restype = None
    L.pov_ogg_vorbis_decode_memory_s16.argtypes = [vp, C.c_char_p, C.c_size_t, C.POINTER(abi.pov_decoded_s16)]
    L.pov_decoded_s16_free.argtypes = [C.POINTER(abi.pov_decoded_s16)]
    L.pov_decoded_s16_free.restype = None
    L.pov_decode_corpus.argtypes = [vp, u32, C.POINTER(C.c_char_p), C.POINTER(C.c_size_t), u32,
                                    C.POINTER(u64), C.POINTER(u64), C.POINTER(C.c_double)]
    L.pov_decode_corpus_pcm.argtypes = [vp, u32, C.POINTER(C.c_char_p), C.POINTER(C.c_size_t), u32, SINK_FN, vp,
                                        C.POINTER(u64), C.POINTER(u64), C.POINTER(C.c_double)]
    L.pov_decode_corpus_s16.argtypes = [vp, u32, C.POINTER(C.c_char_p), C.POINTER(C.c_size_t), u32, SINK_S16_FN, vp,
                                        C.POINTER(u64), C.POINTER(u64), C.POINTER(C.c_int64)]
    L.pov_ogg_vorbis_full_read_from_memory.argtypes = [C.c_char_p, C.c_size_t, C.POINTER(C.c_char_p)]
    L.pov_ogg_parse_memory.argtypes = [C.c_char_p, C.c_size_t, C.POINTER(vp), C.POINTER(C.c_char_p)]
    L.pov_ogg_parse_memory_ex.argtypes = [C.c_char_p, C.c_size_t, u32, C.POINTER(vp), C.POINTER(C.c_char_p)]
    L.pov_ctx_set_device_entropy.argtypes = [vp, i32]
    L.pov_ctx_set_device_entropy.restype = None
    L.pov_ctx_set_page_spanning.argtypes = [vp, i32]
    L.pov_ctx_set_page_spanning.restype = None
    L.pov_ctx_set_cut_damage.argtypes = [vp, i32]
    L.pov_ctx_set_cut_damage.restype = None
    L.pov_corpus_report.argtypes = [vp, u32, C.POINTER(abi.pov_file_report), u64, C.POINTER(u64)]
    L.pov_parsed_stream_count.argtypes = [vp]
    L.pov_parsed_stream_count.restype = u32
    L.pov_parsed_get.argtypes = [vp, u32, C.POINTER(abi.pov_setup), C.POINTER(abi.pov_batch)]
    L.pov_parsed_free.argtypes = [vp]
    L.pov_parsed_free.restype = None
    L.pov_batch_upload_into.argtypes = [vp, C.POINTER(abi.pov_batch), vp, C.POINTER(vp)]
    L.pov_corpus_streams.argtypes = [u32, C.POINTER(C.c_char_p), C.POINTER(C.c_size_t), u32, u32,
                                     C.POINTER(C.POINTER(abi.pov_stream_info)), C.POINTER(u64), C.POINTER(C.c_char_p)]
    L.pov_corpus_streams_free.argtypes = [C.POINTER(abi.pov_stream_info)]
    L.pov_corpus_streams_free.restype = None
    L.pov_decode_corpus_device.argtypes = [vp, u32, C.POINTER(C.c_char_p), C.POINTER(C.c_size_t), u32, C.POINTER(abi.pov_device_pcm),
                                           C.POINTER(u64), C.POINTER(u64)]
    L.pov_resample_filter.argtypes = [u32, u32, C.POINTER(u32), C.POINTER(u32), C.POINTER(u32), C.POINTER(C.c_float), u32]
    L.pov_decode_corpus_device_resampled.argtypes = [vp, u32, C.POINTER(C.c_char_p), C.POINTER(C.c_size_t), u32,
                                                     C.POINTER(abi.pov_device_pcm), C.POINTER(abi.pov_resample),
                                                     C.POINTER(u64), C.POINTER(u64)]
    _LIB = L
    return L


class StreamTable(NamedTuple):
    """One entry per logical stream of a corpus, in decode order (pov_corpus_streams)."""
    file: np.ndarray           # uint32, index into the corpus
    channels: np.ndarray       # uint32
    sample_rate: np.ndarray    # uint32
    frames: np.ndarray         # uint64, frames per channel the decode yields

    def __len__(self):
        return len(self.file)


_STREAM_INFO_DTYPE = np.dtype([("file", "<u4"), ("channels", "<u4"), ("sample_rate", "<u4"), ("reserved", "<u4"), ("frames", "<u8")])
assert _STREAM_INFO_DTYPE.itemsize == C.sizeof(abi.pov_stream_info)


def corpus_streams(files, allow_spanning: bool = False, host_threads: int = 0, cut_damage: bool = False) -> StreamTable:
    """The stream table of a corpus without a GPU: the corpus decode's own parse with the packets discarded, so `frames` is
    what decode_corpus / decode_corpus_device produce. A framing or header error raises PovError with the corpus decode's
    text ("file k: check failed: ..."); with cut_damage (the table of a decode in cut mode) the damaged file's streams end
    there instead."""
    L = load()
    arr, lens = _file_arrays(files)
    out = C.POINTER(abi.pov_stream_info)()
    count = C.c_uint64(0)
    err = C.c_char_p(None)
    flags = (abi.POV_PARSE_ALLOW_SPANNING if allow_spanning else 0) | (abi.POV_PARSE_CUT_DAMAGE if cut_damage else 0)
    rc = L.pov_corpus_streams(len(files), arr, lens, flags, host_threads, C.byref(out), C.byref(count), C.byref(err))
    if rc != 0:
        raise PovError(rc, (err.value or b"?").decode())
    try:
        m = int(count.value)
        rec = np.ctypeslib.as_array(C.cast(out, C.POINTER(C.c_uint8)), shape=(m * C.sizeof(abi.pov_stream_info),)).view(
            _STREAM_INFO_DTYPE) if m else np.zeros(0, _STREAM_INFO_DTYPE)
        return StreamTable(rec["file"].copy(), rec["channels"].copy(), rec["sample_rate"].copy(), rec["frames"].copy())
    finally:
        L.pov_corpus_streams_free(out)


def _resample_ratio(in_rate: int, out_rate: int):
    """(L, M, half_len) of in_rate -> out_rate; PovError past the supported ratios."""
    up, down, hl = C.c_uint32(0), C.c_uint32(0), C.c_uint32(0)
    rc = load().pov_resample_filter(in_rate, out_rate, C.byref(up), C.byref(down), C.byref(hl), None, 0)
    if rc != 0:
        raise PovError(rc, "%d Hz -> %d Hz: max(L, M) = %d is past the supported %d (or a rate is 0)"
                       % (in_rate, out_rate, max(up.value, down.value), abi.POV_RESAMPLE_MAX_PHASES))
    return int(up.value), int(down.value), int(hl.value)


def resample_filter(in_rate: int, out_rate: int):
    """The in_rate -> out_rate filter of the resampled corpus decode, without a GPU: (up L, down M, half_len, float32 taps
    h[0 .. 2 half_len]). L = M = 1 is a copy: half_len 0 and no taps. scipy.signal.resample_poly's default design."""
    L, M, hl = _resample_ratio(in_rate, out_rate)
    if hl == 0:
        return L, M, 0, np.zeros(0, np.float32)
    taps = np.zeros(2 * hl + 1, np.float32)
    up, down, h = C.c_uint32(0), C.c_uint32(0), C.c_uint32(0)
    rc = load().pov_resample_filter(in_rate, out_rate, C.byref(up), C.byref(down), C.byref(h),
                                    taps.ctypes.data_as(C.POINTER(C.c_float)), len(taps))
    if rc != 0:
        raise PovError(rc, "pov_resample_filter")
    return L, M, hl, taps


def resampled_frames(table: "StreamTable", out_rate: int) -> np.ndarray:
    """uint64 output frames per record of `table` at out_rate (0: every stream keeps its rate): ceil(frames L / M)."""
    frames = np.asarray(table.frames, np.uint64)
    out = frames.copy()
    if out_rate == 0:
        return out
    rates = np.asarray(table.sample_rate, np.uint32)
    for r in np.unique(rates):
        L, M, _ = _resample_ratio(int(r), int(out_rate))
        sel = rates == r
        out[sel] = (frames[sel] * np.uint64(L) + np.uint64(M - 1)) // np.uint64(M)
    return out


def _round4(x):
    return (np.asarray(x, np.uint64) + np.uint64(3)) // np.uint64(4) * np.uint64(4)


class DeviceCorpus(NamedTuple):
    """What decode_corpus_device returns: the PCM tensor, the stream table and where each stream lives in the tensor."""
    pcm: "object"              # torch tensor on the context's device
    table: StreamTable
    base: np.ndarray           # uint64 [streams], sample index of channel 0, frame 0 (in pcm's flat storage)
    stride: np.ndarray         # uint64 [streams], samples between channels
    frames_per_file: np.ndarray
    total_values: int
    sample_rate: Optional[int] = None        # resampled / downmixed decode: the target rate (0 = each stream's own rate)
    out_channels: Optional[np.ndarray] = None   # uint32 [streams], channels written per stream
    out_frames: Optional[np.ndarray] = None     # uint64 [streams], frames written per stream
    valid_frames: Optional[np.ndarray] = None   # uint64 [streams], native frames before each stream's cut (= table.frames if clean)
    damaged: Optional[dict] = None              # {file index: message} of the damaged files (cut mode; {} when none is)

    def stream(self, i: int):
        """(channels, frames) view of stream i (output channels and frames of a resampled / downmixed decode)."""
        if self.out_frames is not None:
            c, f = int(self.out_channels[i]), int(self.out_frames[i])
        else:
            c, f = int(self.table.channels[i]), int(self.table.frames[i])
        if self.pcm.dim() == 3:
            return self.pcm[i, :c, :f]
        b, s = int(self.base[i]), int(self.stride[i])
        return self.pcm[b:b + c * s].view(c, s)[:, :f]


class CorpusReport(NamedTuple):
    """pov_corpus_report: what the context's last successful corpus call found, per file and per stream-table record."""
    status: np.ndarray          # uint32 [files]: POV_OK, or POV_ERR_STREAM (damaged and cut)
    n_streams: np.ndarray       # uint32 [files]: records of the file
    frames: np.ndarray          # uint64 [files]: = frames_out
    valid_frames: np.ndarray    # uint64 [files]: summed over the file's streams
    messages: list              # str [files]: "" or the reason
    stream_valid_frames: np.ndarray   # uint64 [records]

    @property
    def damaged(self) -> dict:
        return {i: m for i, (st, m) in enumerate(zip(self.status, self.messages)) if st != abi.POV_OK}


class ParsedOgg:
    """Host-only parse of one Ogg/Vorbis file into descriptor batches (no GPU involved)."""

    def __init__(self, data: bytes, raw_packets: bool = False, allow_spanning: bool = False, cut_damage: bool = False):
        """raw_packets: leave the audio packets as they are (POV_INPUT_PACKETS batches: entropy decode on the device).
        allow_spanning: accept packets that continue on the next page (the reference refuses them, hpp:89).
        cut_damage: damage ends the parse with the packets before it (POV_PARSE_CUT_DAMAGE)."""
        self.L = load()
        self.h = C.c_void_p(None)
        self._data = data
        err = C.c_char_p(None)
        flags = ((abi.POV_PARSE_RAW_PACKETS if raw_packets else 0) | (abi.POV_PARSE_ALLOW_SPANNING if allow_spanning else 0) |
                 (abi.POV_PARSE_CUT_DAMAGE if cut_damage else 0))
        rc = self.L.pov_ogg_parse_memory_ex(data, len(data), flags, C.byref(self.h), C.byref(err))
        if rc != 0:
            raise PovError(rc, (err.value or b"?").decode())

    @property
    def n_streams(self) -> int:
        return int(self.L.pov_parsed_stream_count(self.h))

    def get(self, stream: int = 0):
        """-> (pov_setup, pov_batch) ctypes structs pointing into this handle's memory."""
        s, b = abi.pov_setup(), abi.pov_batch()
        rc = self.L.pov_parsed_get(self.h, stream, C.byref(s), C.byref(b))
        if rc != 0:
            raise PovError(rc, "pov_parsed_get")
        return s, b

    def close(self):
        if self.h:
            self.L.pov_parsed_free(self.h)
            self.h = C.c_void_p(None)

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class BatchHandle:
    def __init__(self, ctx: "SynthContext", batch: abi.Batch):
        self.ctx = ctx
        self.batch = batch          # keeps the host arrays alive
        self.h = C.c_void_p(None)
        self.pcm_out = None         # upload(pcm_out=...): the caller's tensor the kernels write

    def free(self):
        if self.h:
            self.ctx.L.pov_batch_free(self.ctx.ctx, self.h)
            self.h = C.c_void_p(None)

    def __del__(self):
        try:
            self.free()
        except Exception:
            pass


class SynthContext:
    """One context per (thread, GPU) — mirrors the reference's "one decoder per thread" rule (Callbacks.h:16-21)."""

    def __init__(self, device: int = 0):
        self.L = load()
        self.ctx = C.c_void_p(None)
        err = C.c_char_p(None)
        rc = self.L.pov_ctx_create(device, C.byref(self.ctx), C.byref(err))
        if rc != 0:
            raise PovError(rc, (err.value or b"?").decode())
        self._setups = []
        self.device = device
        self._spanning = int(os.environ.get("POV_ALLOW_SPANNING", "0") or 0) != 0     # the context's default (api.cu)
        self._cut = False
        self._corpus_files = None           # files of the last successful corpus call (corpus_report)

    def close(self):
        if self.ctx:
            self.L.pov_ctx_destroy(self.ctx)
            self.ctx = C.c_void_p(None)

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _check(self, rc: int):
        if rc != 0:
            raise PovError(rc, self.L.pov_last_error(self.ctx).decode())

    @property
    def stream_ptr(self) -> int:
        return int(self.L.pov_ctx_stream(self.ctx) or 0)

    @property
    def launch_count(self) -> int:
        return int(self.L.pov_ctx_launch_count(self.ctx))

    def set_page_spanning(self, on: bool):
        self.L.pov_ctx_set_page_spanning(self.ctx, 1 if on else 0)
        self._spanning = bool(on)

    def set_cut_damage(self, on: bool):
        """Cut mode of every corpus call on this context (pov_ctx_set_cut_damage): a damaged stream ends where its damage
        starts, the call goes on, and corpus_report() says what happened to each file."""
        self.L.pov_ctx_set_cut_damage(self.ctx, 1 if on else 0)
        self._cut = bool(on)

    def corpus_report(self) -> CorpusReport:
        """The report of the last successful corpus call on this context (PovError when there is none)."""
        if self._corpus_files is None:
            raise PovError(abi.POV_ERR_ARG, "corpus_report: no successful corpus call on this context")
        n = self._corpus_files
        files = (abi.pov_file_report * max(1, n))()
        self._check(self.L.pov_corpus_report(self.ctx, n, files, 0, None))
        rows = [files[i] for i in range(n)]
        m = sum(int(r.n_streams) for r in rows)
        valid = np.zeros(m, np.uint64)
        self._check(self.L.pov_corpus_report(self.ctx, n, files, m, valid.ctypes.data_as(C.POINTER(C.c_uint64))))
        return CorpusReport(np.array([r.status for r in rows], np.uint32), np.array([r.n_streams for r in rows], np.uint32),
                            np.array([r.frames for r in rows], np.uint64), np.array([r.valid_frames for r in rows], np.uint64),
                            [r.message.decode() for r in rows], valid)

    def set_device_entropy(self, on: bool):
        self.L.pov_ctx_set_device_entropy(self.ctx, 1 if on else 0)

    def io_bytes(self):
        """(host -> device, device -> host) bytes this context has copied so far."""
        a, b = C.c_uint64(0), C.c_uint64(0)
        self.L.pov_ctx_io_bytes(self.ctx, C.byref(a), C.byref(b))
        return int(a.value), int(b.value)

    def register_setup(self, setup: abi.Setup) -> int:
        cs = setup.to_c()
        sid = C.c_uint32(0)
        self._check(self.L.pov_setup_register(self.ctx, C.byref(cs.c), C.byref(sid)))
        self._setups.append(cs)
        return int(sid.value)

    def window(self, setup_id: int, blockflag: int, prev: int, nxt: int, n: int) -> np.ndarray:
        out = np.zeros(n, np.float32)
        self._check(self.L.pov_setup_get_window(self.ctx, setup_id, blockflag, prev, nxt,
                                                out.ctypes.data_as(C.POINTER(C.c_float)), n))
        return out

    def _pcm_tensor(self, t, s16: bool, samples: int, what: str):
        """Checks of a caller's PCM tensor: contiguous, on this context's GPU, dtype of the format, room for `samples`."""
        import torch
        want = torch.int16 if s16 else torch.float32
        if not isinstance(t, torch.Tensor) or t.device != torch.device("cuda", self.device) or not t.is_contiguous():
            raise PovError(abi.POV_ERR_ARG, "%s: a contiguous tensor on cuda:%d is needed" % (what, self.device))
        if t.dtype != want:
            raise PovError(abi.POV_ERR_ARG, "%s: dtype %s, the format needs %s" % (what, t.dtype, want))
        if t.numel() < samples:
            raise PovError(abi.POV_ERR_ARG, "%s: %d samples, %d needed" % (what, t.numel(), samples))

    def _ctx_stream(self):
        import torch
        return torch.cuda.ExternalStream(self.stream_ptr, device=torch.device("cuda", self.device))

    def upload(self, batch: abi.Batch, reuse: Optional[BatchHandle] = None, pcm_out=None) -> BatchHandle:
        """pcm_out: a contiguous CUDA tensor on this context's device (float32, or int16 for a POV_PCM_S16 batch) with room for
        batch.pcm_floats samples; the kernels then write the PCM there (pov_batch_upload_into) instead of the handle's arena.
        The context's stream is ordered after the work queued on torch's current stream, and run() / run_staged() make the
        current stream wait for the kernels, so the tensor is used in plain stream order on both sides."""
        bh = reuse if reuse is not None else BatchHandle(self, batch)
        bh.batch = batch
        cb = batch.to_c()
        if pcm_out is None:
            bh.pcm_out = None
            self._check(self.L.pov_batch_upload(self.ctx, C.byref(cb), C.byref(bh.h)))
            return bh
        import torch
        self._pcm_tensor(pcm_out, bool(batch.pcm_layout & abi.POV_PCM_S16), int(batch.pcm_floats), "upload(pcm_out)")
        ev = torch.cuda.Event()
        ev.record(torch.cuda.current_stream(self.device))
        self._ctx_stream().wait_event(ev)
        self._check(self.L.pov_batch_upload_into(self.ctx, C.byref(cb), C.c_void_p(pcm_out.data_ptr()), C.byref(bh.h)))
        bh.pcm_out = pcm_out
        return bh

    def _after_run(self, bh: BatchHandle):
        if bh.pcm_out is not None:          # torch's current stream waits for the kernels that write the caller's tensor
            import torch
            ev = torch.cuda.Event()
            ev.record(self._ctx_stream())
            torch.cuda.current_stream(self.device).wait_event(ev)

    def run(self, bh: BatchHandle):
        self._check(self.L.pov_batch_run(self.ctx, bh.h))
        self._after_run(bh)

    def kernel_name(self, bh: BatchHandle) -> str:
        """Kernel that run() launches for this batch (k_warp_synth / k_fused_synth / staged)."""
        return self.L.pov_batch_kernel_name(self.ctx, bh.h).decode()

    def run_staged(self, bh: BatchHandle):
        self._check(self.L.pov_batch_run_staged(self.ctx, bh.h))
        self._after_run(bh)

    def sync(self, bh: BatchHandle):
        self._check(self.L.pov_batch_sync(self.ctx, bh.h))

    def fetch_pcm(self, bh: BatchHandle, out: Optional[np.ndarray] = None, sync: bool = True) -> np.ndarray:
        """The batch's PCM arena: float32, or int16 for a batch uploaded with pcm_layout | POV_PCM_S16."""
        n = int(bh.batch.pcm_floats)
        if bh.batch.pcm_layout & abi.POV_PCM_S16:
            return self.fetch_pcm_s16(bh, out, sync)
        if out is None:
            out = np.empty(n, np.float32)
        self._check(self.L.pov_batch_fetch_pcm(self.ctx, bh.h, out.ctypes.data_as(C.POINTER(C.c_float)), n, int(sync)))
        return out

    def fetch_pcm_s16(self, bh: BatchHandle, out: Optional[np.ndarray] = None, sync: bool = True) -> np.ndarray:
        """pov_batch_fetch_pcm_s16: the int16 arena of a POV_PCM_S16 batch (PovError on a float32 batch)."""
        n = int(bh.batch.pcm_floats)
        if out is None:
            out = np.empty(n, np.int16)
        self._check(self.L.pov_batch_fetch_pcm_s16(self.ctx, bh.h, out.ctypes.data_as(C.POINTER(C.c_int16)), n, int(sync)))
        return out

    def pcm_dev_ptr(self, bh: BatchHandle) -> int:
        return int(self.L.pov_batch_pcm_dev(bh.h) or 0)

    def status(self, bh: BatchHandle, check: bool = False) -> np.ndarray:
        st = np.zeros(len(bh.batch.packets), np.uint32)
        rc = self.L.pov_batch_status(self.ctx, bh.h, st.ctypes.data_as(C.POINTER(C.c_uint32)), len(st))
        if check:
            self._check(rc)
        return st

    _STAGE_DTYPE = {abi.POV_STAGE_FINAL_YS: np.uint32, abi.POV_STAGE_STEP2_FLAG: np.uint8,
                    abi.POV_STAGE_FLOOR: np.uint32, abi.POV_STAGE_FLOOR_OUTPUTS: np.float32,
                    abi.POV_STAGE_AFTER_RESIDUE: np.float32, abi.POV_STAGE_AFTER_ENVELOPE: np.float32,
                    abi.POV_STAGE_PCM_AFTER_MDCT: np.float32}

    def fetch_stage(self, bh: BatchHandle, packet: int, channel: int, stage: int, count: int) -> np.ndarray:
        out = np.zeros(count, self._STAGE_DTYPE[stage])
        self._check(self.L.pov_batch_fetch_stage(self.ctx, bh.h, packet, channel, stage, out.ctypes.data, out.nbytes))
        return out

    def mdct_backward(self, x: np.ndarray) -> np.ndarray:
        """Batched drop-in for the reference's mdct_backward (src/mdct.h:105): x [count, n/2] -> [count, n]."""
        x = np.ascontiguousarray(x, np.float32)
        count, half = x.shape
        out = np.empty((count, 2 * half), np.float32)
        self._check(self.L.pov_mdct_backward_batch(self.ctx, 2 * half, count, x.ctypes.data_as(C.POINTER(C.c_float)),
                                                   out.ctypes.data_as(C.POINTER(C.c_float))))
        return out

    def decode_ogg(self, data: bytes, debug_out: Optional[str] = None, s16: bool = False):
        """Whole-file decode through the host front-end + GPU. Returns (pcm [C, frames], sample_rate, n_packets).
        s16: int16 PCM converted on the device (pov_ogg_vorbis_decode_memory_s16; no debug dump)."""
        if s16:
            if debug_out:
                raise ValueError("the debug dump is float32: decode_ogg(s16=True) takes no debug_out")
            d, dtype, free = abi.pov_decoded_s16(), np.int16, self.L.pov_decoded_s16_free
            self._check(self.L.pov_ogg_vorbis_decode_memory_s16(self.ctx, data, len(data), C.byref(d)))
        else:
            d, dtype, free = abi.pov_decoded(), np.float32, self.L.pov_decoded_free
            dbg = debug_out.encode() if debug_out else None
            self._check(self.L.pov_ogg_vorbis_decode_memory(self.ctx, data, len(data), dbg, C.byref(d)))
        try:
            n = int(d.channels) * int(d.frames)
            pcm = np.ctypeslib.as_array(d.pcm, shape=(n,)).copy().reshape(int(d.channels), int(d.frames)) if n else \
                np.zeros((int(d.channels), 0), dtype)
            return pcm, int(d.sample_rate), int(d.audio_packets)
        finally:
            free(C.byref(d))

    FEATURE_KINDS = {"floor_final_ys": 0, "floor_final_ys_rendered": 1, "residue_ys": 2, "residue_ys_with_floor": 3}

    def features_from_raw_bytes(self, raw_bytes: bytes, output_dim: int, kind: str = "floor_final_ys", raw_packets: bool = True):
        """The device-side counterpart of returnn_import.ParseOggVorbisLib.get_features_from_raw_bytes (reference:
        returnn_import.py:74-115), default reader arguments: a (time, output_dim) float32 matrix for the first logical
        stream of an Ogg/Vorbis file. Only the matrix comes back from the device."""
        po = ParsedOgg(raw_bytes, raw_packets=raw_packets)
        try:
            s, b = po.get(0)
            sid = C.c_uint32(0)
            self._check(self.L.pov_setup_register(self.ctx, C.byref(s), C.byref(sid)))
            st = abi.pov_stream.from_address(C.addressof(b.streams.contents))
            st.setup_id = sid.value
            h = C.c_void_p(None)
            try:
                self._check(self.L.pov_batch_upload(self.ctx, C.byref(b), C.byref(h)))
                rows = C.c_uint64(0)
                k = self.FEATURE_KINDS[kind]
                self._check(self.L.pov_batch_features(self.ctx, h, 0, k, output_dim, None, 0, C.byref(rows)))
                out = np.zeros((int(rows.value), output_dim), np.float32)
                self._check(self.L.pov_batch_features(self.ctx, h, 0, k, output_dim, out.ctypes.data_as(C.POINTER(C.c_float)),
                                                      rows.value, C.byref(rows)))
                return out
            finally:
                st.setup_id = 0
                if h:
                    self.L.pov_batch_free(self.ctx, h)
        finally:
            po.close()

    def decode_corpus(self, files, host_threads: int = 0, s16: bool = False):
        """files: list of bytes. Returns (frames per file, total PCM values, checksum). s16: int16 PCM (pov_decode_corpus_s16,
        half the device -> host bytes); the checksum is then the exact integer sum of every sample."""
        return self.decode_corpus_pcm(files, None, host_threads, s16)

    def decode_corpus_pcm(self, files, sink, host_threads: int = 0, s16: bool = False):
        """The corpus decode with its output edge (pov_decode_corpus_pcm): `sink(file_index, pcm)` is called from this thread
        for every logical stream, in file order, with a (channels, frames) float32 array that is only valid during the call;
        a true return value stops the decode (PovError, like the reference's CHECK(callbacks.gotPcmData(...))).
        s16: the arrays are int16 (pov_decode_corpus_s16) and the returned checksum is the exact integer sum."""
        if s16:
            fn, chk, sink_args = self.L.pov_decode_corpus_s16, C.c_int64(0), (_sink_fn(sink, SINK_S16_FN), None)
        elif sink is None:
            fn, chk, sink_args = self.L.pov_decode_corpus, C.c_double(0), ()
        else:
            fn, chk, sink_args = self.L.pov_decode_corpus_pcm, C.c_double(0), (_sink_fn(sink, SINK_FN), None)
        frames, total = self._decode_corpus_call(fn, files, host_threads, sink_args, (C.byref(chk),))
        return frames, total, chk.value

    def _decode_corpus_call(self, fn, files, host_threads: int, before=(), after=()):
        """fn(ctx, n, files, lengths, host_threads, *before, frames, &total, *after), one of the pov_decode_corpus* calls.
        Returns (frames per file, total PCM values)."""
        arr, lens = _file_arrays(files)
        frames = np.zeros(len(files), np.uint64)
        total = C.c_uint64(0)
        self._corpus_files = None
        self._check(fn(self.ctx, len(files), arr, lens, host_threads, *before, frames.ctypes.data_as(C.POINTER(C.c_uint64)),
                       C.byref(total), *after))
        self._corpus_files = len(files)
        return frames, int(total.value)

    def decode_corpus_into(self, files, pcm, table: StreamTable, base, stride, s16: bool = False, host_threads: int = 0,
                           sample_rate: Optional[int] = None, mono: bool = False):
        """pov_decode_corpus_device into a tensor the caller laid out: stream i of `table`, channel c, frame f lands at flat
        sample index base[i] + c * stride[i] + f of `pcm` (contiguous, on this context's GPU, float32 or int16 with s16).
        Nothing else of `pcm` is written. No PCM write starts before the work queued on torch's current stream, and the call
        returns when the PCM is complete. Returns (frames per file, total PCM values).
        sample_rate / mono: every stream resampled to sample_rate (0: its own rate) and / or averaged to one channel on the
        device (pov_decode_corpus_device_resampled); channels and frames are then the output's (resampled_frames)."""
        import torch
        m = len(table)
        base = np.ascontiguousarray(base, np.uint64)
        stride = np.ascontiguousarray(stride, np.uint64)
        if base.shape != (m,) or stride.shape != (m,):
            raise PovError(abi.POV_ERR_ARG, "decode_corpus_into: base and stride need one entry per stream-table record")
        self._pcm_tensor(pcm, s16, 0, "decode_corpus_into(pcm)")
        file = np.ascontiguousarray(table.file, np.uint32)
        channels = np.ascontiguousarray(table.channels, np.uint32)
        tframes = np.ascontiguousarray(table.frames, np.uint64)
        o = abi.pov_device_pcm()
        o.pcm_layout = abi.POV_PCM_PLANAR | (abi.POV_PCM_S16 if s16 else 0)
        o.n_streams = m
        o.pcm_dev = pcm.data_ptr() or None
        o.capacity = pcm.numel()
        o.stream_base = base.ctypes.data_as(C.POINTER(C.c_uint64))
        o.channel_stride = stride.ctypes.data_as(C.POINTER(C.c_uint64))
        o.file = file.ctypes.data_as(C.POINTER(C.c_uint32))
        o.channels = channels.ctypes.data_as(C.POINTER(C.c_uint32))
        o.frames = tframes.ctypes.data_as(C.POINTER(C.c_uint64))
        o.cuda_stream = torch.cuda.current_stream(self.device).cuda_stream or None
        if sample_rate is None and not mono:
            return self._decode_corpus_call(self.L.pov_decode_corpus_device, files, host_threads, (C.byref(o),))
        rates = np.ascontiguousarray(table.sample_rate, np.uint32)
        rs = abi.pov_resample()
        rs.out_rate = int(sample_rate or 0)
        rs.flags = abi.POV_RESAMPLE_MONO if mono else 0
        rs.sample_rate = rates.ctypes.data_as(C.POINTER(C.c_uint32))
        return self._decode_corpus_call(self.L.pov_decode_corpus_device_resampled, files, host_threads, (C.byref(o), C.byref(rs)))

    def decode_corpus_device(self, files, layout: str = "padded", s16: bool = False, host_threads: int = 0,
                             sample_rate: Optional[int] = None, mono: bool = False, cut_damage: bool = False) -> DeviceCorpus:
        """Decode a corpus straight into a new torch tensor on this context's GPU; only compressed packets go to the device
        and only status words come back. layout "padded": (streams, max channels, T) zeros, T = the longest stream rounded
        up to 4; "packed": one flat tensor, each stream's channels `frames rounded up to 4` apart, back to back. Padding
        stays 0. s16: int16 samples (the POV_PCM_S16 conversion). The stream table is parsed with this context's page-spanning
        setting. sample_rate (Hz, 0 = each stream's own) and mono resample / downmix every stream on the device, and the
        layouts are then sized by output channels and frames (DeviceCorpus.out_channels / out_frames).
        cut_damage: cut mode for this call (table and decode); DeviceCorpus.valid_frames and .damaged come from the report."""
        was = self._cut
        self.set_cut_damage(cut_damage)
        try:
            out = self._decode_corpus_device(files, layout, s16, host_threads, sample_rate, mono)
        finally:
            self.set_cut_damage(was)
        rep = self.corpus_report()
        return out._replace(valid_frames=rep.stream_valid_frames, damaged=rep.damaged)

    def _decode_corpus_device(self, files, layout, s16, host_threads, sample_rate, mono) -> DeviceCorpus:
        import torch
        table = corpus_streams(files, allow_spanning=self._spanning, host_threads=host_threads, cut_damage=self._cut)
        m = len(table)
        resampled = sample_rate is not None or mono
        if resampled:
            out_frames = resampled_frames(table, int(sample_rate or 0))
            out_channels = np.ones(m, np.uint32) if mono else table.channels.astype(np.uint32)
            table_frames = out_frames
        else:
            out_frames = out_channels = None
            table_frames = table.frames
        ch = (out_channels if resampled else table.channels).astype(np.uint64)
        dtype = torch.int16 if s16 else torch.float32
        dev = torch.device("cuda", self.device)
        if layout == "padded":
            T = int(_round4(table_frames.max())) if m else 0
            maxc = int(ch.max()) if m else 0
            pcm = torch.zeros((m, maxc, T), dtype=dtype, device=dev)
            stride = np.full(m, T, np.uint64)
            base = np.arange(m, dtype=np.uint64) * np.uint64(maxc * T)
        elif layout == "packed":
            stride = _round4(table_frames)
            sizes = ch * stride
            base = (np.cumsum(sizes) - sizes).astype(np.uint64)
            pcm = torch.zeros(int(sizes.sum()), dtype=dtype, device=dev)
        else:
            raise ValueError("layout must be 'padded' or 'packed'")
        frames, total = self.decode_corpus_into(files, pcm, table, base, stride, s16=s16, host_threads=host_threads,
                                                sample_rate=sample_rate, mono=mono)
        if not resampled:
            return DeviceCorpus(pcm, table, base, stride, frames, total)
        return DeviceCorpus(pcm, table, base, stride, frames, total, int(sample_rate or 0), out_channels, out_frames)
