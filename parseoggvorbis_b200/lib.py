"""ctypes loader for libpov_synth.so (the C ABI of include/pov_synth.h) and a thin object wrapper.

There is no fallback of any kind: if the shared library is missing, or no sm_100 GPU is usable, every entry
point raises. All arithmetic of the decode path happens inside the CUDA kernels behind the C ABI.
"""
from __future__ import annotations

import ctypes as C
import os
from typing import Optional

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
]


SINK_FN = C.CFUNCTYPE(C.c_int, C.c_uint32, C.c_uint32, C.c_uint64, C.POINTER(C.c_float), C.c_void_p)
SINK_S16_FN = C.CFUNCTYPE(C.c_int, C.c_uint32, C.c_uint32, C.c_uint64, C.POINTER(C.c_int16), C.c_void_p)


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
    L.pov_parsed_stream_count.argtypes = [vp]
    L.pov_parsed_stream_count.restype = u32
    L.pov_parsed_get.argtypes = [vp, u32, C.POINTER(abi.pov_setup), C.POINTER(abi.pov_batch)]
    L.pov_parsed_free.argtypes = [vp]
    L.pov_parsed_free.restype = None
    _LIB = L
    return L


class ParsedOgg:
    """Host-only parse of one Ogg/Vorbis file into descriptor batches (no GPU involved)."""

    def __init__(self, data: bytes, raw_packets: bool = False, allow_spanning: bool = False):
        """raw_packets: leave the audio packets as they are (POV_INPUT_PACKETS batches: entropy decode on the device).
        allow_spanning: accept packets that continue on the next page (the reference refuses them, hpp:89)."""
        self.L = load()
        self.h = C.c_void_p(None)
        self._data = data
        err = C.c_char_p(None)
        rc = self.L.pov_ogg_parse_memory_ex(data, len(data), (1 if raw_packets else 0) | (2 if allow_spanning else 0), C.byref(self.h), C.byref(err))
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

    def upload(self, batch: abi.Batch, reuse: Optional[BatchHandle] = None) -> BatchHandle:
        bh = reuse if reuse is not None else BatchHandle(self, batch)
        bh.batch = batch
        cb = batch.to_c()
        self._check(self.L.pov_batch_upload(self.ctx, C.byref(cb), C.byref(bh.h)))
        return bh

    def run(self, bh: BatchHandle):
        self._check(self.L.pov_batch_run(self.ctx, bh.h))

    def kernel_name(self, bh: BatchHandle) -> str:
        """Kernel that run() launches for this batch (k_warp_synth / k_fused_synth / staged)."""
        return self.L.pov_batch_kernel_name(self.ctx, bh.h).decode()

    def run_staged(self, bh: BatchHandle):
        self._check(self.L.pov_batch_run_staged(self.ctx, bh.h))

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
        if s16:
            return self._decode_corpus_s16(files, None, host_threads)
        n = len(files)
        arr = (C.c_char_p * n)(*files)
        lens = (C.c_size_t * n)(*[len(f) for f in files])
        frames = np.zeros(n, np.uint64)
        total = C.c_uint64(0)
        chk = C.c_double(0)
        self._check(self.L.pov_decode_corpus(self.ctx, n, arr, lens, host_threads,
                                             frames.ctypes.data_as(C.POINTER(C.c_uint64)), C.byref(total), C.byref(chk)))
        return frames, int(total.value), float(chk.value)

    def decode_corpus_pcm(self, files, sink, host_threads: int = 0, s16: bool = False):
        """The corpus decode with its output edge (pov_decode_corpus_pcm): `sink(file_index, pcm)` is called from this thread
        for every logical stream, in file order, with a (channels, frames) float32 array that is only valid during the call;
        a true return value stops the decode (PovError, like the reference's CHECK(callbacks.gotPcmData(...))).
        s16: the arrays are int16 (pov_decode_corpus_s16) and the returned checksum is the exact integer sum."""
        if s16:
            return self._decode_corpus_s16(files, sink, host_threads)
        n = len(files)
        arr = (C.c_char_p * n)(*files)
        lens = (C.c_size_t * n)(*[len(f) for f in files])
        frames = np.zeros(n, np.uint64)
        total = C.c_uint64(0)
        chk = C.c_double(0)

        @SINK_FN
        def _sink(file_index, channels, nframes, planar, user):
            pcm = np.ctypeslib.as_array(planar, shape=(int(channels), int(nframes)))
            return 1 if sink(int(file_index), pcm) else 0
        self._check(self.L.pov_decode_corpus_pcm(self.ctx, n, arr, lens, host_threads, _sink, None,
                                                 frames.ctypes.data_as(C.POINTER(C.c_uint64)), C.byref(total), C.byref(chk)))
        return frames, int(total.value), float(chk.value)

    def _decode_corpus_s16(self, files, sink, host_threads: int):
        n = len(files)
        arr = (C.c_char_p * n)(*files)
        lens = (C.c_size_t * n)(*[len(f) for f in files])
        frames = np.zeros(n, np.uint64)
        total = C.c_uint64(0)
        chk = C.c_int64(0)
        _sink = C.cast(None, SINK_S16_FN)
        if sink is not None:
            @SINK_S16_FN
            def _sink(file_index, channels, nframes, planar, user):
                pcm = np.ctypeslib.as_array(planar, shape=(int(channels), int(nframes)))
                return 1 if sink(int(file_index), pcm) else 0
        self._check(self.L.pov_decode_corpus_s16(self.ctx, n, arr, lens, host_threads, _sink, None,
                                                 frames.ctypes.data_as(C.POINTER(C.c_uint64)), C.byref(total), C.byref(chk)))
        return frames, int(total.value), int(chk.value)
