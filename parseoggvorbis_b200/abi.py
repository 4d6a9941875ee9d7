"""ctypes mirror of include/pov_synth.h (POD structs only) plus numpy-friendly builders.

The struct layouts here must match the header field for field; tests/test_abi.py cross-checks every sizeof
against the C compiler's. Nothing in this module computes anything on the decode path.
"""
from __future__ import annotations

import ctypes as C
from dataclasses import dataclass, field
from typing import List, Optional, Sequence

import numpy as np

POV_ABI_VERSION = 2
POV_MAX_CHANNELS = 8
POV_MAX_POSTS = 256
POV_MAX_COUPLINGS = 256
POV_MAX_SUBMAPS = 16
POV_MAX_CLASSES = 64
POV_MAX_MODES = 64
POV_NO_BOOK = 255

POV_OK, POV_ERR_ARG, POV_ERR_CUDA, POV_ERR_STREAM, POV_ERR_UNSUPPORTED = range(5)
POV_PKT_OK, POV_PKT_FLOOR_PREDICTED, POV_PKT_FLOOR_RANGE, POV_PKT_VQ_ENTRY = 0, 1, 2, 4
POV_INPUT_DENSE, POV_INPUT_ENTRIES, POV_INPUT_PACKETS = 0, 1, 2
POV_PCM_PLANAR, POV_PCM_INTERLEAVED = 0, 1
POV_PCM_S16 = 0x100          # OR-ed into pcm_layout: the kernels store int16 PCM (see include/pov_synth.h)
POV_PARSE_RAW_PACKETS, POV_PARSE_ALLOW_SPANNING = 1, 2     # flags of pov_ogg_parse_memory_ex / pov_corpus_streams
POV_PARSE_CUT_DAMAGE = 4     # cut mode: damage ends the damaged stream instead of failing (see include/pov_synth.h)
POV_RESAMPLE_MONO = 1        # pov_resample.flags: average the channels before resampling
POV_RESAMPLE_MAX_PHASES = 2048   # largest max(L, M) of a supported resampling ratio

(POV_STAGE_FINAL_YS, POV_STAGE_STEP2_FLAG, POV_STAGE_FLOOR, POV_STAGE_FLOOR_OUTPUTS,
 POV_STAGE_AFTER_RESIDUE, POV_STAGE_AFTER_ENVELOPE, POV_STAGE_PCM_AFTER_MDCT) = range(7)


class pov_codebook(C.Structure):
    _fields_ = [("dim", C.c_uint32), ("n_entries", C.c_uint32), ("lookup_type", C.c_uint32),
                ("reserved", C.c_uint32), ("vq", C.POINTER(C.c_float)), ("lengths", C.POINTER(C.c_uint8))]


class pov_floor1_syntax(C.Structure):
    _fields_ = [("n_partitions", C.c_uint8), ("n_classes", C.c_uint8), ("reserved", C.c_uint8 * 2),
                ("partition_class", C.c_uint8 * 32), ("class_dim", C.c_uint8 * 16),
                ("class_subclass_bits", C.c_uint8 * 16), ("class_masterbook", C.c_uint8 * 16),
                ("class_books", (C.c_int16 * 8) * 16)]


class pov_floor1(C.Structure):
    _fields_ = [("n_posts", C.c_uint16), ("multiplier", C.c_uint8), ("reserved", C.c_uint8),
                ("xs", C.c_uint16 * POV_MAX_POSTS)]


class pov_residue(C.Structure):
    _fields_ = [("type", C.c_uint32), ("begin", C.c_uint32), ("end", C.c_uint32),
                ("partition_size", C.c_uint32), ("n_class", C.c_uint32), ("classbook", C.c_uint32),
                ("books", C.c_uint8 * (POV_MAX_CLASSES * 8))]


class pov_mapping(C.Structure):
    _fields_ = [("n_submaps", C.c_uint32), ("n_couplings", C.c_uint32),
                ("mux", C.c_uint8 * POV_MAX_CHANNELS),
                ("submap_floor", C.c_uint8 * POV_MAX_SUBMAPS),
                ("submap_residue", C.c_uint8 * POV_MAX_SUBMAPS),
                ("coupling_mag", C.c_uint8 * POV_MAX_COUPLINGS),
                ("coupling_ang", C.c_uint8 * POV_MAX_COUPLINGS)]


class pov_mode(C.Structure):
    _fields_ = [("blockflag", C.c_uint8), ("mapping", C.c_uint8)]


class pov_setup(C.Structure):
    _fields_ = [("abi_version", C.c_uint32), ("channels", C.c_uint32), ("sample_rate", C.c_uint32),
                ("blocksize", C.c_uint32 * 2),
                ("n_codebooks", C.c_uint32), ("codebooks", C.POINTER(pov_codebook)),
                ("n_floors", C.c_uint32), ("floors", C.POINTER(pov_floor1)),
                ("n_residues", C.c_uint32), ("residues", C.POINTER(pov_residue)),
                ("n_mappings", C.c_uint32), ("mappings", C.POINTER(pov_mapping)),
                ("n_modes", C.c_uint32), ("modes", C.POINTER(pov_mode)),
                ("floor_syntax", C.POINTER(pov_floor1_syntax))]


class pov_stream(C.Structure):
    _fields_ = [("setup_id", C.c_uint32), ("first_packet", C.c_uint32), ("n_packets", C.c_uint32),
                ("reserved", C.c_uint32), ("pcm_frames", C.c_uint64), ("pcm_base", C.c_uint64)]


class pov_packet(C.Structure):
    _fields_ = [("stream", C.c_uint32), ("mode", C.c_uint8), ("window_flags", C.c_uint8),
                ("floor_used", C.c_uint16), ("emit_frames", C.c_uint32), ("packet_bytes", C.c_uint32),
                ("pcm_off", C.c_uint64), ("ys_off", C.c_uint64), ("spec_off", C.c_uint64)]


class pov_batch(C.Structure):
    _fields_ = [("input_kind", C.c_uint32), ("pcm_layout", C.c_uint32),
                ("n_streams", C.c_uint32), ("streams", C.POINTER(pov_stream)),
                ("n_packets", C.c_uint32), ("packets", C.POINTER(pov_packet)),
                ("ys", C.POINTER(C.c_uint16)), ("n_ys", C.c_uint64),
                ("payload", C.c_void_p), ("payload_bytes", C.c_uint64),
                ("pcm_floats", C.c_uint64)]


class pov_decoded(C.Structure):
    _fields_ = [("channels", C.c_uint32), ("sample_rate", C.c_uint32), ("frames", C.c_uint64),
                ("audio_packets", C.c_uint32), ("reserved", C.c_uint32), ("pcm", C.POINTER(C.c_float))]


class pov_decoded_s16(C.Structure):
    _fields_ = [("channels", C.c_uint32), ("sample_rate", C.c_uint32), ("frames", C.c_uint64),
                ("audio_packets", C.c_uint32), ("reserved", C.c_uint32), ("pcm", C.POINTER(C.c_int16))]


class pov_stream_info(C.Structure):
    """One record of pov_corpus_streams' stream table."""
    _fields_ = [("file", C.c_uint32), ("channels", C.c_uint32), ("sample_rate", C.c_uint32), ("reserved", C.c_uint32),
                ("frames", C.c_uint64)]


class pov_file_report(C.Structure):
    """One file of pov_corpus_report: what the last corpus call found in it."""
    _fields_ = [("status", C.c_uint32), ("n_streams", C.c_uint32), ("frames", C.c_uint64), ("valid_frames", C.c_uint64),
                ("message", C.c_char * 192)]


class pov_device_pcm(C.Structure):
    """Output description of pov_decode_corpus_device: per stream-table record a planar region of the caller's device memory."""
    _fields_ = [("pcm_layout", C.c_uint32), ("n_streams", C.c_uint32), ("pcm_dev", C.c_void_p), ("capacity", C.c_uint64),
                ("stream_base", C.POINTER(C.c_uint64)), ("channel_stride", C.POINTER(C.c_uint64)),
                ("file", C.POINTER(C.c_uint32)), ("channels", C.POINTER(C.c_uint32)), ("frames", C.POINTER(C.c_uint64)),
                ("cuda_stream", C.c_void_p)]


class pov_resample(C.Structure):
    """Resampling / downmix of pov_decode_corpus_device_resampled."""
    _fields_ = [("out_rate", C.c_uint32), ("flags", C.c_uint32), ("sample_rate", C.POINTER(C.c_uint32))]


# numpy dtypes with the same layout as pov_stream / pov_packet (so big batches are built vectorised)
STREAM_DTYPE = np.dtype([("setup_id", "<u4"), ("first_packet", "<u4"), ("n_packets", "<u4"),
                         ("reserved", "<u4"), ("pcm_frames", "<u8"), ("pcm_base", "<u8")], align=True)
PACKET_DTYPE = np.dtype([("stream", "<u4"), ("mode", "u1"), ("window_flags", "u1"), ("floor_used", "<u2"),
                         ("emit_frames", "<u4"), ("packet_bytes", "<u4"), ("pcm_off", "<u8"), ("ys_off", "<u8"),
                         ("spec_off", "<u8")], align=True)
assert STREAM_DTYPE.itemsize == C.sizeof(pov_stream)
assert PACKET_DTYPE.itemsize == C.sizeof(pov_packet)


# ------------------------------------------------------------------------------------------------------------
# Python-side description of a setup, convertible to the C struct (keeps the backing arrays alive)
# ------------------------------------------------------------------------------------------------------------
@dataclass
class Codebook:
    dim: int
    n_entries: int
    lookup_type: int = 0
    vq: Optional[np.ndarray] = None  # float32 [n_entries*dim]


@dataclass
class Floor1:
    xs: Sequence[int]
    multiplier: int


@dataclass
class Residue:
    type: int
    begin: int
    end: int
    partition_size: int
    n_class: int
    classbook: int
    books: np.ndarray  # uint8 [n_class*8], 255 = none


@dataclass
class Mapping:
    mux: Sequence[int]
    submap_floor: Sequence[int]
    submap_residue: Sequence[int]
    couplings: Sequence[Sequence[int]] = ()  # (magnitude, angle)


@dataclass
class Mode:
    blockflag: int
    mapping: int


@dataclass
class Setup:
    channels: int
    sample_rate: int
    blocksize: Sequence[int]
    floors: List[Floor1]
    mappings: List[Mapping]
    modes: List[Mode]
    codebooks: List[Codebook] = field(default_factory=list)
    residues: List[Residue] = field(default_factory=list)

    def to_c(self) -> "CSetup":
        return CSetup(self)


class CSetup:
    """Owns the ctypes arrays behind one pov_setup."""

    def __init__(self, s: Setup):
        self.py = s
        self._keep = []
        cb = (pov_codebook * max(1, len(s.codebooks)))()
        for i, b in enumerate(s.codebooks):
            cb[i].dim, cb[i].n_entries, cb[i].lookup_type = b.dim, b.n_entries, b.lookup_type
            if b.vq is not None and b.lookup_type != 0:
                arr = np.ascontiguousarray(b.vq, dtype=np.float32)
                self._keep.append(arr)
                cb[i].vq = arr.ctypes.data_as(C.POINTER(C.c_float))
        fl = (pov_floor1 * max(1, len(s.floors)))()
        for i, f in enumerate(s.floors):
            fl[i].n_posts, fl[i].multiplier = len(f.xs), f.multiplier
            for j, x in enumerate(f.xs):
                fl[i].xs[j] = int(x)
        rs = (pov_residue * max(1, len(s.residues)))()
        for i, r in enumerate(s.residues):
            rs[i].type, rs[i].begin, rs[i].end = r.type, r.begin, r.end
            rs[i].partition_size, rs[i].n_class, rs[i].classbook = r.partition_size, r.n_class, r.classbook
            for j in range(POV_MAX_CLASSES * 8):
                rs[i].books[j] = POV_NO_BOOK
            for j, v in enumerate(np.asarray(r.books, dtype=np.uint8).ravel()):
                rs[i].books[j] = int(v)
        mp = (pov_mapping * max(1, len(s.mappings)))()
        for i, m in enumerate(s.mappings):
            mp[i].n_submaps, mp[i].n_couplings = len(m.submap_floor), len(m.couplings)
            for j, v in enumerate(m.mux):
                mp[i].mux[j] = int(v)
            for j, v in enumerate(m.submap_floor):
                mp[i].submap_floor[j] = int(v)
            for j, v in enumerate(m.submap_residue):
                mp[i].submap_residue[j] = int(v)
            for j, (mg, an) in enumerate(m.couplings):
                mp[i].coupling_mag[j], mp[i].coupling_ang[j] = int(mg), int(an)
        md = (pov_mode * max(1, len(s.modes)))()
        for i, m in enumerate(s.modes):
            md[i].blockflag, md[i].mapping = m.blockflag, m.mapping
        self._keep += [cb, fl, rs, mp, md]
        c = pov_setup()
        c.abi_version = POV_ABI_VERSION
        c.channels, c.sample_rate = s.channels, s.sample_rate
        c.blocksize[0], c.blocksize[1] = s.blocksize
        c.n_codebooks, c.codebooks = len(s.codebooks), cb
        c.n_floors, c.floors = len(s.floors), fl
        c.n_residues, c.residues = len(s.residues), rs
        c.n_mappings, c.mappings = len(s.mappings), mp
        c.n_modes, c.modes = len(s.modes), md
        self.c = c


@dataclass
class Batch:
    """A batch in numpy form. `packets`/`streams` are structured arrays with PACKET_DTYPE/STREAM_DTYPE."""
    streams: np.ndarray
    packets: np.ndarray
    ys: np.ndarray                    # uint16
    payload: np.ndarray               # float32 (dense) or uint8 (entries)
    pcm_floats: int
    input_kind: int = POV_INPUT_DENSE
    pcm_layout: int = POV_PCM_PLANAR

    def to_c(self) -> pov_batch:
        assert self.streams.dtype == STREAM_DTYPE and self.packets.dtype == PACKET_DTYPE
        self.streams = np.ascontiguousarray(self.streams)
        self.packets = np.ascontiguousarray(self.packets)
        self.ys = np.ascontiguousarray(self.ys, dtype=np.uint16)
        self.payload = np.ascontiguousarray(self.payload)
        b = pov_batch()
        b.input_kind, b.pcm_layout = self.input_kind, self.pcm_layout
        b.n_streams = len(self.streams)
        b.streams = C.cast(self.streams.ctypes.data, C.POINTER(pov_stream))
        b.n_packets = len(self.packets)
        b.packets = C.cast(self.packets.ctypes.data, C.POINTER(pov_packet))
        b.ys = C.cast(self.ys.ctypes.data, C.POINTER(C.c_uint16))
        b.n_ys = len(self.ys)
        b.payload = self.payload.ctypes.data
        b.payload_bytes = self.payload.nbytes
        b.pcm_floats = int(self.pcm_floats)
        return b
