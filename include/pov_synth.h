/*
 * pov_synth.h — C ABI of the B200-native Vorbis *synthesis stage* (libpov_synth.so).
 *
 * What this boundary replaces in the reference (albertz/ParseOggVorbis, paths relative to its root):
 * the reference has no plugin seam around synthesis — the arithmetic is inlined in
 * VorbisStream::parse_audio (src/ParseOggVorbis.hpp:1128-1274). This header is the seam a maintainer would
 * cut there: everything in parse_audio that does NOT consume the bit reader moves behind these calls, batched
 * over many packets/streams:
 *
 *   floor1 curve synthesis       src/ParseOggVorbis.hpp:521-591, src/Utils.hpp:60-183, src/inverse_db_table.h:13-78
 *   residue VQ application       src/ParseOggVorbis.hpp:685-694, 734-752 (the adds; the Huffman walk stays on the host)
 *   nonzero propagate + coupling src/ParseOggVorbis.hpp:1174-1180, 1213-1241
 *   floor * residue              src/ParseOggVorbis.hpp:1243-1255
 *   inverse MDCT                 src/mdct.h:99-105 (extern "C" mdct_init/mdct_backward/mdct_clear), src/mdct.cpp:433-527
 *   window + overlap-add + emit  src/ParseOggVorbis.hpp:837-886, 1008-1059, 1061-1109
 *
 * Conventions mirror the reference's C API (src/ParseOggVorbis.hpp:1488-1494, src/ParseOggVorbis.cpp:12-41):
 * every call returns int, 0 = ok, non-zero = error; the message is available through pov_last_error() (a
 * per-context buffer instead of the reference's process-wide static one). Nothing throws, nothing aborts on
 * bad data. Only PODs, plain pointers and sizes cross the boundary. All pointers are HOST pointers unless a
 * name says `_dev`. One context per (host thread, GPU); contexts share no mutable state.
 *
 * There is no CPU fallback: every compute entry point fails with POV_ERR_CUDA if no sm_100 device is usable.
 */
#ifndef POV_SYNTH_H
#define POV_SYNTH_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define POV_ABI_VERSION      2u
#define POV_MAX_CHANNELS     8u    /* reference: uint8_t audio_channels (hpp:107); this build: <= 8 */
#define POV_MAX_POSTS        256u  /* floor1 syntax bound 2 + 31*8 = 250 (hpp:426,437) */
#define POV_MAX_COUPLINGS    256u  /* hpp:783 */
#define POV_MAX_SUBMAPS      16u   /* hpp:781 */
#define POV_MAX_CLASSES      64u   /* hpp:640 */
#define POV_MAX_MODES        64u   /* hpp:950 */
#define POV_NO_BOOK          255u  /* hpp:658 book_t(-1) */

/* ---- error codes (return values) ------------------------------------------------------------------------- */
enum {
	POV_OK            = 0,
	POV_ERR_ARG       = 1,  /* malformed descriptor / bad argument (host-side validation) */
	POV_ERR_CUDA      = 2,  /* CUDA runtime error or no usable device */
	POV_ERR_STREAM    = 3,  /* a reference CHECK(...) failed while parsing/decoding a stream */
	POV_ERR_UNSUPPORTED = 4 /* valid per the reference but outside this build's limits (e.g. > 8 channels) */
};

/* per-packet device status word (pov_batch_status): which of the reference's fatal per-packet CHECKs fired */
enum {
	POV_PKT_OK               = 0,
	POV_PKT_FLOOR_PREDICTED  = 1, /* hpp:536  CHECK(predicted <= range) */
	POV_PKT_FLOOR_RANGE      = 2, /* hpp:587  CHECK(floor[i] < 256) */
	POV_PKT_VQ_ENTRY         = 4  /* hpp:739,748 decodeVector: entry >= num_entries or lookup_type 0 */
};

/* ---- stream setup (the tables VorbisStreamSetup::parse produces, hpp:889-963) ---------------------------- */
typedef struct pov_codebook {
	uint32_t dim;          /* hpp:121 dimensions_ */
	uint32_t n_entries;    /* hpp:122 num_entries_ */
	uint32_t lookup_type;  /* hpp:142; 0 = scalar-only book, no VQ table */
	uint32_t reserved;
	const float* vq;       /* hpp:149 lookup_table_ [n_entries * dim]; NULL iff lookup_type == 0 */
	const uint8_t* lengths;/* hpp:126 Entry::len_ per entry, 0 = unused entry (hpp:270-272); only read for POV_INPUT_PACKETS
	                          batches (device-side entropy decode), may be NULL otherwise */
} pov_codebook;

/* How a floor1's coded Y list is laid out in the packet (hpp:425-447, read by hpp:498-517): needed only for
 * POV_INPUT_PACKETS batches, where the device walks the packet bits itself. */
typedef struct pov_floor1_syntax {
	uint8_t n_partitions;             /* hpp:426 (<= 31) */
	uint8_t n_classes;                /* hpp:429 maximum class + 1 (<= 16) */
	uint8_t reserved[2];
	uint8_t partition_class[32];      /* hpp:428 */
	uint8_t class_dim[16];            /* hpp:433, 1..8 */
	uint8_t class_subclass_bits[16];  /* hpp:434, 0..3 */
	uint8_t class_masterbook[16];     /* hpp:436 (only if subclass_bits > 0) */
	int16_t class_books[16][8];       /* hpp:441 subclass book number, -1 = none (the Y is 0) */
} pov_floor1_syntax;

typedef struct pov_floor1 {
	uint16_t n_posts;      /* == xs.size(), >= 2 */
	uint8_t  multiplier;   /* 1..4 (hpp:446) */
	uint8_t  reserved;
	uint16_t xs[POV_MAX_POSTS]; /* hpp:448-456, bitstream order; xs[0]=0, xs[1]=1<<rangebits; must be distinct */
} pov_floor1;

typedef struct pov_residue {
	uint32_t type;            /* 0,1,2 (hpp:633) */
	uint32_t begin, end;      /* hpp:636-637 */
	uint32_t partition_size;  /* hpp:639 */
	uint32_t n_class;         /* hpp:640 num_classifications */
	uint32_t classbook;       /* hpp:641 (host entropy decode only; ignored by the device) */
	uint8_t  books[POV_MAX_CLASSES * 8]; /* hpp:652-660 [class*8+pass], POV_NO_BOOK = none */
} pov_residue;

typedef struct pov_mapping {
	uint32_t n_submaps;       /* hpp:779-781 */
	uint32_t n_couplings;     /* hpp:783 */
	uint8_t  mux[POV_MAX_CHANNELS];          /* hpp:795-801 channel -> submap */
	uint8_t  submap_floor[POV_MAX_SUBMAPS];  /* hpp:806 */
	uint8_t  submap_residue[POV_MAX_SUBMAPS];/* hpp:808 */
	uint8_t  coupling_mag[POV_MAX_COUPLINGS];/* hpp:786 */
	uint8_t  coupling_ang[POV_MAX_COUPLINGS];/* hpp:787 */
} pov_mapping;

typedef struct pov_mode {
	uint8_t blockflag;        /* hpp:826: 1 = long window (blocksize1) */
	uint8_t mapping;          /* hpp:831 */
} pov_mode;

typedef struct pov_setup {
	uint32_t abi_version;     /* POV_ABI_VERSION */
	uint32_t channels;        /* hpp:107 */
	uint32_t sample_rate;     /* hpp:108 */
	uint32_t blocksize[2];    /* hpp:114-115; powers of two 64..8192, [0] <= [1] (hpp:1295-1298) */
	uint32_t n_codebooks;  const pov_codebook* codebooks;
	uint32_t n_floors;     const pov_floor1*   floors;
	uint32_t n_residues;   const pov_residue*  residues;
	uint32_t n_mappings;   const pov_mapping*  mappings;
	uint32_t n_modes;      const pov_mode*     modes;
	const pov_floor1_syntax* floor_syntax; /* [n_floors], or NULL (then POV_INPUT_PACKETS batches are refused for this setup) */
} pov_setup;

/* ---- batch description ----------------------------------------------------------------------------------- */
/* One logical stream inside a batch. Its packets are packets[first_packet .. first_packet+n_packets), in
 * decode order. A stream's first packet only primes the overlap (hpp:1021); to continue a stream across
 * batches re-submit the previous batch's last packet first with emit_frames = 0. */
typedef struct pov_stream {
	uint32_t setup_id;        /* from pov_setup_register */
	uint32_t first_packet;
	uint32_t n_packets;
	uint32_t reserved;
	uint64_t pcm_frames;      /* sum of emit_frames of its packets = frames this stream yields in this batch. Planar: this is
	                             also the channel stride, and it may exceed that sum (a padded layout); frames past the sum
	                             are not written. The kernels use no other property of it. */
	uint64_t pcm_base;        /* float index of channel 0 / frame 0 in the PCM arena. Planar: channel c, frame f
	                             lives at pcm_base + c*pcm_frames + f. Interleaved: pcm_base + f*channels + c. */
} pov_stream;

typedef struct pov_packet {
	uint32_t stream;          /* index into the batch's stream table */
	uint8_t  mode;            /* mode number (hpp:1146) -> blockflag + mapping */
	uint8_t  window_flags;    /* bit0 = prev_window_flag, bit1 = next_window_flag; long blocks only (hpp:1149-1153) */
	uint16_t floor_used;      /* bit c: channel c decoded a floor curve (hpp:478-482), BEFORE nonzero propagate */
	uint32_t emit_frames;     /* frames released by this packet: 0 for a stream's first packet, else
	                             prev/4 + cur/4 (hpp:1026), shortened at a page end by the granule rule (hpp:1028-1033) */
	uint32_t packet_bytes;    /* POV_INPUT_PACKETS: length of the raw audio packet; otherwise unused (0) */
	uint64_t pcm_off;         /* frame index inside the stream's PCM where this packet's chunk starts */
	uint64_t ys_off;          /* index (uint16 units) into the Y arena: for every channel WITH floor_used set, in
	                             channel order, that channel's coded Y list "floor1 ys" (hpp:498-518), n_posts each.
	                             POV_INPUT_PACKETS: ignored (floor_used and the Y lists are decoded on the device) */
	uint64_t spec_off;        /* POV_INPUT_DENSE:   float index into the spectra arena of this packet's
	                                                 "after_residue" vectors, [channels][blocksize/2] (hpp:1211)
	                             POV_INPUT_ENTRIES: byte offset into the residue payload arena (layout below)
	                             POV_INPUT_PACKETS: byte offset (multiple of 4) of the raw audio packet in the payload arena;
	                                                the bytes after it up to the next multiple of 4 must be zero */
} pov_packet;

/* Residue payload of ONE packet in POV_INPUT_ENTRIES mode (everything little-endian, 4-byte aligned):
 *   for each submap s of the packet's mapping, in order (hpp:1184):
 *       uint32 n_entries
 *       uint8  cls[nch_s][parts_s]       classification of every partition (hpp:719), padded to 4 bytes.
 *                                        nch_s = channels muxed to s (1 for residue type 2, hpp:689),
 *                                        parts_s = (min(end,L)-min(begin,L)) / partition_size, L = decode length
 *       uintE  entries[n_entries]        VQ entry numbers in DECODE ORDER (pass, partition, channel, vector:
 *                                        hpp:711-757), padded to 4 bytes. E = 16 bits if every codebook of the
 *                                        setup has <= 65536 entries, else 32 (pov_setup_entry_bits()).
 */
/* POV_INPUT_PACKETS: the payload arena holds the raw Vorbis audio packets (what hpp:1375-1381 hands to parse_audio).
 * mode, window_flags, emit_frames and pcm_off come from the host (they need the first bits of the packet and the page
 * granule only); the device reads everything else from the bits: floor flags and coded Ys (hpp:478-518), residue
 * classifications and VQ entry numbers (hpp:696-760) — the entropy decode of SURVEY.md §8(f)-2. Reading past the end of a
 * packet yields zero bits, as in the reference (Utils.hpp:389-392). The setup must carry codebook lengths and floor syntax. */
enum { POV_INPUT_DENSE = 0, POV_INPUT_ENTRIES = 1, POV_INPUT_PACKETS = 2 };
enum { POV_PCM_PLANAR = 0, POV_PCM_INTERLEAVED = 1 };
/* Flag OR-ed into pov_batch.pcm_layout (POV_PCM_PLANAR | POV_PCM_S16, POV_PCM_INTERLEAVED | POV_PCM_S16): the kernels store signed
 * 16-bit PCM instead of float32, converted at the store, so that half the bytes reach device memory and cross PCIe. Every float32
 * sample x the same batch would hold becomes
 *     s = clamp(round_half_even(x * 32768), -32768, 32767),   NaN -> 0
 * (x * 32768 is exact, so s depends on x alone). On finite samples this is libvorbisfile's ov_read on x86-64; NaN, which ov_read
 * turns into -32768, becomes 0 here (the device's saturating conversion). The intermediates of pov_batch_fetch_stage and
 * pov_batch_features stay float32. */
#define POV_PCM_S16 0x100u

typedef struct pov_batch {
	uint32_t input_kind;      /* POV_INPUT_DENSE | POV_INPUT_ENTRIES */
	uint32_t pcm_layout;      /* POV_PCM_PLANAR (matches gotPcmData, hpp:971) | POV_PCM_INTERLEAVED, optionally | POV_PCM_S16 */
	uint32_t n_streams;  const pov_stream* streams;
	uint32_t n_packets;  const pov_packet* packets;
	const uint16_t* ys;       uint64_t n_ys;        /* Y arena */
	const void*     payload;  uint64_t payload_bytes; /* dense spectra (float) or residue payload */
	uint64_t pcm_floats;      /* size of the PCM arena this batch writes, in samples: floats, or int16_t with POV_PCM_S16
	                             (pov_stream.pcm_base, pcm_frames and pov_packet.pcm_off count samples in both cases) */
} pov_batch;

/* debug stages, named after the reference's dump entries (hpp:518,560,561,585,1171,1211,1254,1265,1051) */
enum {
	POV_STAGE_FINAL_YS = 0,    /* uint32 [posts]      per used channel-packet     "floor1 final_ys"   */
	POV_STAGE_STEP2_FLAG = 1,  /* uint8  [posts]                                   "floor1 step2_flag" */
	POV_STAGE_FLOOR = 2,       /* uint32 [n]                                       "floor1 floor"      */
	POV_STAGE_FLOOR_OUTPUTS = 3,/* float [n]                                       "floor_outputs"     */
	POV_STAGE_AFTER_RESIDUE = 4,/* float [n/2]        per channel-packet           "after_residue"     */
	POV_STAGE_AFTER_ENVELOPE = 5,/* float [n/2]                                    "after_envelope"    */
	POV_STAGE_PCM_AFTER_MDCT = 6 /* float [n]                                      "pcm_after_mdct"    */
};

/* ---- context --------------------------------------------------------------------------------------------- */
typedef struct pov_ctx pov_ctx;

uint32_t    pov_abi_version(void);
/* Create a context on CUDA device `device`. Fails (POV_ERR_CUDA) when no sm_100 GPU is usable. */
int         pov_ctx_create(int device, pov_ctx** out, const char** error_out);
void        pov_ctx_destroy(pov_ctx* ctx);
const char* pov_last_error(const pov_ctx* ctx);
/* The CUDA stream (cudaStream_t as void*) all of this context's work is issued on. */
void*       pov_ctx_stream(pov_ctx* ctx);
/* Number of kernel launches issued by this context so far (for bench accounting). */
uint64_t    pov_ctx_launch_count(const pov_ctx* ctx);
/* Whole-file and corpus decode hand the audio packets to the device as they are (entropy decode in k_packet_decode) when
 * `on` is non-zero — the default; environment POV_DEVICE_ENTROPY=0 turns it off — and walk them on the host otherwise. */
void        pov_ctx_set_device_entropy(pov_ctx* ctx, int on);
/* Whole-file and corpus decode accept packets spanning pages when `on` is non-zero (default off = the reference's hpp:89;
 * environment POV_ALLOW_SPANNING=1 turns it on). */
void        pov_ctx_set_page_spanning(pov_ctx* ctx, int on);
/* Corpus decodes of this context cut damaged streams instead of failing when `on` is non-zero (default off: the first damaged
 * file fails the call). See "Cut mode" below; the whole-file and batch calls are not affected. */
void        pov_ctx_set_cut_damage(pov_ctx* ctx, int on);
/* Bytes this context has copied host -> device and device -> host so far (descriptor/payload arenas, PCM, status words). */
void        pov_ctx_io_bytes(const pov_ctx* ctx, uint64_t* h2d_out, uint64_t* d2h_out);

/* The 256-entry floor1_inverse_dB_table this library uses (reference: src/inverse_db_table.h:13-78). Host only. */
void        pov_inverse_db_table(float out[256]);
/* The window of a block (hpp:837-862: VorbisModeNumber::precalc / getWindow) as the kernels' slope tables define it:
 * n = blocksize[blockflag] floats. Host-only (no context, no device): the overlap-add stage multiplies by exactly
 * these values. Returns POV_ERR_ARG for block sizes outside 64..8192 / not powers of two / bs0 > bs1 / n mismatch. */
int         pov_window(uint32_t blocksize0, uint32_t blocksize1, int blockflag, int prev, int next, float* out, uint32_t n);

/* Validate + upload one stream setup; derived tables (neighbours, sort order, windows, twiddles) are built here. */
int         pov_setup_register(pov_ctx* ctx, const pov_setup* setup, uint32_t* setup_id_out);
int         pov_setup_entry_bits(const pov_ctx* ctx, uint32_t setup_id); /* 16 or 32; <0 on bad id */
/* Copy the window table the library generated for (setup, blockflag, prev, next) — hpp:837-886 — n floats. */
int         pov_setup_get_window(const pov_ctx* ctx, uint32_t setup_id, int blockflag, int prev, int next,
                                 float* out, uint32_t n);

/* ---- batches --------------------------------------------------------------------------------------------- */
typedef struct pov_batch_handle pov_batch_handle;

/* Validate a batch, build the device work lists and copy descriptors + arenas host->device (async on the
 * context stream; the host buffers must stay valid until pov_batch_sync or the next synchronising call). */
int  pov_batch_upload(pov_ctx* ctx, const pov_batch* batch, pov_batch_handle** out);
/* Launch the production path: [residue apply] -> fused floor1/coupling/dot/IMDCT/window/OLA -> PCM arena (device). */
int  pov_batch_run(pov_ctx* ctx, pov_batch_handle* h);
/* Name of the kernel pov_batch_run launches for this batch: "k_warp_synth" (persistent warp-autonomous kernel: block
 * sizes 256/512/1024/2048, <= 32 posts per floor), "k_fused_synth" (one CTA per run, any block sizes) or "staged".
 * Static string. */
const char* pov_batch_kernel_name(const pov_ctx* ctx, const pov_batch_handle* h);
/* Launch the staged path instead: one kernel per reference stage, every intermediate materialised in HBM so
 * that pov_batch_fetch_stage can return it. Produces the same PCM. */
int  pov_batch_run_staged(pov_ctx* ctx, pov_batch_handle* h);
/* Device->host copy of the PCM arena (pcm_floats floats; async unless `sync`). POV_ERR_ARG on a POV_PCM_S16 batch. */
int  pov_batch_fetch_pcm(pov_ctx* ctx, pov_batch_handle* h, float* out, uint64_t n_floats, int sync);
/* The same for a POV_PCM_S16 batch: n_values int16 samples (<= pcm_floats). POV_ERR_ARG on a float32 batch. */
int  pov_batch_fetch_pcm_s16(pov_ctx* ctx, pov_batch_handle* h, int16_t* out, uint64_t n_values, int sync);
/* Device pointer of the PCM arena (for callers that consume PCM on the GPU): float[pcm_floats], or int16_t[pcm_floats] for a
 * POV_PCM_S16 batch; after pov_batch_upload_into, the caller's pcm_dev. */
void* pov_batch_pcm_dev(pov_batch_handle* h);
/* pov_batch_upload with the PCM going to memory the caller owns: the kernels of every later run of the handle (pov_batch_run,
 * pov_batch_run_staged, the staged run pov_batch_features may start) write the PCM to `pcm_dev`, device memory of the context's
 * GPU holding batch->pcm_floats samples (float32, or int16 with POV_PCM_S16), aligned to a sample. The handle allocates no PCM
 * arena; pov_batch_pcm_dev returns pcm_dev and the fetch calls copy from it. The writes are issued on pov_ctx_stream(ctx): the
 * caller orders its own work against that stream. Only the PCM regions of the batch's streams are written (planar: channels x
 * emitted frames at pcm_base + c*pcm_frames), so padding between and after them keeps what the caller put there. A handle that
 * a plain pov_batch_upload reuses gets its own arena again. */
int  pov_batch_upload_into(pov_ctx* ctx, const pov_batch* batch, void* pcm_dev, pov_batch_handle** out);
/* One debug stage of one (packet, channel) after pov_batch_run_staged; `out_bytes` must match the stage size. */
int  pov_batch_fetch_stage(pov_ctx* ctx, pov_batch_handle* h, uint32_t packet, uint32_t channel, int stage,
                           void* out, uint64_t out_bytes);
/* Per-packet status words (POV_PKT_*), n_packets entries; synchronises. Returns POV_ERR_STREAM if any is non-zero. */
int  pov_batch_status(pov_ctx* ctx, pov_batch_handle* h, uint32_t* out_status, uint32_t n);
int  pov_batch_sync(pov_ctx* ctx, pov_batch_handle* h);
void pov_batch_free(pov_ctx* ctx, pov_batch_handle* h);

/* ---- drop-in for the reference's only C symbols on the path: mdct_backward (src/mdct.h:105) ---------------- */
/* `count` independent inverse MDCTs of size n (R^(n/2) -> R^n, no scaling), host buffers in/out. */
/* Parity hook of the production kernel: its own floor1 step-1 result (what hpp:521-559 computes), [n_packets][max channels][72]
 * bytes: 64 final Ys in ascending-x order, clamped to 255 | 64-bit step-2 mask in the same order. Warp-kernel batches only. */
int  pov_batch_fetch_fast_floor(pov_ctx* ctx, pov_batch_handle* h, uint8_t* out, uint64_t out_bytes);

/* Feature matrices straight from the device (the reference's downstream use: returnn_import.py:74-115 builds them in
 * Python from a debug dump, demo_live_extract.py:262-505): `kind` as below with the readers' default arguments, for one
 * stream of the batch; (rows, output_dim) floats, row-major, only the matrix crosses PCIe. Runs the staged kernels if they
 * have not run yet. out == NULL: only *rows_out is set (size query).
 *   FLOOR_FINAL_YS           get_features_from_raw_bytes(kind="floor_final_ys")            one row per decoded floor curve
 *   FLOOR_FINAL_YS_RENDERED  kind="floor_final_ys_rendered"
 *   RESIDUE_YS               kind="residue_ys"               rows of the packets whose (last channel's) floor has most posts
 *   RESIDUE_YS_WITH_FLOOR    kind="residue_ys_with_floor"    (exp() is the device's: within 1e-6 relative of numpy's) */
#define POV_ALL_STREAMS 0xFFFFFFFFu   /* `stream`: the rows of every stream of the batch, one after the other (one setup) */
enum { POV_FEAT_FLOOR_FINAL_YS = 0, POV_FEAT_FLOOR_FINAL_YS_RENDERED = 1, POV_FEAT_RESIDUE_YS = 2, POV_FEAT_RESIDUE_YS_WITH_FLOOR = 3 };
int  pov_batch_features(pov_ctx* ctx, pov_batch_handle* h, uint32_t stream, int kind, uint32_t output_dim,
                        float* out, uint64_t rows_cap, uint64_t* rows_out);

int  pov_mdct_backward_batch(pov_ctx* ctx, uint32_t n, uint64_t count, const float* in, float* out);

/* ---- whole-stream decode through the host front-end (mirrors ogg_vorbis_full_read_from_memory, hpp:1493) - */
typedef struct pov_decoded {
	uint32_t channels;
	uint32_t sample_rate;
	uint64_t frames;          /* frames per channel */
	uint32_t audio_packets;
	uint32_t reserved;
	float*   pcm;             /* planar [channels][frames]; owned by the library, free with pov_decoded_free */
} pov_decoded;

/* Decode one Ogg/Vorbis file held in memory. `debug_out` (may be NULL) names a file that receives the reference's
 * "ParseOggVorbis-header-v1" dump (src/Callbacks.cpp:146-185), produced from the staged device path. */
int  pov_ogg_vorbis_decode_memory(pov_ctx* ctx, const uint8_t* data, size_t len, const char* debug_out,
                                  pov_decoded* out);
void pov_decoded_free(pov_decoded* d);

/* The same decode with signed 16-bit output (the POV_PCM_S16 conversion, done by the kernels): `pcm` equals that rule applied to
 * what pov_ogg_vorbis_decode_memory returns. No debug dump: its format is float32. */
typedef struct pov_decoded_s16 {
	uint32_t channels;
	uint32_t sample_rate;
	uint64_t frames;          /* frames per channel */
	uint32_t audio_packets;
	uint32_t reserved;
	int16_t* pcm;             /* planar [channels][frames]; owned by the library, free with pov_decoded_s16_free */
} pov_decoded_s16;
int  pov_ogg_vorbis_decode_memory_s16(pov_ctx* ctx, const uint8_t* data, size_t len, pov_decoded_s16* out);
void pov_decoded_s16_free(pov_decoded_s16* d);

/* Decode a corpus of independent files with `host_threads` front-end threads (0 = all cores but one, which is left to
 * the calling thread) feeding this context's GPU. The context keeps the sibling stream, device arenas and pinned
 * staging buffers of the call for the next one; POV_CORPUS_TIMING=1 prints where the calling thread's time went.
 * Returns per-file frame counts (frames_out[n_files], may be NULL) and the total number of PCM values. */
int  pov_decode_corpus(pov_ctx* ctx, uint32_t n_files, const uint8_t* const* data, const size_t* len,
                       uint32_t host_threads, uint64_t* frames_out, uint64_t* total_values_out,
                       double* checksum_out);

/* The same decode with an output edge: `sink` receives the PCM of every logical stream, in file order, from the calling
 * thread, as the chunk that holds it retires — the batch form of ParseCallbacks::gotPcmData (hpp:966-973, 1047-1053).
 * `planar` is [channels][frames] (channel c at planar + c * frames) and is valid during the call only. A non-zero return
 * stops the decode, which then fails with POV_ERR_STREAM like the reference's CHECK(callbacks.gotPcmData(...)). */
typedef int (*pov_pcm_sink)(uint32_t file_index, uint32_t channels, uint64_t frames, const float* planar, void* user);
int  pov_decode_corpus_pcm(pov_ctx* ctx, uint32_t n_files, const uint8_t* const* data, const size_t* len,
                           uint32_t host_threads, pov_pcm_sink sink, void* user,
                           uint64_t* frames_out, uint64_t* total_values_out, double* checksum_out);

/* The corpus decode with signed 16-bit output (POV_PCM_S16 conversion on the device): half the device -> host bytes per sample.
 * `sink` (may be NULL: decode and count only) has the semantics of pov_decode_corpus_pcm's — file order, `planar` valid during
 * the call only, a non-zero return stops the decode with POV_ERR_STREAM. `sum_out` is the exact integer sum of every delivered
 * sample (independent of summation order, unlike the float64 checksum). */
typedef int (*pov_pcm_sink_s16)(uint32_t file_index, uint32_t channels, uint64_t frames, const int16_t* planar, void* user);
int  pov_decode_corpus_s16(pov_ctx* ctx, uint32_t n_files, const uint8_t* const* data, const size_t* len,
                           uint32_t host_threads, pov_pcm_sink_s16 sink, void* user,
                           uint64_t* frames_out, uint64_t* total_values_out, int64_t* sum_out);

/* Host-only (no GPU needed): one record per logical stream the corpus decode decodes — every Vorbis stream of every file that
 * reaches a complete setup, in file order and, inside a file, in the order the corpus decode delivers them (a chained file has
 * several). It runs the corpus decode's own parse (raw-packet mode, `host_threads` threads, 0 = all cores but one) and discards
 * the packets, so `frames` is what the decode produces. flags: POV_PARSE_ALLOW_SPANNING (see pov_ogg_parse_memory_ex; the
 * corpus decode follows pov_ctx_set_page_spanning) and POV_PARSE_CUT_DAMAGE (cut mode, below; the corpus decode follows
 * pov_ctx_set_cut_damage). Without it a framing or header error fails with POV_ERR_STREAM and the text pov_decode_corpus
 * gives for it ("file k: check failed: ..."), in *error_out (per-thread buffer). On success *out holds
 * *n_streams_out records (NULL when there are none), allocated by the library: free with pov_corpus_streams_free.
 * Callers use it to size and lay out the output of pov_decode_corpus_device, or to bucket files by length. */
typedef struct pov_stream_info {
	uint32_t file;            /* index into the corpus */
	uint32_t channels;
	uint32_t sample_rate;
	uint32_t reserved;
	uint64_t frames;          /* frames per channel the decode yields for this stream */
} pov_stream_info;
int  pov_corpus_streams(uint32_t n_files, const uint8_t* const* data, const size_t* len, uint32_t flags, uint32_t host_threads,
                        pov_stream_info** out, uint64_t* n_streams_out, const char** error_out);
void pov_corpus_streams_free(pov_stream_info* p);

/* Where pov_decode_corpus_device writes: one planar region per record of the stream table (pov_corpus_streams), in device
 * memory the caller owns on the context's GPU (a torch tensor, for example). Stream i, channel c, frame f lands at sample index
 * stream_base[i] + c * channel_stride[i] + f of pcm_dev. Strides and bases that are multiples of 4 keep the kernels on their
 * vector stores; any values work. */
typedef struct pov_device_pcm {
	uint32_t pcm_layout;              /* POV_PCM_PLANAR, optionally | POV_PCM_S16 (int16 samples); interleaved is refused */
	uint32_t n_streams;               /* records of the stream table */
	void*    pcm_dev;                 /* float32 or int16 samples on the context's device, aligned to a sample */
	uint64_t capacity;                /* samples at pcm_dev */
	const uint64_t* stream_base;      /* [n_streams] sample index of channel 0, frame 0 */
	const uint64_t* channel_stride;   /* [n_streams] samples between channels, >= frames */
	const uint32_t* file;             /* [n_streams] from the table: checked against what is parsed */
	const uint32_t* channels;         /* [n_streams] from the table: checked against what is parsed */
	const uint64_t* frames;           /* [n_streams] from the table: checked against what is parsed */
	void*    cuda_stream;             /* the caller's cudaStream_t, or NULL (legacy default stream): no PCM write starts before
	                                     the work queued on it when the call is made */
} pov_device_pcm;
/* The corpus decode with the PCM landing in the caller's device memory: only compressed packets go host -> device and only the
 * per-packet status words come back (pov_ctx_io_bytes counts 4 bytes per audio packet device -> host). Same workers, chunks
 * and errors as pov_decode_corpus_pcm.
 * - Before anything is launched the regions are validated: layout, null pointers, channels > 0, stride >= frames,
 *   base + channels * stride <= capacity, no two regions [base, base + channels * stride) overlapping. POV_ERR_ARG otherwise.
 * - Every parsed stream is compared with the record at its index (file, channels, frames) before its chunk is uploaded; a
 *   mismatch, more streams than n_streams, or fewer at the end, is POV_ERR_ARG naming the file. Chunks uploaded before that
 *   point have written their streams.
 * - The library writes exactly [base + c * stride, base + c * stride + frames) for c < channels of every stream: padding keeps
 *   whatever the caller put there.
 * - The call returns after every chunk has finished on the device, so on success the PCM is complete and visible to any stream.
 * frames_out[n_files] (may be NULL) and *total_values_out are as in pov_decode_corpus. */
int  pov_decode_corpus_device(pov_ctx* ctx, uint32_t n_files, const uint8_t* const* data, const size_t* len, uint32_t host_threads,
                              const pov_device_pcm* out, uint64_t* frames_out, uint64_t* total_values_out);

/* Resampling and mono downmix of the device corpus decode (pov_decode_corpus_device_resampled).
 * A stream at rate `in` resampled to rate `out`: g = gcd(in, out), L = out / g (up), M = in / g (down).
 * - L = M = 1: the output is a copy of the decoded samples (no filter).
 * - Otherwise R = max(L, M), hl = 10 R (half_len), N = 2 hl + 1 taps, the design of scipy.signal.resample_poly's default:
 *   h[n] = fc sinc(fc (n - hl)) I0(5 sqrt(1 - ((n - hl) / hl)^2)) / I0(5) with fc = 1 / R, normalised to unit sum, times L;
 *   computed in float64 on the host and rounded once to float32.
 * - Output frames: ceil(frames L / M). Output sample y[j] = sum_i x[i] h[j M + hl - i L] over taps inside [0, N) and inputs inside
 *   [0, frames), zero outside: scipy.signal.resample_poly(x, out, in) with padtype='constant'. The kernel evaluates it in
 *   polyphase form, phase (j M + hl) mod L with inputs x[floor((j M + hl) / L) - k] and taps h[phase + k L], k ascending from 0,
 *   one fmaf each, from 0.0f; the result does not depend on chunks, tiles or layouts.
 * - POV_RESAMPLE_MONO: the channels are averaged first, s = x0; s = s + x1 (rounded); ...; m = s * (1.0f / C) (rounded), then
 *   resampled as one channel. Without it every channel is resampled on its own.
 * - int16 output (POV_PCM_S16) is the POV_PCM_S16 rule applied to the float32 y at the store; the filter can overshoot full
 *   scale, and such samples saturate.
 * - Supported: max(L, M) <= POV_RESAMPLE_MAX_PHASES (tables of up to 40961 taps). Larger ratios (2048 -> 2049 Hz, 44056 -> 48000
 *   Hz) are POV_ERR_UNSUPPORTED. */
#define POV_RESAMPLE_MONO 1u
#define POV_RESAMPLE_MAX_PHASES 2048u
typedef struct pov_resample {
	uint32_t out_rate;              /* Hz; 0 = each stream keeps its rate (L = M = 1: downmix only, or a plain copy) */
	uint32_t flags;                 /* POV_RESAMPLE_MONO */
	const uint32_t* sample_rate;    /* [n_streams] from the stream table: checked against what is parsed, like channels / frames */
} pov_resample;

/* Host only (no GPU): the reduced ratio (*up = L, *down = M), *half_len = hl and, when `taps` is not NULL, the N = 2 hl + 1
 * float32 taps h[0..N) of the in_rate -> out_rate filter above. L = M = 1 (out_rate 0 or equal to in_rate) is a copy:
 * *half_len = 0 and no taps are written. taps_cap < N with taps != NULL, or in_rate = 0, is POV_ERR_ARG; max(L, M) past
 * POV_RESAMPLE_MAX_PHASES is POV_ERR_UNSUPPORTED (the ratio is still reported). */
int  pov_resample_filter(uint32_t in_rate, uint32_t out_rate, uint32_t* up, uint32_t* down, uint32_t* half_len,
                         float* taps, uint32_t taps_cap);

/* pov_decode_corpus_device with every stream downmixed (POV_RESAMPLE_MONO) and/or resampled to rs->out_rate on the device, as
 * defined above, before it lands in the caller's memory (float32, or int16 with POV_PCM_S16). The synthesis writes each chunk
 * into a float32 device arena of the context (every channel 4-aligned, so the decoded samples equal what
 * pov_decode_corpus_device writes into 4-aligned regions), and one resample kernel per chunk reads it and writes the regions.
 * - out->file, channels and frames are the native stream table, checked against what is parsed as in pov_decode_corpus_device;
 *   rs->sample_rate is checked the same way (a mismatch is POV_ERR_ARG naming the file).
 * - Stream i owns out_channels x channel_stride[i] samples from stream_base[i], out_channels = 1 with POV_RESAMPLE_MONO and
 *   channels[i] otherwise; channel_stride[i] must be at least its output frames. Exactly
 *   [base + c * stride, base + c * stride + output frames) is written for c < out_channels.
 * - Before anything is launched: the checks of pov_decode_corpus_device on these output regions, a null `rs`, a null
 *   rs->sample_rate with n_streams > 0, unknown flags (POV_ERR_ARG), and a ratio past POV_RESAMPLE_MAX_PHASES for any record
 *   (POV_ERR_UNSUPPORTED naming the stream, both rates and the phase count).
 * - frames_out[n_files] (may be NULL) are the native frames per file; *total_values_out counts the samples written.
 * Device memory: besides the caller's regions, up to four float32 chunk arenas stay allocated on the context (about 190 MB
 * each for chunks of 256 stereo files of 2 s at 44.1 kHz) and a filter table per ratio used (at most 160 KB each). */
int  pov_decode_corpus_device_resampled(pov_ctx* ctx, uint32_t n_files, const uint8_t* const* data, const size_t* len,
                                        uint32_t host_threads, const pov_device_pcm* out, const pov_resample* rs,
                                        uint64_t* frames_out, uint64_t* total_values_out);

/* Cut mode (pov_ctx_set_cut_damage, POV_PARSE_CUT_DAMAGE): every corpus call — pov_decode_corpus, _pcm, _s16, _device,
 * _device_resampled — and pov_corpus_streams go on past damaged files; each damaged stream ends where its damage starts.
 * Damage is found at two levels, and the level decides whether a stream's frame count changes.
 * 1. Geometry damage: a failing check of the raw-packet parse that pov_corpus_streams runs — Ogg framing (capture pattern,
 *    truncated segment table or body, CRC), stream bookkeeping (unknown serial, duplicate begin-of-stream, the continuation
 *    flag), the three headers, an audio packet's type bit, mode number and window flags, and the granule checks. The parse of
 *    the file stops there: every stream keeps the audio packets completed before the failure; the failing packet, the rest of
 *    its page and all later pages are dropped; a stream without a complete setup has no record. Its `frames` shrink, in the
 *    stream table and in the decode alike (they run the same parse).
 * 2. Content damage: a non-zero status word (POV_PKT_*) of a stream's packet, or with the host walk (POV_DEVICE_ENTROPY=0, or
 *    a setup the device walk cannot take) a failing walk of its floors and residues. The stream keeps its frames. With p its
 *    first damaged packet, its valid frames are pcm_off[p], and samples [pcm_off[p], frames) of every channel are exact zeros.
 *    A packet whose host walk fails enters the batch as silence (no floor used, residues that decode nothing), so the geometry
 *    stays; every later packet of that stream is silence too, which does not matter because everything after the cut is zero.
 * Consequences:
 * - Before the cut the samples are bit-identical to a strict decode, with the same alignment, of the undamaged file (content
 *   damage) or of the file truncated before the damaged page (geometry damage): packets < p are unchanged, and equal frames
 *   give equal PCM.
 * - Output regions keep their rule: exactly [base + c * stride, base + c * stride + frames) is written, padding is untouched.
 * - Resampled output is the resample of the zero-tailed stream; int16 output is the POV_PCM_S16 rule applied to it (0 in the
 *   tail). The float64 checksum, the int16 sum and the sinks see the zero-tailed PCM. frames_out stays the frames written.
 * - The stream table and the decode must use the same mode (as with page spanning): otherwise the records do not match what is
 *   parsed and the decode fails with POV_ERR_ARG as for any mismatch.
 * - Out of memory, CUDA failures, a stream-table mismatch and a sink asking to stop still fail the call in both modes.
 * Not done: resynchronising after damage (scanning for the next capture pattern and decoding on past a hole), concealing one
 * bad packet and decoding on, and cut mode for pov_ogg_vorbis_decode_memory* and the batch calls. Strict-mode texts are as before.
 *
 * What the last successful corpus call of the context found, per file (pov_corpus_report), in both modes: */
typedef struct pov_file_report {
	uint32_t status;          /* POV_OK, or POV_ERR_STREAM: damaged, cut as above */
	uint32_t n_streams;       /* its records in the stream table */
	uint64_t frames;          /* = frames_out[file] */
	uint64_t valid_frames;    /* summed over its streams: frames before each stream's cut */
	char     message[192];    /* "" or the reason: for geometry damage exactly the strict decode's and pov_corpus_streams'
	                             "file k: check failed: ..." text; otherwise "file k: stream s: check failed: audio packet p: <reason>"
	                             with s the stream's index among the file's records, p its packet index and the status word's
	                             reason. A file with both kinds reports its geometry damage. */
} pov_file_report;
/* Copies the report of the context's last corpus call when that call succeeded: files[n_files] and, when stream_valid_frames
 * is not NULL, the valid frames of every record of its stream table, stream_valid_frames[n_streams] (n_streams is the sum of
 * the files' n_streams). POV_ERR_ARG when the last corpus call failed in any way (argument checks included) or there was
 * none, and when n_files, or with the array n_streams, is not that call's. */
int  pov_corpus_report(const pov_ctx* ctx, uint32_t n_files, pov_file_report* files, uint64_t n_streams, uint64_t* stream_valid_frames);

/* Host-only front-end (no GPU needed): parse a whole Ogg/Vorbis file into descriptor batches, one per logical stream
 * (Ogg framing hpp:51-102,1433-1484; headers hpp:1283-1373; per-packet entropy decode hpp:498-517, 711-757). The
 * setup/batch returned by pov_parsed_get point into memory owned by the handle (POV_INPUT_ENTRIES, setup_id 0). */
typedef struct pov_parsed pov_parsed;
int      pov_ogg_parse_memory(const uint8_t* data, size_t len, pov_parsed** out, const char** error_out);
/* flags: POV_PARSE_RAW_PACKETS — do not entropy-decode the audio packets; the batches are POV_INPUT_PACKETS (a stream whose
 * setup cannot be walked on the device — floor0, a submap without channels — still comes back as POV_INPUT_ENTRIES). */
#define POV_PARSE_RAW_PACKETS 1u
/*        POV_PARSE_ALLOW_SPANNING — accept packets that continue on the next page of their stream (RFC 3533). The reference
 * refuses such files (hpp:89: "we don't support packets spanning pages"), which stays the default for parity. */
#define POV_PARSE_ALLOW_SPANNING 2u
/*        POV_PARSE_CUT_DAMAGE — cut mode (above): geometry damage ends the parse with success and the packets before it; with
 * the host walk a packet whose walk fails is kept as silence. Also a flag of pov_corpus_streams, whose records then shrink. */
#define POV_PARSE_CUT_DAMAGE 4u
int      pov_ogg_parse_memory_ex(const uint8_t* data, size_t len, uint32_t flags, pov_parsed** out, const char** error_out);
uint32_t pov_parsed_stream_count(const pov_parsed* p);
int      pov_parsed_get(const pov_parsed* p, uint32_t stream, pov_setup* setup_out, pov_batch* batch_out);
void     pov_parsed_free(pov_parsed* p);

/* Same signature/semantics as the reference's entry point (hpp:1493), on device 0; error string is per-thread. */
int  pov_ogg_vorbis_full_read_from_memory(const char* data, size_t data_len, const char** error_out);

#ifdef __cplusplus
}
#endif
#endif /* POV_SYNTH_H */
