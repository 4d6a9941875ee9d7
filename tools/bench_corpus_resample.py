"""Native device corpus decode against the resampled / downmixed one, measured in one process, the modes alternating round by
round, on bench.py's `e2e` corpus (--corpus-files copies of the 44.1 kHz stereo fixture):

  native_f32:    pov_decode_corpus_device into one packed float32 tensor (each stream's channels `frames rounded up to 4` apart)
  r16k_mono_f32: pov_decode_corpus_device_resampled, 16 kHz mono, float32, packed by output frames
  r16k_mono_s16: the same with int16 samples
  r48k_f32:      48 kHz, every channel, float32

Per round and mode: ms per step, decoded (native) samples/s, output samples and H2D / D2H bytes per step. Then, in a separate
torch.profiler run (one step per resampling mode), k_resample's kernel time, its bytes (arena samples read plus output samples
written, from shapes) and bytes/s as a share of the HBM data-sheet peak. The card's name and power limit are read in the same run.
Prints one JSON line; --out also writes it.
"""
import argparse
import json
import os
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

from bench import CORPUS_FILE  # noqa: E402
from tools.bench_pcm_s16 import captured_stderr, card  # noqa: E402

MODES = {"native_f32": (None, False, False), "r16k_mono_f32": (16000, True, False), "r16k_mono_s16": (16000, True, True),
         "r48k_f32": (48000, False, False)}
HBM_PEAK = 7.7e12          # bytes/s, NVIDIA's HGX B200 data sheet, one GPU


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--corpus-files", type=int, default=10000)
    ap.add_argument("--corpus-steps", type=int, default=3, help="decode calls per timed round")
    ap.add_argument("--corpus-threads", type=int, default=0, help="front-end threads (0 = cores - 1)")
    ap.add_argument("--out")
    args = ap.parse_args()

    import numpy as np
    import torch
    from parseoggvorbis_b200 import lib
    from parseoggvorbis_b200.lib import SynthContext

    if not torch.cuda.is_available():
        raise SystemExit("bench_corpus_resample.py: no CUDA device")
    result = {"card": card(), "device": torch.cuda.get_device_name(0)}
    with open(CORPUS_FILE, "rb") as f:
        one = f.read()
    files = [bytes(bytearray(one)) for _ in range(args.corpus_files)]
    threads = args.corpus_threads or max(1, len(os.sched_getaffinity(0)) - 1)
    table = lib.corpus_streams(files, host_threads=threads)
    native_values = int((table.channels.astype(np.uint64) * table.frames).sum())
    ctx = SynthContext(0)
    lay = {}
    for mode, (rate, mono, s16) in MODES.items():
        ofr = table.frames if rate is None else lib.resampled_frames(table, rate)
        och = np.ones(len(table), np.uint64) if mono else table.channels.astype(np.uint64)
        stride = (ofr + 3) // 4 * 4
        sizes = och * stride
        base = (np.cumsum(sizes) - sizes).astype(np.uint64)
        pcm = torch.empty(int(sizes.sum()), dtype=torch.int16 if s16 else torch.float32, device="cuda")
        lay[mode] = (pcm, base, stride, int((och * ofr).sum()))

    def decode(mode):
        rate, mono, s16 = MODES[mode]
        pcm, base, stride, _ = lay[mode]
        if rate is None:
            return ctx.decode_corpus_into(files, pcm, table, base, stride, host_threads=threads)[1]
        return ctx.decode_corpus_into(files, pcm, table, base, stride, s16=s16, host_threads=threads, sample_rate=rate, mono=mono)[1]

    for mode in list(MODES) * 2:              # warm-up: slot arenas, pinned pools, setups and filter tables at full size
        assert decode(mode) == lay[mode][3]
    rows = {m: [] for m in MODES}
    for _ in range(args.rounds):
        for mode in MODES:
            b0 = ctx.io_bytes()
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            vals = 0
            for _ in range(args.corpus_steps):
                vals += decode(mode)
            torch.cuda.synchronize()
            wall = time.perf_counter() - t0
            b1 = ctx.io_bytes()
            rows[mode].append({"ms_per_step": wall * 1e3 / args.corpus_steps,
                               "decoded_samples_per_s": native_values * args.corpus_steps / wall,
                               "output_samples_per_step": vals // args.corpus_steps,
                               "h2d_bytes_per_step": (b1[0] - b0[0]) // args.corpus_steps,
                               "d2h_bytes_per_step": (b1[1] - b0[1]) // args.corpus_steps})
    timing = {}
    os.environ["POV_CORPUS_TIMING"] = "1"
    for mode in MODES:
        timing[mode] = captured_stderr(lambda: decode(mode))
    del os.environ["POV_CORPUS_TIMING"]

    # k_resample in a profiler run of its own: kernel time summed over the step's launches
    from torch.profiler import ProfilerActivity, profile
    kernels = {}
    arena_bytes = 4 * int((table.channels.astype(np.uint64) * ((table.frames + 3) // 4 * 4)).sum())
    for mode in [m for m in MODES if MODES[m][0] is not None]:
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            decode(mode)
            torch.cuda.synchronize()
        us = sum(e.device_time_total for e in prof.key_averages() if "k_resample" in e.key)
        n = sum(e.count for e in prof.key_averages() if "k_resample" in e.key)
        out_bytes = lay[mode][3] * (2 if MODES[mode][2] else 4)
        nbytes = 4 * native_values + out_bytes          # every decoded sample read once (mono: each channel), output written once
        kernels[mode] = {"k_resample_launches": n, "k_resample_ms": us * 1e-3, "bytes": nbytes, "arena_bytes_allocated": arena_bytes,
                         "bytes_per_s": nbytes / (us * 1e-6) if us else None,
                         "share_of_hbm_peak": nbytes / (us * 1e-6) / HBM_PEAK if us else None}

    def summary(r):
        v = sorted(x["ms_per_step"] for x in r)
        return {"median_ms_per_step": v[len(v) // 2], "min": v[0], "max": v[-1], "rounds": r}
    out = {m: summary(rows[m]) for m in MODES}
    for m in MODES:
        if m != "native_f32":
            out[m]["ms_over_native"] = out[m]["median_ms_per_step"] / out["native_f32"]["median_ms_per_step"]
    result["corpus"] = {"files_per_step": len(files), "streams_per_step": len(table), "native_samples_per_step": native_values,
                        "steps_per_round": args.corpus_steps, "host_threads": threads, "timing_breakdown": timing,
                        "timing": "host clock around the decode calls, synchronize on both sides; modes alternate by round",
                        **out}
    result["k_resample"] = kernels
    result["k_resample_note"] = ("torch.profiler device time of every k_resample launch of one step; bytes from shapes: the "
                                 "decoded float32 samples read once plus the output written once; HBM peak %.1f TB/s (data sheet)"
                                 % (HBM_PEAK * 1e-12))
    ctx.close()
    line = json.dumps(result)
    print(line)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
