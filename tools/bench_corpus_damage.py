"""Cut mode of the corpus decode (pov_ctx_set_cut_damage) against the strict decode, measured in one process, the modes
alternating round by round, on bench.py's `e2e` corpus (--corpus-files copies of the 44.1 kHz stereo fixture):

  f32:         pov_decode_corpus_device into one packed float32 tensor, strict and cut mode
  r16k_mono:   pov_decode_corpus_device_resampled, 16 kHz mono float32, strict and cut mode
  damaged_f32: the same corpus with 1 % of its files damaged (half truncated inside a page, half replaced by
               the fixture synth_bad_vq_book.ogg, which a status word flags), cut mode only (strict mode stops at the first
               of them). Its content-damaged streams are short and mono: the zeroing of a long multichannel tail is not timed.

Per round and mode: ms per step; within each strict / cut pair the order alternates between rounds. Then, in a separate
torch.profiler run (one step per mode), k_cut_damaged's device time per step and its launch count. The card's name and power limit are read in the same run. Prints one JSON line; --out also writes it.
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
from tools.bench_pcm_s16 import card  # noqa: E402


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
        raise SystemExit("bench_corpus_damage.py: no CUDA device")
    result = {"card": card(), "device": torch.cuda.get_device_name(0)}
    with open(CORPUS_FILE, "rb") as f:
        one = f.read()
    ctx = SynthContext(0)
    clean = [bytes(bytearray(one)) for _ in range(args.corpus_files)]
    with open(os.path.join(ROOT, "tests", "golden", "synth_bad_vq_book.ogg"), "rb") as f:
        content = f.read()                    # its first packet using a scalar book as VQ book gets a status word
    damaged = list(clean)
    every = 100
    for i in range(every // 2, len(damaged), every):
        damaged[i] = one[:int(len(one) * 0.7)] if (i // every) % 2 else content
    threads = args.corpus_threads or max(1, len(os.sched_getaffinity(0)) - 1)
    tables = {"clean": lib.corpus_streams(clean, host_threads=threads),
              "damaged": lib.corpus_streams(damaged, host_threads=threads, cut_damage=True)}
    MODES = {"strict_f32": ("clean", False, None), "cut_f32": ("clean", True, None),
             "strict_r16k_mono": ("clean", False, 16000), "cut_r16k_mono": ("clean", True, 16000),
             "cut_damaged_f32": ("damaged", True, None)}
    lay = {}
    for mode, (which, cut, rate) in MODES.items():
        table = tables[which]
        ofr = table.frames if rate is None else lib.resampled_frames(table, rate)
        och = np.ones(len(table), np.uint64) if rate else table.channels.astype(np.uint64)
        stride = (ofr + 3) // 4 * 4
        sizes = och * stride
        base = (np.cumsum(sizes) - sizes).astype(np.uint64)
        lay[mode] = (torch.empty(int(sizes.sum()), dtype=torch.float32, device="cuda"), base, stride)

    def decode(mode):
        which, cut, rate = MODES[mode]
        pcm, base, stride = lay[mode]
        ctx.set_cut_damage(cut)
        files = clean if which == "clean" else damaged
        if rate is None:
            return ctx.decode_corpus_into(files, pcm, tables[which], base, stride, host_threads=threads)[1]
        return ctx.decode_corpus_into(files, pcm, tables[which], base, stride, host_threads=threads, sample_rate=rate, mono=True)[1]

    for mode in list(MODES) * 2:              # warm-up: slot arenas, pinned pools, setups and filter tables at full size
        decode(mode)
    rep = ctx.corpus_report()
    result["damaged_files"] = len(rep.damaged)
    rows = {m: [] for m in MODES}
    for r in range(args.rounds):
        order = list(MODES)
        if r % 2:                             # every other round the cut run of each pair goes first
            order = ["cut_f32", "strict_f32", "cut_r16k_mono", "strict_r16k_mono", "cut_damaged_f32"]
        for mode in order:
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            for _ in range(args.corpus_steps):
                decode(mode)
            torch.cuda.synchronize()
            rows[mode].append((time.perf_counter() - t0) * 1e3 / args.corpus_steps)

    from torch.profiler import ProfilerActivity, profile
    kernels = {}
    for mode in MODES:
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            decode(mode)
            torch.cuda.synchronize()
        ev = [e for e in prof.key_averages() if "k_cut_damaged" in e.key]
        kernels[mode] = {"k_cut_damaged_ms_per_step": sum(e.device_time_total for e in ev) * 1e-3, "launches": sum(e.count for e in ev)}
    ctx.set_cut_damage(False)

    out = {}
    for m, v in rows.items():
        s = sorted(v)
        out[m] = {"median_ms_per_step": s[len(s) // 2], "min": s[0], "max": s[-1], "rounds_ms": v, **kernels[m]}
    result["corpus"] = {"files_per_step": args.corpus_files, "damaged_every": every, "steps_per_round": args.corpus_steps,
                        "host_threads": threads,
                        "timing": "host clock around the decode calls, synchronize on both sides; modes alternate by round; "
                                  "k_cut_damaged from a separate torch.profiler run of one step", **out}
    ctx.close()
    line = json.dumps(result)
    print(line)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
