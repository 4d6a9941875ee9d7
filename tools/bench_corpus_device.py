"""Corpus decode into host memory against corpus decode into caller-owned device memory, measured in one process, the modes
alternating round by round.

  host_f32: bench.py's `e2e` workload — --corpus-files distinct copies of the stereo fixture in host memory -> float32 PCM in
            pinned host memory — through pov_decode_corpus (no sink).
  dev_f32:  the same corpus through pov_decode_corpus_device into one packed float32 torch tensor on the GPU (each stream's
            channels `frames rounded up to 4` apart), allocated once; only compressed packets go host -> device and only status
            words come back.
  dev_s16:  the same with int16 samples (POV_PCM_S16).

Per round and mode: samples/s, ms per step, H2D / D2H bytes per step. The stream-table pass (pov_corpus_streams, host only) is
timed on its own: a caller that lays out its tensor from the table pays it once per corpus on top of the device decode. One
POV_CORPUS_TIMING=1 breakdown per mode (untimed call). The card's name, power limit and max SM clock are read in the same run.

Under torchrun (one rank per GPU, as bench.py) every rank decodes its own copy of the corpus at once and the job's rate is
sharding.aggregate_throughput (samples summed over ranks / the slowest rank's time). Prints one JSON line; --out also writes it.
"""
import argparse
import ctypes as C
import json
import os
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

from bench import CORPUS_FILE, bind_to_gpu_numa  # noqa: E402
from tools.bench_pcm_s16 import captured_stderr, card  # noqa: E402

MODES = ("host_f32", "dev_f32", "dev_s16")


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=3, help="alternating rounds of the three modes")
    ap.add_argument("--corpus-files", type=int, default=10000)
    ap.add_argument("--corpus-steps", type=int, default=3, help="decode calls per timed round")
    ap.add_argument("--corpus-threads", type=int, default=0, help="front-end threads per rank (0 = cores - 1)")
    ap.add_argument("--out")
    args = ap.parse_args()

    import numpy as np
    import torch
    from parseoggvorbis_b200 import lib, sharding
    from parseoggvorbis_b200.lib import SynthContext

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench_corpus_device.py: no CUDA device")
    torch.cuda.set_device(local)
    numa = bind_to_gpu_numa(local, world)
    dist = None
    if world > 1:
        import torch.distributed as dist
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    result = {"card": card() if rank == 0 else None, "device": torch.cuda.get_device_name(local), "world": world, "numa": numa}
    with open(CORPUS_FILE, "rb") as f:
        one = f.read()
    files = [bytes(bytearray(one)) for _ in range(args.corpus_files)]
    threads = args.corpus_threads or max(1, len(os.sched_getaffinity(0)) - 1)
    n = len(files)

    # stream table, timed on its own (host only)
    t0 = time.perf_counter()
    table = lib.corpus_streams(files, host_threads=threads)
    table_ms = [(time.perf_counter() - t0) * 1e3]
    for _ in range(2):
        t0 = time.perf_counter()
        lib.corpus_streams(files, host_threads=threads)
        table_ms.append((time.perf_counter() - t0) * 1e3)

    # one context per destination, so that neither keeps resizing the other's slot buffers
    hctx, dctx = SynthContext(local), SynthContext(local)
    c_data = (C.c_char_p * n)(*files)
    c_len = (C.c_size_t * n)(*[len(f) for f in files])
    c_frames = np.zeros(n, np.uint64)
    c_total, c_chk = C.c_uint64(0), C.c_double(0)
    fr = c_frames.ctypes.data_as(C.POINTER(C.c_uint64))
    stride = (table.frames + 3) // 4 * 4
    sizes = table.channels.astype(np.uint64) * stride
    base = (np.cumsum(sizes) - sizes).astype(np.uint64)
    pcm = {"dev_f32": torch.empty(int(sizes.sum()), dtype=torch.float32, device="cuda"),
           "dev_s16": torch.empty(int(sizes.sum()), dtype=torch.int16, device="cuda")}

    def decode(mode):
        if mode == "host_f32":
            hctx._check(hctx.L.pov_decode_corpus(hctx.ctx, n, c_data, c_len, threads, fr, C.byref(c_total), C.byref(c_chk)))
            return int(c_total.value)
        return dctx.decode_corpus_into(files, pcm[mode], table, base, stride, s16=mode == "dev_s16", host_threads=threads)[1]

    for mode in MODES + MODES:                # warm-up: pinned pools, slot buffers and setups at full size for every mode
        decode(mode)
    ref_total = decode("host_f32")
    same = {m: decode(m) == ref_total for m in MODES[1:]}
    rows = {m: [] for m in MODES}
    for _ in range(args.rounds):
        for mode in MODES:
            ctx = hctx if mode == "host_f32" else dctx
            b0 = ctx.io_bytes()
            barrier()
            t0 = time.perf_counter()
            vals = 0
            for _ in range(args.corpus_steps):
                vals += decode(mode)
            barrier()
            wall = time.perf_counter() - t0
            b1 = ctx.io_bytes()
            units, ms = sharding.aggregate_throughput(vals, wall * 1e3, dist, device=torch.device("cuda", local))
            rows[mode].append({"samples_per_s": units / (ms * 1e-3), "ms_per_step": ms / args.corpus_steps,
                               "h2d_bytes_per_step": (b1[0] - b0[0]) // args.corpus_steps,
                               "d2h_bytes_per_step": (b1[1] - b0[1]) // args.corpus_steps,
                               "pcm_values_per_step": vals // args.corpus_steps})
    timing = {}
    os.environ["POV_CORPUS_TIMING"] = "1"
    for mode in MODES:
        timing[mode] = captured_stderr(lambda: decode(mode))
    del os.environ["POV_CORPUS_TIMING"]

    def summary(r):
        v = sorted(x["samples_per_s"] for x in r)
        return {"median_samples_per_s": v[len(v) // 2], "min": v[0], "max": v[-1], "rounds": r}
    out = {m: summary(rows[m]) for m in MODES}
    result["corpus"] = {"files_per_step_per_gpu": n, "streams_per_step_per_gpu": len(table), "steps_per_round": args.corpus_steps,
                        "host_threads_per_rank": threads, "stream_table_ms_per_corpus": table_ms,
                        "total_values_equal_host_decode": same, "timing_breakdown": timing,
                        "timing": "host clock around the decode calls, barrier + synchronize on both sides; job rate = samples "
                                  "summed over ranks / max time over ranks (sharding.aggregate_throughput). The stream-table "
                                  "pass is not inside the timed window", **out}
    for m in MODES[1:]:
        result["corpus"][m + "_over_host_f32"] = out[m]["median_samples_per_s"] / out["host_f32"]["median_samples_per_s"]
    del pcm
    hctx.close()
    dctx.close()
    barrier()
    if rank == 0:
        line = json.dumps(result)
        print(line)
        if args.out:
            with open(args.out, "w") as f:
                f.write(line + "\n")
    if dist is not None:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
