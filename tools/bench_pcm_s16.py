"""float32 against signed 16-bit PCM output (POV_PCM_S16), measured in one process, the two formats alternating.

  corpus: bench.py's `e2e` workload — --corpus-files copies of the stereo fixture in host memory -> PCM in pinned host memory —
          through pov_decode_corpus and pov_decode_corpus_s16 (no sink): samples/s, ms per step, H2D / D2H bytes and GB/s per
          step, and one POV_CORPUS_TIMING=1 breakdown per format (untimed call).
  kernel: bench.py's `value` workload — config 2 x --streams streams, spectra resident in HBM — one k_warp_synth launch per
          step, CUDA events on the library's stream, float32 and s16 uploaded from the same batch. Algorithmic bytes: 4 B of
          spectrum in + 4 B (float32) or 2 B (int16) of PCM out per sample, against a device-to-device copy measured here.

Under torchrun (one rank per GPU, as bench.py) the corpus comparison runs on every rank at once and reports the job's rate.
Prints one JSON line; --out also writes it to a file.
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

from bench import CORPUS_FILE, bind_to_gpu_numa  # noqa: E402


def card():
    try:
        out = subprocess.check_output(["nvidia-smi", "--query-gpu=index,name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                                      text=True, timeout=30)
        return [l.strip() for l in out.strip().splitlines()]
    except Exception as e:
        return ["nvidia-smi unavailable: %s" % e]


def captured_stderr(fn):
    """Run fn() with file descriptor 2 redirected to a temporary file (the library's POV_CORPUS_TIMING report): its text."""
    sys.stderr.flush()
    saved = os.dup(2)
    with tempfile.TemporaryFile(mode="w+b") as tmp:
        os.dup2(tmp.fileno(), 2)
        try:
            fn()
        finally:
            os.dup2(saved, 2)
            os.close(saved)
        tmp.seek(0)
        return tmp.read().decode(errors="replace").strip()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=3, help="alternating (float32, s16) rounds of each measurement")
    ap.add_argument("--corpus-files", type=int, default=10000)
    ap.add_argument("--corpus-steps", type=int, default=3, help="pov_decode_corpus calls per timed round")
    ap.add_argument("--corpus-threads", type=int, default=0, help="front-end threads per rank (0 = cores - 1)")
    ap.add_argument("--streams", type=int, default=128)
    ap.add_argument("--packets", type=int, default=4096)
    ap.add_argument("--kernel-steps", type=int, default=20, help="launches per timed kernel round")
    ap.add_argument("--out")
    args = ap.parse_args()

    import numpy as np
    import torch
    from parseoggvorbis_b200 import abi, workloads
    from parseoggvorbis_b200.lib import SynthContext

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench_pcm_s16.py: no CUDA device")
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

    # ---- corpus decode ----
    with open(CORPUS_FILE, "rb") as f:
        one = f.read()
    files = [bytes(bytearray(one)) for _ in range(args.corpus_files)]
    threads = args.corpus_threads or max(1, len(os.sched_getaffinity(0)) - 1)
    cctx = SynthContext(local)
    n = len(files)
    c_data = (C.c_char_p * n)(*files)
    c_len = (C.c_size_t * n)(*[len(f) for f in files])
    c_frames = np.zeros(n, np.uint64)
    c_total, c_chk, c_sum = C.c_uint64(0), C.c_double(0), C.c_int64(0)
    no_sink = C.cast(None, C.CFUNCTYPE(C.c_int, C.c_uint32, C.c_uint32, C.c_uint64, C.POINTER(C.c_int16), C.c_void_p))
    fr = c_frames.ctypes.data_as(C.POINTER(C.c_uint64))

    def decode(fmt):
        if fmt == "f32":
            cctx._check(cctx.L.pov_decode_corpus(cctx.ctx, n, c_data, c_len, threads, fr, C.byref(c_total), C.byref(c_chk)))
        else:
            cctx._check(cctx.L.pov_decode_corpus_s16(cctx.ctx, n, c_data, c_len, threads, no_sink, None, fr, C.byref(c_total),
                                                     C.byref(c_sum)))
        return int(c_total.value)

    for fmt in ("f32", "s16", "f32", "s16"):          # warm-up: pinned pools and arenas at full size for both formats
        decode(fmt)
    corpus = {"f32": [], "s16": []}
    for _ in range(args.rounds):
        for fmt in ("f32", "s16"):
            b0 = cctx.io_bytes()
            barrier()
            t0 = time.perf_counter()
            vals = 0
            for _ in range(args.corpus_steps):
                vals += decode(fmt)
            barrier()
            wall = time.perf_counter() - t0
            b1 = cctx.io_bytes()
            tt = torch.tensor([wall], dtype=torch.float64, device="cuda")
            tv = torch.tensor([float(vals)], dtype=torch.float64, device="cuda")
            if dist is not None:
                dist.all_reduce(tt, op=dist.ReduceOp.MAX)
                dist.all_reduce(tv, op=dist.ReduceOp.SUM)
            h2d, d2h = (b1[0] - b0[0]) / args.corpus_steps, (b1[1] - b0[1]) / args.corpus_steps
            corpus[fmt].append({"samples_per_s": float(tv.item()) / float(tt.item()), "ms_per_step": float(tt.item()) * 1e3 / args.corpus_steps,
                                "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h),
                                "rank0_h2d_gb_per_s": h2d * args.corpus_steps / wall / 1e9, "rank0_d2h_gb_per_s": d2h * args.corpus_steps / wall / 1e9,
                                "pcm_values_per_step": int(c_total.value)})
    timing = {}
    os.environ["POV_CORPUS_TIMING"] = "1"
    for fmt in ("f32", "s16"):
        timing[fmt] = captured_stderr(lambda: decode(fmt))
    del os.environ["POV_CORPUS_TIMING"]
    cctx.close()
    del files

    def summary(rows):
        v = sorted(r["samples_per_s"] for r in rows)
        return {"median_samples_per_s": v[len(v) // 2], "min": v[0], "max": v[-1], "rounds": rows}
    result["corpus"] = {"files_per_step_per_gpu": args.corpus_files, "steps_per_round": args.corpus_steps, "host_threads_per_rank": threads,
                        "f32": summary(corpus["f32"]), "s16": summary(corpus["s16"]), "timing_breakdown": timing,
                        "timing": "host clock around pov_decode_corpus / pov_decode_corpus_s16 (no sink), barrier + synchronize on both "
                                  "sides, max over ranks"}
    result["corpus"]["s16_over_f32"] = result["corpus"]["s16"]["median_samples_per_s"] / result["corpus"]["f32"]["median_samples_per_s"]

    # ---- kernel only (rank 0's GPU; the other ranks wait) ----
    if rank == 0:
        setup, batch = workloads.config2(P=args.packets, streams=args.streams, distinct=min(4, args.streams), seed=0)
        samples = int(batch.pcm_floats)
        ctx = SynthContext(local)
        batch.streams["setup_id"] = ctx.register_setup(setup)
        stream = torch.cuda.ExternalStream(ctx.stream_ptr, device=torch.device("cuda", local))
        import dataclasses
        bh = {"f32": ctx.upload(batch), "s16": ctx.upload(dataclasses.replace(batch, pcm_layout=abi.POV_PCM_S16))}
        names = {k: ctx.kernel_name(h) for k, h in bh.items()}
        for _ in range(3):
            for h in bh.values():
                ctx.run(h)
        ctx.sync(bh["f32"])
        f32 = ctx.fetch_pcm(bh["f32"])
        s16 = ctx.fetch_pcm(bh["s16"])
        ref = np.where(np.isnan(f32), 0, np.clip(np.rint(f32.astype(np.float64) * 32768), -32768, 32767)).astype(np.int16)
        same = bool(np.array_equal(s16, ref))
        del f32, s16, ref
        # device-to-device copy peak of this card, measured here (read + write bytes of a 4 GiB copy)
        src = torch.empty(1 << 30, dtype=torch.float32, device="cuda")
        dst = torch.empty_like(src)
        for _ in range(3):
            dst.copy_(src)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(10):
            dst.copy_(src)
        e1.record()
        torch.cuda.synchronize()
        copy_gbs = 2 * src.numel() * 4 * 10 / (e0.elapsed_time(e1) * 1e-3) / 1e9
        del src, dst
        kern = {"f32": [], "s16": []}
        for _ in range(max(3, args.rounds)):
            for fmt in ("f32", "s16"):
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                with torch.cuda.stream(stream):
                    e0.record(stream)
                    for _ in range(args.kernel_steps):
                        ctx.run(bh[fmt])
                    e1.record(stream)
                torch.cuda.synchronize()
                kern[fmt].append(e0.elapsed_time(e1) / args.kernel_steps)
        out = {"workload": "config 2 x %d streams x %d packets, device-resident, %d PCM samples per launch" % (args.streams, args.packets, samples),
               "kernel_names": names, "s16_equals_rule_of_f32": same, "measured_d2d_copy_gb_per_s": copy_gbs}
        for fmt, bps in (("f32", 8.0), ("s16", 6.0)):
            ms = sorted(kern[fmt])
            med = ms[len(ms) // 2]
            out[fmt] = {"ms_per_launch_median": med, "ms_per_launch": kern[fmt], "samples_per_s": samples / (med * 1e-3),
                        "algorithmic_bytes_per_sample": bps, "algorithmic_gb_per_s": samples * bps / (med * 1e-3) / 1e9,
                        "fraction_of_measured_copy_peak": samples * bps / (med * 1e-3) / 1e9 / copy_gbs}
        out["s16_over_f32_time"] = out["s16"]["ms_per_launch_median"] / out["f32"]["ms_per_launch_median"]
        result["kernel"] = out
        for h in bh.values():
            h.free()
        ctx.close()
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
