#!/usr/bin/env python3
"""Benchmark of the B200-native Vorbis synthesis stage (BASELINE.json metric: decoded PCM samples/s).

    python bench.py --gpus N --steps K --warmup W            # our arm (CUDA path through the C ABI)
    python bench.py --impl reference --gpus N --steps K ...  # the reference's CPU decoder on the host cores
    python bench.py ... --dump-outputs DIR                    # also write the last timed step's outputs to DIR/*.npy

A *step* is one pass of the hot path (floor1 -> coupling -> floor multiply -> IMDCT -> window/overlap-add -> PCM,
one fused kernel) over one batch of synthetic config-2 input (BASELINE.json configs[1]: 44.1 kHz stereo, 4096
packets per stream, mixed 256/2048 blocks, one coupling step), replicated to --streams independent streams so
that one step reads and writes far more than the 126 MB L2.

`value`: inputs already resident in HBM, CUDA-event time on the library's stream, max over ranks.
`e2e`:   the metric through the reference-facing call with HOST buffers (BASELINE.json configs[4], the sharded corpus
         decode): Ogg/Vorbis files in host memory -> pov_decode_corpus (host front end, H2D of the packet data, entropy
         decode + synthesis kernels, D2H of the PCM into pinned host memory) -> PCM in host memory. This is the work the
         reference arm does (OggReader::full_read_from_memory on every file), on the same files, so the two are like for like.
`e2e_dense`: the config-2 step itself through pov_batch_upload/run/fetch_pcm with pinned host arenas (dense f32 spectra in,
         PCM out): bounded by PCIe, kept to explain the copy cost of the synthesis stage alone.
Multi-GPU: streams / files are independent, so every rank decodes its own shard; no collective on the data path.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

METRIC = "decoded PCM samples/sec (IMDCT+floor+OLA)"
UNIT = "samples/s"
BYTES_PER_SAMPLE = 8.0  # SURVEY.md §8(d): 2n B spectrum in + 2n B PCM out per channel-packet = 8 B per PCM sample


def measured_peak_gbs():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


class ClockSampler:
    """nvidia-smi clocks + throttle reasons sampled every 200 ms while the timed region runs."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.proc = None
        self.lines = []
        self.gpu = gpu_index
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(gpu_index), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "50"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._pump, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            parts = [x.strip() for x in ln.split(",")]
            if len(parts) < 9:
                continue
            try:
                sm.append(float(parts[1])); mx.append(float(parts[2]))
            except ValueError:
                continue
            for name, v in zip(names, parts[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "samples": len(sm), "reasons": sorted(reasons)}


def _cpulist(text):
    out = []
    for part in text.strip().split(","):
        if not part:
            continue
        a, _, b = part.partition("-")
        out += list(range(int(a), int(b or a) + 1))
    return out


def bind_to_gpu_numa(local, world):
    """Pin this rank (and every thread it starts: parser workers, CUDA's helper threads) to its share of the cores of the
    NUMA node its GPU hangs off, BEFORE any pinned allocation is made, so that staging buffers and PCM land in that node's
    memory (first touch) and the ranks do not time-slice each other's parser threads. Returns what was done."""
    import torch
    info = {"node": None, "cpus": None}
    try:
        def node_of(g):
            pr = torch.cuda.get_device_properties(g)
            pci = "%04x:%02x:%02x.0" % (pr.pci_domain_id, pr.pci_bus_id, pr.pci_device_id)
            with open("/sys/bus/pci/devices/%s/numa_node" % pci) as f:
                return int(f.read())
        nodes = [node_of(g) for g in range(world)]
        mine = nodes[local]
        allowed = sorted(os.sched_getaffinity(0))
        if mine >= 0:
            with open("/sys/devices/system/node/node%d/cpulist" % mine) as f:
                cpus = [c for c in _cpulist(f.read()) if c in allowed] or allowed
        else:
            cpus = allowed
        peers = [g for g in range(world) if nodes[g] == mine]
        k, n = peers.index(local), len(peers)
        share = cpus[k * len(cpus) // n:(k + 1) * len(cpus) // n] or cpus
        os.sched_setaffinity(0, share)
        info = {"node": mine, "cpus": len(share), "ranks_on_node": n}
    except Exception as e:      # no sysfs / no permission: run unpinned
        info["error"] = str(e)
    return info


def pinned_like(arr):
    import torch
    t = torch.empty(arr.shape, dtype=getattr(torch, str(arr.dtype)) if arr.dtype.names is None else torch.uint8,
                    pin_memory=True)
    out = t.numpy()
    out[...] = arr
    return t, out


def pin_batch(batch):
    """Move a batch's host arenas into pinned memory (returns the tensors that own the storage)."""
    import numpy as np
    import torch
    from parseoggvorbis_b200 import abi
    keep = []

    def pin_bytes(a):
        a = np.ascontiguousarray(a)
        t = torch.empty(a.nbytes, dtype=torch.uint8, pin_memory=True)
        v = t.numpy().view(a.dtype).reshape(a.shape)
        v[...] = a
        keep.append(t)
        return v

    pb = abi.Batch(pin_bytes(batch.streams), pin_bytes(batch.packets), pin_bytes(batch.ys), pin_bytes(batch.payload),
                   batch.pcm_floats, batch.input_kind, batch.pcm_layout)
    return pb, keep


def cpu_baseline_port(setup, batch, n_streams_sample):
    """Oracle port (oracle/synth_oracle.c) on the host cores, IMDCT = the reference's own mdct_backward when
    oracle/_ref is present. One sub-batch of whole streams per thread."""
    import numpy as np
    from parseoggvorbis_b200 import abi
    from tests import oracle_binding as ob
    cores = os.cpu_count() or 1
    S = min(n_streams_sample, len(batch.streams))
    threads = max(1, min(cores, S))
    kind = "reference" if ob.reference_lib() is not None else "fast"
    ob.lib().por_inverse_db_table()
    # split streams [0,S) into `threads` sub-batches (views of the same arenas)
    subs = []
    per = (S + threads - 1) // threads
    for t in range(threads):
        s0, s1 = t * per, min(S, (t + 1) * per)
        if s0 >= s1:
            break
        st = batch.streams[s0:s1].copy()
        p0 = int(st["first_packet"][0]); p1 = int(st["first_packet"][-1] + st["n_packets"][-1])
        pk = batch.packets[p0:p1].copy()
        pk["stream"] -= s0
        st["first_packet"] -= p0
        base = int(st["pcm_base"][0])
        st["pcm_base"] -= base
        st["setup_id"] = 0
        floats = int((st["pcm_frames"] * setup.channels).sum())
        subs.append(abi.Batch(st, pk, batch.ys, batch.payload, floats, batch.input_kind, batch.pcm_layout))
    reps = 6          # ~1 s of wall time = ~16 s of CPU work on 16 cores: long enough to time, short enough for the default run
    samples = reps * sum(int(s.pcm_floats) for s in subs)

    def work(b):
        for _ in range(reps):
            ob.synth_batch([setup], b, imdct=kind)
    t0 = time.perf_counter()
    ths = [threading.Thread(target=work, args=(b,)) for b in subs]
    for th in ths:
        th.start()
    for th in ths:
        th.join()
    dt = time.perf_counter() - t0
    return {"value": samples / dt, "unit": UNIT, "cores": len(subs), "kind": "port",
            "sample": "%d of the workload's streams x %d passes (%d PCM samples) through oracle/synth_oracle.c, one stream "
                      "group per thread, %s; %.2f s" % (S, reps, samples, "IMDCT = reference mdct_backward (oracle/_ref)"
                                                         if kind == "reference" else "IMDCT = oracle FFT", dt)}


CORPUS_FILE = os.path.join(ROOT, "tests", "golden", "test.stereo44khz.ogg")
DUMP_PCM_SAMPLES = 1 << 23        # 32 MB of float32 PCM values
DUMP_STATUS_SAMPLES = 1 << 20     # 8 MB of float64 status words: a dump stays under 40 MB at any --streams / --packets


def sample_positions(size, k):
    """The positions a dump samples out of an array of `size` values: all of them up to k, else k drawn with a fixed seed."""
    import numpy as np
    if size <= k:
        return np.arange(size)
    return np.sort(np.random.default_rng(0).choice(size, size=k, replace=False))


def dump_outputs(out_dir, pcm, status):
    """Write what one step of the device-resident leg hands its caller, for comparing two builds output for output:
    pcm.npy, the PCM arena (float32), and status.npy, the per-packet status words (float64, exact for uint32), each at
    sample_positions(len, DUMP_*_SAMPLES): the same positions for the same command line."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "pcm.npy"), pcm[sample_positions(pcm.size, DUMP_PCM_SAMPLES)].astype(np.float32))
    np.save(os.path.join(out_dir, "status.npy"), status[sample_positions(status.size, DUMP_STATUS_SAMPLES)].astype(np.float64))


def workload_config(args):
    """The `config` object: identical for both arms (it depends on the command line only)."""
    return {"workload": "value/roofline: config2, synthetic 44.1 kHz stereo, %d packets/stream, mixed 256/2048 blocks, 1 coupling "
                        "step, %d streams per GPU (%d distinct, seed=rank), spectra resident in HBM; e2e (and the reference arm): "
                        "config5, the bundled 44.1 kHz stereo fixture x %d files per GPU, bytes in host memory -> PCM in host memory" %
                        (args.packets, args.streams, min(args.distinct, args.streams), args.corpus_files),
            "corpus_files_per_gpu": args.corpus_files,
            "l2_policy": "inputs+outputs of a step (7 GB for config2, 7.5 GB for the corpus) far exceed the 126 MB L2; no flush needed",
            "parallelism": "independent streams / files sharded across ranks, no collective"}


def run_reference_arm(args):
    """The reference's own CPU decoder (oracle/_ref/ref_decode_bench around OggReader::full_read_from_memory,
    src/ParseOggVorbis.hpp:1428) on all host cores, on the corpus of the e2e leg. Rank 0 only."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    exe = os.path.join(ROOT, "oracle", "_ref", "ref_decode_bench")
    ogg = CORPUS_FILE
    cores = os.cpu_count() or 1
    if not os.path.exists(exe):
        print(json.dumps({"impl": "reference", "unavailable": "oracle/_ref/ref_decode_bench not built (make -C oracle ref)"}))
        return 0
    # one step = the per-GPU corpus of the e2e leg (a bounded sample of the N-GPU job: the files are identical)
    per_thread = max(1, (args.corpus_files + cores - 1) // cores) if args.ref_decodes <= 0 else args.ref_decodes
    times, samples = [], 0
    for i in range(args.warmup + args.steps):
        out = subprocess.check_output([exe, ogg, str(cores), str(per_thread)], text=True)
        r = json.loads(out.strip().splitlines()[-1])
        if i >= args.warmup:
            times.append(r["seconds"]); samples = r["samples"]
    total_t = sum(times)
    value = samples * len(times) / total_t
    sample = ("the corpus of the e2e leg: full reference decode (Ogg framing + Huffman + synthesis) of "
              "tests/audio/test.stereo44khz.ogg (44.1 kHz stereo, 256/2048 blocks, 182272 samples) x %d decodes on %d "
              "threads per step (one GPU's share of the job; at N GPUs the job is N such shares)" % (cores * per_thread, cores))
    line = {"impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": 1e3 * total_t / len(times), "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32", "data": "bundled fixture replicated",
            "config": workload_config(args),
            "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": "reference", "sample": sample},
            "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line))
    return 0


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--streams", type=int, default=128, help="independent config-2 streams per GPU per step")
    ap.add_argument("--packets", type=int, default=4096, help="packets per stream")
    ap.add_argument("--distinct", type=int, default=4, help="independently generated streams (rest are replicas)")
    ap.add_argument("--e2e-steps", type=int, default=6)
    ap.add_argument("--e2e-depth", type=int, default=2, help="contexts (= streams) the end-to-end steps are pipelined over")
    ap.add_argument("--cpu-streams", type=int, default=0, help="streams of the CPU-baseline sample (0 = one per core)")
    ap.add_argument("--ref-decodes", type=int, default=0, help="reference arm: decodes per thread per step (0 = corpus_files / cores)")
    ap.add_argument("--corpus-files", type=int, default=10000, help="files per GPU per step of the corpus (e2e) leg")
    ap.add_argument("--corpus-steps", type=int, default=3)
    ap.add_argument("--corpus-threads", type=int, default=0, help="front-end threads per rank (0 = cores / ranks - 1)")
    ap.add_argument("--no-e2e-dense", action="store_true")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the outputs of the last timed step to DIR/*.npy (rank 0)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.warmup < 3:
        args.warmup = 3
    if args.impl == "reference":
        return run_reference_arm(args)

    import numpy as np
    import torch
    from parseoggvorbis_b200 import workloads
    from parseoggvorbis_b200.lib import SynthContext

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device (the product has no CPU fallback)")
    torch.cuda.set_device(local)
    full_affinity = os.sched_getaffinity(0)
    numa = bind_to_gpu_numa(local, world)
    dist = None
    if world > 1:
        import torch.distributed as dist
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))

    # ---- workload: config 2, replicated; every rank decodes its own shard of independent streams (weak scaling) ----
    setup, batch = workloads.config2(P=args.packets, streams=args.streams, distinct=min(args.distinct, args.streams),
                                     seed=rank)
    samples_per_step = int(batch.pcm_floats)
    ctx = SynthContext(local)
    batch.streams["setup_id"] = ctx.register_setup(setup)
    stream = torch.cuda.ExternalStream(ctx.stream_ptr, device=torch.device("cuda", local))

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- device-resident leg ----
    bh = ctx.upload(batch)
    ctx.sync(bh)
    kernel_name = ctx.kernel_name(bh)
    for _ in range(args.warmup):
        ctx.run(bh)
    ctx.sync(bh)
    status_bad = int(np.count_nonzero(ctx.status(bh)))
    launches0 = ctx.launch_count
    sampler = ClockSampler(local) if rank == 0 else None
    barrier()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    with torch.cuda.stream(stream):
        ev0.record(stream)
        for _ in range(args.steps):
            ctx.run(bh)
        ev1.record(stream)
    barrier()
    ms = ev0.elapsed_time(ev1)
    launches = ctx.launch_count - launches0
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, ctx.fetch_pcm(bh), ctx.status(bh))
    clocks = None
    if sampler:
        # the timed region lasts tens of milliseconds, nvidia-smi samples every 50 ms: keep the same kernel running
        # back to back (untimed) for about a second so that the clock / throttle record is taken under this load
        t_end = time.perf_counter() + 1.0
        while time.perf_counter() < t_end:
            for _ in range(8):
                ctx.run(bh)
            ctx.sync(bh)
        clocks = sampler.stop()
        clocks["note"] = "sampled from warm-up through the timed region and 1 s of the same launches repeated untimed"
    launches_timed = launches
    from parseoggvorbis_b200 import sharding
    total_units, ms_max = sharding.aggregate_throughput(samples_per_step * args.steps, ms, dist, device="cuda")
    value = total_units / (ms_max * 1e-3)          # whole job: units of all ranks / slowest rank's device time
    kernel_ms = ms / args.steps          # this rank's fused-kernel launch duration (one launch per step)

    # correctness spot check of what was just timed (first stream vs the oracle) — outside the timed region
    check = None
    if rank == 0:
        from tests import oracle_binding as ob
        from parseoggvorbis_b200 import abi
        st = batch.streams[:1].copy(); st["setup_id"] = 0
        pk = batch.packets[:int(st["n_packets"][0])].copy()
        sub = abi.Batch(st, pk, batch.ys, batch.payload, int(st["pcm_frames"][0]) * setup.channels)
        ref, _ = ob.synth_batch([setup], sub, imdct="fast")
        got = ctx.fetch_pcm(bh)[:sub.pcm_floats]
        check = {"max_abs_err": float(np.abs(got - ref).max()), "peak": float(np.abs(ref).max()),
                 "snr_db": float(ob.snr_db(got, ref)),
                 "packets_with_status": status_bad}

    # ---- end-to-end leg (the headline): config 5, files in host memory -> PCM in host memory through pov_decode_corpus ----
    e2e = None
    if not args.no_e2e:
        with open(CORPUS_FILE, "rb") as f:
            one = f.read()
        files = [bytes(bytearray(one)) for _ in range(args.corpus_files)]       # distinct host copies (255 MB for 10 000)
        cores = len(os.sched_getaffinity(0))        # this rank's share (bind_to_gpu_numa)
        threads = args.corpus_threads or max(1, cores - 1)
        cctx = SynthContext(local)
        # the C call itself, with its argument arrays built once (a Python list of 10 000 bytes objects -> two ctypes arrays)
        import ctypes as C
        nfl = len(files)
        c_data = (C.c_char_p * nfl)(*files)
        c_len = (C.c_size_t * nfl)(*[len(f) for f in files])
        c_frames = np.zeros(nfl, np.uint64)
        c_total, c_chk = C.c_uint64(0), C.c_double(0)

        def decode_all():
            cctx._check(cctx.L.pov_decode_corpus(cctx.ctx, nfl, c_data, c_len, threads, c_frames.ctypes.data_as(C.POINTER(C.c_uint64)),
                                                 C.byref(c_total), C.byref(c_chk)))
            return c_frames, int(c_total.value), float(c_chk.value)
        for _ in range(2):                   # warm-up: tables, pinned pools and arenas settle at full size during the second call
            frames, total, chk = decode_all()
        b0 = cctx.io_bytes()
        barrier()
        t0 = time.perf_counter()
        vals = 0
        for _ in range(args.corpus_steps):
            frames, total, chk = decode_all()
            vals += total
        barrier()
        wall = time.perf_counter() - t0
        b1 = cctx.io_bytes()
        tt = torch.tensor([wall * 1e3], dtype=torch.float64, device="cuda")
        tv = torch.tensor([float(vals)], dtype=torch.float64, device="cuda")
        if dist is not None:
            dist.all_reduce(tt, op=dist.ReduceOp.MAX)
            dist.all_reduce(tv, op=dist.ReduceOp.SUM)
        expect = 182272 * args.corpus_files                         # 2 channels x 91136 frames per file
        e2e = {"value": float(tv.item()) / (float(tt.item()) * 1e-3), "unit": UNIT,
               "h2d_bytes_per_step": int((b1[0] - b0[0]) // args.corpus_steps), "d2h_bytes_per_step": int((b1[1] - b0[1]) // args.corpus_steps),
               "steps": args.corpus_steps, "ms_per_step": float(tt.item()) / args.corpus_steps,
               "files_per_step_per_gpu": args.corpus_files, "ogg_bytes_per_step_per_gpu": len(one) * args.corpus_files,
               "host_threads_per_rank": threads, "host_cores_of_rank": cores, "numa": numa,
               "per_rank_gb_per_s": {"h2d": (b1[0] - b0[0]) / wall / 1e9, "d2h": (b1[1] - b0[1]) / wall / 1e9},
               "pcm_values_per_step_ok": bool(total == expect), "checksum": chk,
               "timing": "host clock around pov_decode_corpus (parse + H2D + kernels + D2H into pinned host memory), barrier + "
                         "synchronize on both sides, max over ranks"}
        cctx.close()
        del files

    # ---- the config-2 step through the batch API with host buffers (dense spectra in, PCM out): PCIe-bound ----
    # Every step validates the descriptors, copies all input arenas from pinned host memory to the device, runs the
    # kernel and copies the whole PCM arena back into pinned host memory. Steps are issued as a pipeline over --e2e-depth
    # contexts (= CUDA streams), so that the H2D copy of step k+1 overlaps the D2H copy of step k on the two copy
    # engines — the way a corpus decode streams batches through the device. Timed with the host clock around the whole
    # pipeline (barrier + synchronize on both sides), which includes every copy and every launch.
    e2e_dense = None
    if not args.no_e2e and not args.no_e2e_dense:
        depth = max(1, args.e2e_depth)
        pb, keep = pin_batch(batch)
        ctxs = [ctx] + [SynthContext(local) for _ in range(depth - 1)]
        handles, outs = [bh], []
        for c in ctxs[1:]:
            sid2 = c.register_setup(setup)
            assert sid2 == int(batch.streams["setup_id"][0])
            handles.append(c.upload(pb))
        for _ in range(depth):
            t_out = torch.empty(int(batch.pcm_floats), dtype=torch.float32, pin_memory=True)
            keep.append(t_out)
            outs.append(t_out.numpy())
        h2d = int(pb.streams.nbytes + pb.packets.nbytes + pb.ys.nbytes + pb.payload.nbytes + 8 * len(pb.packets))
        d2h = int(outs[0].nbytes)

        def e2e_issue(k):
            c, h = ctxs[k % depth], handles[k % depth]
            c.sync(h)                               # the previous step on this context has delivered its PCM
            c.upload(pb, reuse=h)
            c.run(h)
            c.fetch_pcm(h, out=outs[k % depth], sync=False)

        def e2e_drain():
            for c, h in zip(ctxs, handles):
                c.sync(h)

        for k in range(depth):
            e2e_issue(k)
        e2e_drain()
        barrier()
        t0 = time.perf_counter()
        for k in range(args.e2e_steps):
            e2e_issue(k)
        e2e_drain()
        barrier()
        wall = time.perf_counter() - t0
        e2e_ok = all(bool(np.array_equal(outs[0][:1 << 20], o[:1 << 20])) for o in outs[1:min(depth, args.e2e_steps)])
        tt = torch.tensor([wall * 1e3], dtype=torch.float64, device="cuda")
        if dist is not None:
            dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        e2e_dense = {"value": world * samples_per_step * args.e2e_steps / (float(tt.item()) * 1e-3), "unit": UNIT,
               "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h, "steps": args.e2e_steps,
               "ms_per_step": float(tt.item()) / args.e2e_steps, "pipeline_depth": depth,
               "timing": "host clock around the pipelined steps (upload+run+fetch each), max over ranks",
               "outputs_identical_across_contexts": e2e_ok}
        for c, h in list(zip(ctxs, handles))[1:]:
            h.free()
            c.close()

    if rank == 0:
        peak, peak_src = measured_peak_gbs()
        achieved = samples_per_step * BYTES_PER_SAMPLE / (kernel_ms * 1e-3) / 1e9
        # DRAM traffic of one launch from the committed ncu --set full capture of this very workload (per launch, GB)
        traffic = None
        try:
            with open(os.path.join(ROOT, "profiles", "r02_traffic.json")) as f:
                tj = json.load(f)
            if tj["kernel"] == kernel_name and int(tj["samples_per_launch"]) == samples_per_step:
                traffic = tj["traffic_bytes_per_launch"] / 1e9
        except Exception:
            traffic = None
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms_max / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic",
            "config": workload_config(args), "samples_per_step_per_gpu": samples_per_step,
            "roofline": {"bound": "hbm", "kernel": kernel_name, "achieved": achieved, "peak": peak, "unit": "GB/s",
                         "frac": achieved / peak, "traffic": traffic,
                         "traffic_unit": "GB per launch (dram read+write of the committed ncu --set full capture of this workload, "
                                         "profiles/r02_traffic.json; not re-measured in this run)",
                         "peak_source": peak_src,
                         "algorithmic_bytes_per_launch": samples_per_step * BYTES_PER_SAMPLE,
                         "kernel_ms": kernel_ms},
            "gpu_launches": int(launches_timed), "clocks": clocks, "check": check,
        }
        if e2e:
            line["e2e"] = e2e
        if e2e_dense:
            line["e2e_dense"] = e2e_dense
        if world == 1 and not args.no_cpu_baseline:
            os.sched_setaffinity(0, full_affinity)          # the CPU baseline gets every core of the box
            line["cpu_baseline"] = cpu_baseline_port(setup, batch, args.cpu_streams or (os.cpu_count() or 1))
        print(json.dumps(line))
    bh.free()
    ctx.close()
    if dist is not None:
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
