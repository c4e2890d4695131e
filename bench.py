#!/usr/bin/env python3
"""bench.py — BASELINE.json metric: 352x192 MPEG-1 frames/sec/GPU (decoded YUV bit-exact vs reference).

Workload (BASELINE.json configs[3], SURVEY.md 8d "Config 4"): 4,096 independent synthetic streams
per GPU, each one GOP of 12 pictures (1 I + 11 P, 12 slices/picture, ~7.4 KB/picture), D=64 distinct
seeds replicated 64x (replication only bounds generation time; parity of the distinct streams is
checked in tests/). A step = one pass of the hot path over the batch: K0 index + K1a (one parse launch over
all 589,824 slices) + 12 launches of K1b (reconstruction, one per picture index) = 49,152 decoded pictures per GPU.

  value   whole-job frames/s with the elementary streams already resident in HBM (CUDA events, max over ranks)
  e2e     same metric through the C-ABI with HOST buffers: pinned ES -> H2D -> index -> decode -> D2H of the
          LAST picture of every stream (1/12 of what was decoded), all inside the timed region
  e2e_all the same with EVERY decoded picture copied back (ef_decode_all_to_host = the reference's push_video
          hand-over of every picture): 12x the read-back, PCIe bound
  roofline  K1 (= K1a + K1b): algorithmic bytes (ES + frame written + reference frame read, SURVEY.md 8d) / time of the pair
  cpu_baseline / --impl reference   the UNMODIFIED reference decoder (oracle/_ref/efref_decode, one process per
          core, Q11) on the box's host cores; falls back to the C restatement (kind "port") if _ref is absent
Multi-GPU: independent streams shard one batch per rank, no data-path collective; one all_gather of per-rank
frame counts for the report (SURVEY.md 8e). Default = weak scaling (4,096 streams per GPU, the driver's SCALE run);
--scaling strong = BASELINE config 5 as written: 32,768 streams in total, split over the ranks.
Every rank pins itself (and with it its pinned host buffers) to the NUMA node of its GPU before allocating.
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

METRIC = "352x192 MPEG-1 frames/sec (decoded YUV bit-exact vs reference)"
UNIT = "frames/s"
STREAMS_PER_GPU = 4096
DISTINCT = 64
PICTURES = 12
FRAME_BYTES = 101376


def env_int(name, default):
    try:
        return int(os.environ.get(name, default))
    except ValueError:
        return default


def workload_config(n_gpus, streams, scaling="weak"):
    name = "config4" if scaling == "weak" else "config5 (strong scaling: %d streams in total)" % (streams * n_gpus)
    return {
        "workload": "%s: %d independent 352x192 streams per GPU x 1 GOP (1 I + 11 P, 12 slices/picture), "
                    "%d distinct seeds replicated" % (name, streams, min(DISTINCT, streams)),
        "streams_per_gpu": streams, "pictures_per_stream": PICTURES, "slices_per_picture": 12,
        "parallelism": "independent-stream sharding x%d" % n_gpus,
        "l2": "inputs exceed L2 (ES + frame stores > 126 MB per GPU), no explicit flush",
    }


def make_streams(streams, rank=0):
    """D distinct synthetic streams (rank-specific window of the seed space) replicated to `streams`."""
    from espflix_b200 import shard, synth
    d = min(DISTINCT, streams)
    gen = synth.generate_many(d, first_index=shard.stream_seed_index(rank, 0, d), n_pictures=PICTURES, gop=PICTURES, slices=12)
    return gen, [gen[i % d][0] for i in range(streams)]


class ClockSampler(threading.Thread):
    """nvidia-smi clocks + throttle reasons during the timed region (B200_PROFILING.md recipe)."""

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.rows, self.stop_flag = index, [], False

    def run(self):
        q = "clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
            "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"
        while not self.stop_flag:
            try:
                r = subprocess.run(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + q, "--format=csv,noheader,nounits"],
                                   capture_output=True, text=True, timeout=5)
                if r.returncode == 0 and r.stdout.strip():
                    self.rows.append([c.strip() for c in r.stdout.strip().split(",")])
            except Exception:
                pass
            time.sleep(0.05)

    def summary(self):
        self.stop_flag = True
        if not self.rows:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        sm = sorted(int(float(r[0])) for r in self.rows)
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for k, n in enumerate(names) if any(r[2 + k].lower().startswith("active") for r in self.rows)]
        return {"sm_mhz": sm[len(sm) // 2], "sm_max_mhz": int(float(self.rows[0][1])), "reasons": reasons, "samples": len(sm)}


# ------------------------------------------------------------------------------------------------
# CPU arm: the reference's own decoder on the host cores
# ------------------------------------------------------------------------------------------------
def cpu_decode_sample(gen, cores, loops):
    """Every core decodes one distinct stream `loops` times back to back (one process per core: the
    reference keeps decoder scratch in process globals, Q11). Returns (frames, seconds, kind)."""
    from espflix_b200 import synth
    ref_bin = os.path.join(ROOT, "oracle", "_ref", "efref_decode")
    tmp = tempfile.mkdtemp(prefix="efbench_")
    paths = []
    for i in range(min(cores, len(gen))):
        p = os.path.join(tmp, "s%d.ts" % i)
        with open(p, "wb") as f:
            f.write(synth.wrap_ts(*gen[i]).tobytes())
        paths.append(p)
    if os.path.exists(ref_bin):
        t0 = time.perf_counter()
        procs = [subprocess.Popen([ref_bin, paths[c % len(paths)], "-", str(loops)], stdout=subprocess.PIPE) for c in range(cores)]
        frames = 0
        for p in procs:
            out, _ = p.communicate(timeout=600)
            frames += json.loads(out)["frames"]
        return frames, time.perf_counter() - t0, "reference"
    # fallback: the C restatement, one thread per core (it has no global state)
    from concurrent.futures import ThreadPoolExecutor
    from tests.oracle_lib import Oracle
    o = Oracle()
    data = [synth.wrap_ts(*gen[i]).tobytes() * max(1, loops // 8) for i in range(min(cores, len(gen)))]
    t0 = time.perf_counter()
    with ThreadPoolExecutor(cores) as ex:
        frames = sum(ex.map(lambda c: int(o.decode_ts(data[c % len(data)], max_frames=PICTURES * max(1, loops // 8) + 2).shape[0]), range(cores)))
    return frames, time.perf_counter() - t0, "port"


def calibrate_loops(gen, target_s):
    frames, secs, _ = cpu_decode_sample(gen, 1, 20)
    per_loop = secs / 20.0
    return max(10, int(target_s / max(per_loop, 1e-6)))


def host_description():
    """What the CPU arm ran on: the rate per process differs 4x between hosts of this pool (BASELINE.md 3)."""
    d = {"cpu_count": os.cpu_count(), "affinity": len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else None}
    try:
        for ln in open("/proc/cpuinfo"):
            if ln.startswith("model name"):
                d["cpu_model"] = ln.split(":", 1)[1].strip()
                break
    except OSError:
        pass
    for path in ("/sys/fs/cgroup/cpu.max", "/sys/fs/cgroup/cpu/cpu.cfs_quota_us"):
        try:
            d["cgroup_cpu_max"] = open(path).read().strip()
            break
        except OSError:
            pass
    try:
        d["loadavg"] = open("/proc/loadavg").read().split()[0]
    except OSError:
        pass
    return d


def usable_cpus():
    return len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)


def best_process_count(gen):
    """The reference runs a decoder thread plus a producer thread per process; on an SMT host one
    process per hardware thread can be slower than one per core. Try both briefly, keep the faster."""
    hw = usable_cpus()
    best, best_rate = hw, 0.0
    loops = calibrate_loops(gen, 1.5)
    for p in sorted({hw, max(1, hw // 2)}, reverse=True):
        f, s, _ = cpu_decode_sample(gen, p, loops)
        if f / s > best_rate:
            best, best_rate = p, f / s
    return best


def run_reference(args):
    rank, world = env_int("RANK", 0), env_int("WORLD_SIZE", 1)
    if rank != 0:
        return 0
    gen, _ = make_streams(DISTINCT)
    cores = best_process_count(gen)
    total_budget = 100.0
    per_step = min(15.0, total_budget / max(1, args.steps + args.warmup))
    loops = max(10, calibrate_loops(gen, per_step) // 3)     # a loaded host runs each process ~3x slower than a lone one
    for _ in range(args.warmup):
        cpu_decode_sample(gen, cores, max(10, loops // 4))
    frames = secs = 0.0
    kind = "reference"
    for _ in range(args.steps):
        f, s, kind = cpu_decode_sample(gen, cores, loops)
        frames += f
        secs += s
    value = frames / secs
    sample = "%d processes (of %d usable hardware threads) x %d loops of one 12-picture synthetic stream each (TS-wrapped, same seeds as the GPU arm)" % (cores, usable_cpus(), loops)
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": 1000.0 * secs / max(1, args.steps), "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "int32/u8", "data": "synthetic", "config": workload_config(args.gpus, STREAMS_PER_GPU),
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": kind, "sample": sample, "per_process": value / cores, "host": host_description()},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)
    return 0


# ------------------------------------------------------------------------------------------------
# GPU arm
# ------------------------------------------------------------------------------------------------
def bind_to_gpu_numa(local):
    """Pin this rank to the CPUs of its GPU's NUMA node and prefer that node's memory, BEFORE any pinned buffer
    exists: cudaHostAlloc'ed pages are placed by first touch, and round 1's 8-GPU end-to-end rate collapsed on
    cross-socket host copies (VERDICT r01, weak #4). Returns what was done (goes into the JSON line)."""
    info = {"bound": False}
    try:
        r = subprocess.run(["nvidia-smi", "-i", str(local), "--query-gpu=pci.bus_id", "--format=csv,noheader"], capture_output=True, text=True, timeout=10)
        bus = r.stdout.strip().splitlines()[0].strip().lower()          # 00000000:1b:00.0
        if bus.count(":") == 2 and len(bus.split(":")[0]) == 8:
            bus = bus[4:]
        node = int(open("/sys/bus/pci/devices/%s/numa_node" % bus).read().strip())
        info.update({"pci": bus, "node": node})
        if node < 0:
            return info
        cpus = set()
        for part in open("/sys/devices/system/node/node%d/cpulist" % node).read().strip().split(","):
            a, _, b = part.partition("-")
            cpus.update(range(int(a), int(b or a) + 1))
        allowed = cpus & os.sched_getaffinity(0)
        if allowed:
            os.sched_setaffinity(0, allowed)
            info.update({"bound": True, "cpus": len(allowed)})
        try:                                                            # set_mempolicy(MPOL_PREFERRED, {node})
            import ctypes
            mask = (ctypes.c_ulong * 16)()
            mask[node // 64] = 1 << (node % 64)
            rc = ctypes.CDLL(None, use_errno=True).syscall(238, 1, mask, 16 * 64 + 1)
            info["mempolicy"] = "preferred" if rc == 0 else "errno %d" % ctypes.get_errno()
        except Exception as e:                                          # noqa: BLE001
            info["mempolicy"] = "unavailable: %s" % e
    except Exception as e:                                              # noqa: BLE001
        info["error"] = str(e)[:120]
    return info


DUMP_STREAMS = 64          # 64 streams x 2 pictures x 101,376 samples x 4 bytes = 52 MB


def dump_outputs(ctx, out_dir, streams):
    """What the last timed step left in the frame store, as a caller of ef_decode_all reads it back: the last and
    the second-to-last picture (I420) of a fixed, seeded sample of this rank's streams, in stream order, as float32
    arrays DIR/frames_last.npy and DIR/frames_prev.npy of shape (min(64, streams), 101376)."""
    os.makedirs(out_dir, exist_ok=True)
    sample = np.sort(np.random.default_rng(0).choice(streams, size=min(DUMP_STREAMS, streams), replace=False))
    last = np.stack([ctx.read_frame_i420(int(i), -1) for i in sample])
    prev = np.stack([ctx.read_frame_i420(int(i), ((ctx.stream_info(int(i))[1] + PICTURES) & 1) ^ 1) for i in sample])
    np.save(os.path.join(out_dir, "frames_last.npy"), last.astype(np.float32))
    np.save(os.path.join(out_dir, "frames_prev.npy"), prev.astype(np.float32))


def run_gpu(args):
    rank, world, local = env_int("RANK", 0), env_int("WORLD_SIZE", 1), env_int("LOCAL_RANK", 0)
    if args.gpus > 1 and world == 1:       # convenience: re-launch under torchrun
        cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", str(args.gpus),
               "--master-addr", "127.0.0.1", "--master-port", str(29500 + os.getpid() % 2000), os.path.abspath(__file__)] + sys.argv[1:]
        return subprocess.call(cmd)
    os.environ.setdefault("CUDA_DEVICE_ORDER", "PCI_BUS_ID")             # nvidia-smi index == CUDA ordinal
    orig_affinity = os.sched_getaffinity(0)
    numa = {"bound": False, "disabled": True} if args.no_numa else bind_to_gpu_numa(local)

    import torch
    import espflix_b200

    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the product has no CPU path (use --impl reference for the CPU arm)")
    torch.cuda.set_device(local)
    dist = None
    if world > 1:
        import torch.distributed as dist
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        # stdout must carry exactly one JSON line: NCCL prints its version banner to stdout while the
        # communicator is created, so fd 1 points at stderr until the first collective has run
        sys.stdout.flush()
        saved_fd = os.dup(1)
        os.dup2(2, 1)
        try:
            dist.init_process_group("nccl", device_id=torch.device("cuda", local))
            dist.barrier()
            torch.cuda.synchronize()
        finally:
            sys.stdout.flush()
            os.dup2(saved_fd, 1)
            os.close(saved_fd)

    if args.scaling == "strong":
        if args.total_streams % world:
            raise SystemExit("--total-streams must be a multiple of the number of GPUs")
        streams = args.total_streams // world
    else:
        streams = args.streams
    gen, stream_list = make_streams(streams, rank)
    sizes = np.diff(gen[0][1].astype(np.int64))
    from espflix_b200 import synth
    ts_distinct = [synth.wrap_ts(*g) for g in gen]            # the reference's wire format (188-byte TS, PID 0x100) of the same streams
    ts_bytes_total = sum(len(ts_distinct[i % len(gen)]) for i in range(streams))
    ctx = espflix_b200.Context(n_streams=streams, max_pictures=PICTURES, max_slices_per_picture=12,
                               es_capacity=max(sum(len(s) for s in stream_list), ts_bytes_total) + 4096, device=local, fields=True)
    blob_np, off_np = ctx.pack(stream_list)
    es_bytes = int(off_np[-1])
    pinned_es = torch.empty(es_bytes, dtype=torch.uint8, pin_memory=True)
    pinned_es.numpy()[:] = blob_np
    del blob_np
    pinned_out = [torch.empty((streams, FRAME_BYTES), dtype=torch.uint8, pin_memory=True) for _ in range(2)]
    dev_es = pinned_es.cuda()
    dev_off = torch.from_numpy(off_np.astype(np.int64)).cuda()
    st = 0                                                # legacy default stream == torch's default stream

    # algorithmic bytes of K1 per step (SURVEY.md 8d): I: S + 101,376 ; P: S + 202,752
    n_i = 1
    algo_bytes = es_bytes + streams * (n_i * FRAME_BYTES + (PICTURES - n_i) * 2 * FRAME_BYTES)

    def step_resident(events=None):
        ctx.index(st)
        if events is not None:
            events[0].record()
        ctx.decode_all(PICTURES, st)          # K1a once over all 12 picture indices, then K1b per picture index
        if events is not None:
            events[1].record()

    def barrier():
        torch.cuda.synchronize()
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    # host <-> device link probe, all ranks at once (names the ceiling of the end-to-end legs with a number)
    probe = torch.empty(256 << 20, dtype=torch.uint8, pin_memory=True)
    probe_dev = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")
    probe_dev2 = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")
    probe2 = torch.empty(256 << 20, dtype=torch.uint8, pin_memory=True)
    side = torch.cuda.Stream()
    link = {}
    for name in ("h2d", "d2h", "both"):
        for timed in (False, True):
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            barrier()
            a.record()
            for _ in range(4):
                if name in ("h2d", "both"):
                    probe_dev.copy_(probe, non_blocking=True)
                if name == "d2h":
                    probe.copy_(probe_dev, non_blocking=True)
                if name == "both":
                    with torch.cuda.stream(side):
                        probe2.copy_(probe_dev2, non_blocking=True)
            side.synchronize()
            b.record()
            barrier()
            if timed:
                link[name + "_gbs"] = 4 * (256 << 20) / (a.elapsed_time(b) / 1000.0) / 1e9
    del probe, probe2, probe_dev, probe_dev2

    ctx.submit_es(dev_es.data_ptr(), dev_off.data_ptr(), st, device=True)
    for _ in range(args.warmup):
        step_resident()

    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    ev = [[torch.cuda.Event(enable_timing=True) for _ in range(2)] for _ in range(args.steps)]
    t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    launches0 = ctx.launch_count()
    barrier()
    t0.record()
    for k in range(args.steps):
        step_resident(ev[k])
    t1.record()
    barrier()
    launches = ctx.launch_count() - launches0
    ms_total = t0.elapsed_time(t1)
    k1_ms = sum(ev[k][0].elapsed_time(ev[k][1]) for k in range(args.steps))
    info = ctx.index_info()
    assert info["total_pictures"] == streams * PICTURES, info
    if args.dump_outputs and rank == 0:
        dump_outputs(ctx, args.dump_outputs, streams)

    # --verify (checker only, after the timed region): this rank's first distinct streams through the oracle
    verified = None
    if not args.no_verify:
        from tests.oracle_lib import Oracle
        oracle = Oracle()
        verified = 0
        for i in range(min(2, len(gen))):
            want = oracle.decode_es(gen[i][0])
            base = ctx.stream_info(i)[1]
            ok = np.array_equal(ctx.read_frame_i420(i, -1), want[-1]) and np.array_equal(ctx.read_frame_i420(i, ((base + PICTURES) & 1) ^ 1), want[-2])
            if not ok:
                raise SystemExit("bench.py --verify: rank %d stream %d differs from the oracle" % (rank, i))
            verified += 1

    # per-stage split (K0 index / K1a parse / K1b reconstruction) from the library's own events, on untimed extra steps
    ctx.set_profiling(True)
    stage = np.zeros(3)
    for _ in range(3):
        step_resident()
        stage += np.array(ctx.stage_ms())
    stage /= 3.0
    ctx.set_profiling(False)

    # e2e: host buffers through the C-ABI, copies inside the timed region
    # Every step uploads its input from pinned host memory and brings its result back to pinned host
    # memory. The C-ABI double-buffers both directions, so the upload of step k+1 and the read-back of
    # step k overlap the decode kernels; the clock stops only after everything has landed on the host.
    def step_e2e(k):
        ctx.submit_es(pinned_es.data_ptr(), off_np, st, device=False)
        ctx.index(st)
        ctx.decode_all(PICTURES, st)
        ctx.read_latest_i420_async(0, streams, pinned_out[k & 1].data_ptr(), st)

    def timed_host_loop(step, n):
        step(0)
        ctx.sync(st)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        barrier()
        e0.record()
        w0 = time.perf_counter()
        for k in range(n):
            step(k)
        e1.record()
        ctx.sync(st)
        wall_ms = 1000.0 * (time.perf_counter() - w0)
        barrier()
        return max(e0.elapsed_time(e1), wall_ms)          # copies run on the library's own streams: the wall clock up to ef_sync covers them

    e2e_ms = timed_host_loop(step_e2e, args.steps)
    clocks = sampler.summary() if rank == 0 else None

    # e2e_ts: the same end-to-end step fed with transport streams (device-side TS/PES demux in front of the index)
    e2e_ts_ms, ts_steps = None, 0
    if not args.no_e2e_ts:
        ts_off = np.zeros(streams + 1, dtype=np.uint64)
        ts_off[1:] = np.cumsum([len(ts_distinct[i % len(gen)]) for i in range(streams)])
        pinned_ts = torch.empty(int(ts_off[-1]), dtype=torch.uint8, pin_memory=True)
        view = pinned_ts.numpy()
        for i in range(streams):
            view[int(ts_off[i]):int(ts_off[i + 1])] = ts_distinct[i % len(gen)]

        def step_ts(k):
            ctx.submit_ts(pinned_ts.data_ptr(), ts_off, st, device=False)
            ctx.index(st)
            ctx.decode_all(PICTURES, st)
            ctx.read_latest_i420_async(0, streams, pinned_out[k & 1].data_ptr(), st)

        ts_steps = max(1, min(args.steps, 10))
        e2e_ts_ms = timed_host_loop(step_ts, ts_steps)
        ts_total_bytes = int(ts_off[-1])
        if not args.no_verify:
            ctx.sync(st)
            want = oracle.decode_es(gen[0][0])
            if not np.array_equal(ctx.read_frame_i420(0, -1), want[-1]):
                raise SystemExit("bench.py --verify: rank %d: TS-fed decode differs from the oracle" % rank)
        del pinned_ts

    # e2e_all: every decoded picture handed to the host (12x the read-back of `e2e`): PCIe bound
    all_steps, e2e_all_ms, all_bytes = 0, None, PICTURES * streams * FRAME_BYTES
    if not args.no_e2e_all and all_bytes <= (8 << 30):
        pinned_all = torch.empty((PICTURES, streams, FRAME_BYTES), dtype=torch.uint8, pin_memory=True)

        def step_all(k):
            ctx.submit_es(pinned_es.data_ptr(), off_np, st, device=False)
            ctx.index(st)
            ctx.decode_all_to_host(PICTURES, pinned_all.data_ptr(), st)

        all_steps = max(1, min(args.steps, 4))
        e2e_all_ms = timed_host_loop(step_all, all_steps)
        if not args.no_verify:
            want = oracle.decode_es(gen[0][0])
            got = pinned_all.numpy()
            if not all(np.array_equal(got[p, 0], want[p]) for p in range(PICTURES)):
                raise SystemExit("bench.py --verify: rank %d: a picture handed over by ef_decode_all_to_host differs from the oracle" % rank)
        del pinned_all

    # K2: composite field synthesis of the most recent picture of every stream (one launch per field)
    k2 = {}
    for ntsc, name, samples in ((1, "ntsc", 262 * 912), (0, "pal", 312 * 1136)):
        ctx.video_init(ntsc)
        for fc in range(3):
            ctx.composite_field(-1, fc, st)
        c0, c1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        barrier()
        c0.record()
        for fc in range(args.steps):
            ctx.composite_field(-1, fc, st)
        c1.record()
        barrier()
        ms = c0.elapsed_time(c1) / args.steps
        bytes_per_field = FRAME_BYTES + samples * 2                     # frame read once, whole field written (SURVEY.md 8d)
        k2[name] = {"fields_per_s": streams / (ms / 1000.0), "ms_per_launch": ms,
                    "achieved_gbs": streams * bytes_per_field / (ms / 1000.0) / 1e9, "algorithmic_bytes_per_field": bytes_per_field}
    ctx.video_init(1)

    # max over ranks, total frames via one all_gather (reporting only)
    frames_done = streams * PICTURES * args.steps
    link_min, link_sum = dict(link), dict(link)
    if dist is not None:
        t = torch.tensor([ms_total, k1_ms, e2e_ms, e2e_all_ms or 0.0, e2e_ts_ms or 0.0], device="cuda", dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms_total, k1_ms, e2e_ms, e2e_all_max, e2e_ts_max = [float(x) for x in t.tolist()]
        e2e_all_ms = e2e_all_max if e2e_all_ms is not None else None
        e2e_ts_ms = e2e_ts_max if e2e_ts_ms is not None else None
        lt = torch.tensor([link["h2d_gbs"], link["d2h_gbs"], link["both_gbs"]], device="cuda", dtype=torch.float64)
        lmin, lsum = lt.clone(), lt.clone()
        dist.all_reduce(lmin, op=dist.ReduceOp.MIN)
        dist.all_reduce(lsum, op=dist.ReduceOp.SUM)
        link_min = dict(zip(("h2d_gbs", "d2h_gbs", "both_gbs"), [float(x) for x in lmin.tolist()]))
        link_sum = dict(zip(("h2d_gbs", "d2h_gbs", "both_gbs"), [float(x) for x in lsum.tolist()]))
        counts = [torch.zeros(1, dtype=torch.int64, device="cuda") for _ in range(world)]
        dist.all_gather(counts, torch.tensor([frames_done], dtype=torch.int64, device="cuda"))
        total_frames = int(sum(int(c.item()) for c in counts))
        numa_all = [None] * world
        dist.all_gather_object(numa_all, numa)
    else:
        total_frames = frames_done
        numa_all = [numa]
    value = total_frames / (ms_total / 1000.0)
    e2e_value = total_frames / (e2e_ms / 1000.0)

    if rank == 0:
        peaks_path = os.path.join(ROOT, "MEASURED_PEAKS.json")
        if os.path.exists(peaks_path):
            peak, peak_src = float(json.load(open(peaks_path))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        else:
            peak, peak_src = 6650.0, "fallback (B200_PROFILING.md)"
        achieved = algo_bytes * args.steps / (k1_ms / 1000.0) / 1e9
        traffic = None
        tpath = os.path.join(ROOT, "profiles", "k1_traffic.json")
        if os.path.exists(tpath):
            traffic = json.load(open(tpath)).get("dram_bytes_per_launch")
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms_total / args.steps, "higher_is_better": True, "scaling": args.scaling, "vs_baseline": None,
            "dtype": "int32/u8", "data": "synthetic", "config": workload_config(world, streams, args.scaling),
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": es_bytes + int(off_np.nbytes),
                    "d2h_bytes_per_step": streams * FRAME_BYTES, "ms_per_step": e2e_ms / args.steps,
                    "pictures_read_back_per_stream": 1, "pictures_decoded_per_stream": PICTURES,
                    "what": "per step: pinned ES -> ef_submit_es_host -> ef_index -> ef_decode_all(12) -> ef_read_latest_i420_async: ONLY the last of the 12 decoded pictures of every stream goes back to pinned host memory (1/12 of the decoded bytes; e2e_all hands over all 12); copies double-buffered, clock stops after ef_sync"},
            "gpu_launches": int(launches),
            "clocks": clocks,
            "roofline": {"bound": "hbm", "kernel": "K1 = ef_parse_kernel (1 launch per step) + ef_recon_kernel (12 launches per step); achieved = algorithmic decode bytes / time of the pair", "achieved": achieved, "peak": peak, "unit": "GB/s",
                         "frac": achieved / peak, "traffic": traffic, "peak_source": peak_src,
                         "algorithmic_bytes_per_step": algo_bytes, "k1_ms_per_step": k1_ms / args.steps,
                         "k1_share_of_step": k1_ms / ms_total},
            "composite": {k: dict(v, frac=v["achieved_gbs"] / peak) for k, v in k2.items()},
            "stages_ms": {"k0_index": round(float(stage[0]), 4), "k1a_parse": round(float(stage[1]), 4), "k1b_recon_x12": round(float(stage[2]), 4)},
            "host_link": {"per_rank_min_gbs": link_min, "all_ranks_sum_gbs": link_sum, "probe": "4 x 256 MiB pinned copies per direction, all ranks at once; 'both' = H2D and D2H concurrently (rate per direction)"},
            "numa": numa_all,
            "verify": None if verified is None else "ok: %d distinct streams per rank (last two pictures) + all 12 handed-over pictures of stream 0 equal the oracle" % verified,
            "per_gpu_frames_per_s": value / world,
            "es_bytes_per_picture": es_bytes / (streams * PICTURES),
            "picture_bytes_first_stream": [int(x) for x in sizes],
        }
        if e2e_all_ms is not None:
            line["e2e_all"] = {"value": (total_frames / args.steps * all_steps) / (e2e_all_ms / 1000.0), "unit": UNIT, "steps": all_steps,
                               "h2d_bytes_per_step": es_bytes + int(off_np.nbytes), "d2h_bytes_per_step": all_bytes, "ms_per_step": e2e_all_ms / all_steps,
                               "what": "per step: pinned ES -> ef_submit_es_host -> ef_index -> ef_decode_all_to_host(12): every decoded picture of every stream is exported after its reconstruction launch and copied to pinned host memory while the next picture index is rebuilt (the reference's push_video hand-over of every picture)"}
        if e2e_ts_ms is not None:
            line["e2e_ts"] = {"value": (total_frames / args.steps * ts_steps) / (e2e_ts_ms / 1000.0), "unit": UNIT, "steps": ts_steps,
                              "h2d_bytes_per_step": ts_total_bytes, "d2h_bytes_per_step": streams * FRAME_BYTES, "ms_per_step": e2e_ts_ms / ts_steps,
                              "what": "as e2e, but the input is the reference's wire format: 188-byte transport packets, PID 0x100, one PES per picture (ef_submit_ts_host: packet kernel + per-stream scan + compaction on the device, player.cpp:381-493)"}
        if world == 1 and not args.no_cpu:
            os.sched_setaffinity(0, orig_affinity)                       # the CPU arm uses every core the job may use, not the GPU's NUMA node only
            cores = best_process_count(gen)
            loops = max(10, calibrate_loops(gen, 12.0) // 3)
            f, s, kind = cpu_decode_sample(gen, cores, loops)
            line["cpu_baseline"] = {"value": f / s, "unit": UNIT, "cores": cores, "kind": kind, "per_process": f / s / cores, "host": host_description(),
                                    "sample": "%d processes (of %d usable hardware threads) x %d loops of one 12-picture synthetic stream each (TS-wrapped), %.1f s" % (cores, usable_cpus(), loops, s)}
        print(json.dumps(line), flush=True)
    ctx.close()
    if dist is not None:
        dist.destroy_process_group()
    return 0


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=40)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--streams", type=int, default=STREAMS_PER_GPU, help="streams per GPU (default: the BASELINE config)")
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg (profiling runs)")
    ap.add_argument("--scaling", default="weak", choices=["weak", "strong"], help="weak: --streams per GPU (default); strong: --total-streams split over the GPUs (BASELINE config 5)")
    ap.add_argument("--total-streams", type=int, default=32768, help="strong scaling: streams of the whole job")
    ap.add_argument("--no-verify", action="store_true", help="skip the oracle check of this rank's first distinct streams after the timed region")
    ap.add_argument("--no-e2e-all", action="store_true", help="skip the all-pictures read-back leg (5 GB pinned per GPU)")
    ap.add_argument("--no-e2e-ts", action="store_true", help="skip the transport-stream input leg")
    ap.add_argument("--no-numa", action="store_true", help="do not pin the rank to its GPU's NUMA node")
    ap.add_argument("--dump-outputs", metavar="DIR", help="after the timed steps, write the decoded pictures of the last step "
                    "(last two pictures of 64 seeded-sampled streams of rank 0) to DIR as float32 .npy files")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the GPU path's pictures; --impl reference has none")
    args.warmup = max(args.warmup, 0)
    import __graft_entry__
    if not os.path.exists(os.path.join(ROOT, "espflix_b200", "libespflix_b200.so")):
        __graft_entry__.build()
    if args.impl == "reference":
        return run_reference(args)
    return run_gpu(args)


if __name__ == "__main__":
    sys.exit(main())
