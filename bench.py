#!/usr/bin/env python
"""bench.py -- mapped query Gbp/s of the B200 mapping hot path (BASELINE.json metric).

Workload (BASELINE.json configs[1]): 1 M synthetic ONT-like reads x 10 kb (per-read error ~ U[2 %,14 %],
sub:ins:del 4:3:3) against a 3 Gbp uniform-random reference, MashMap defaults `-s 5000 --pi 85`
(k = 19, sketch size = Stat::recommendedSketchSize for a 3.05 GB FASTA = 220).

A "step" = one pass of the hot path over the whole read batch (2 M segments):
  value  -- inputs resident in HBM: K1 sketch -> K2 L1 -> K3 L2 (mm_map_resident of the C ABI), timed with CUDA
            events on the launching stream (first launch -> last kernel end, including the counter read-backs).
  e2e    -- the same batch through the reference-facing host API (skch::BatchMapper = mm_map_segments with HOST
            buffers + the host tail to PAF text): H2D and D2H copies and the host tail inside the timed region.
N > 1 (torchrun): weak scaling -- every rank maps its own 1 M reads against the same index; rank 0 builds the
index and broadcasts the device image (one NCCL broadcast over NVLink); mapping records of all ranks are
gathered on rank 0 at the end of every e2e step (one all_gather of counts + one of padded records).

--impl reference: the reference's CPU implementation of the same path on the host cores (bounded sample per
step), see cpu_arm().
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

K = 19
REF_FASTA_BYTES_PER_BASE = 81.0 / 80.0  # 80-column FASTA: what recommendedSketchSize is fed (file size in bytes)

# BASELINE.json configs[1..4] (configs[0], the yeast self-map, is the reference's own CPU-runnable case: tests/test_gpu_cli.py)
CONFIGS = {
    2: dict(tag="configs[1]", kind="reads", reads=1_000_000, read_len=10_000, err=(0.02, 0.14), seg=5000, pi=0.85, dense=False,
            filt="map", scaling="weak", what="synthetic ONT reads"),
    3: dict(tag="configs[2]", kind="reads", reads=1_000_000, read_len=10_000, err=(0.02, 0.14), seg=5000, pi=0.95, dense=True,
            filt="map", scaling="weak", what="synthetic ONT reads"),
    4: dict(tag="configs[3]", kind="reads", reads=100_000, read_len=20_000, err=(0.004, 0.006), seg=5000, pi=0.95, dense=False,
            filt="one-to-one", scaling="strong", what="synthetic HiFi-like reads"),
    5: dict(tag="configs[4]", kind="assembly", seg=10_000, pi=0.90, dense=False, filt="one-to-one", scaling="strong",
            snp=0.03, indel=0.003, inversions=100, translocations=100, what="contigs of a second synthetic assembly"),
}


def log(*a):
    print("[bench]", *a, file=sys.stderr, flush=True)


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--config", type=int, default=2, choices=sorted(CONFIGS), help="BASELINE.json configuration (2 = configs[1], the "
                    "one the metric is quoted on; 3 = --dense --pi 95; 4 = HiFi one-to-one, strong scaling; 5 = assembly vs assembly)")
    # workload overrides (tests / quick runs only; the defaults are the BASELINE configuration)
    ap.add_argument("--reads", type=int, default=0, help="0 = the configuration's own number of reads")
    ap.add_argument("--ref-bp", type=int, default=3_000_000_000)
    ap.add_argument("--contigs", type=int, default=256)
    ap.add_argument("--cpu-sample-reads", type=int, default=0, help="reads per CPU-baseline sample (0 = auto)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--cpu-kind", default="auto", choices=["auto", "reference", "port"], help="cpu_baseline leg of the b200 arm: 'reference' = the "
                    "unmodified reference (oracle/_ref/libmm_ref.so builds its own index from the FASTA of the bench's reference: + 1.5 min "
                    "of set-up at 3 Gbp); 'port' = the oracle restatement on the product's index content; 'auto' = reference when the "
                    "library is there")
    ap.add_argument("--sketch", type=int, default=0, help="sketch size override (0 = the reference's automatic choice)")
    ap.add_argument("--ref-kind", default="auto", choices=["auto", "real", "port"], help="--impl reference: 'real' = the unmodified reference "
                    "(oracle/_ref/libmm_ref.so: its own index build from FASTA, its own mapModule); 'port' = the oracle restatement on the "
                    "product's index content; 'auto' = real when the library is there")
    ap.add_argument("--as-rank", type=int, default=-1, help="debug: generate the reads rank R of a multi-GPU run would get (read seed 2 + R)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None, help="after the timed steps, write what the last step computed as "
                    "DIR/<name>.npy (float64; a fixed, seeded sample of the fragments and reads), see dump_outputs()")
    return ap.parse_args()


class ClockSampler:
    """samples nvidia-smi clocks / throttle reasons during the timed region"""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index = index
        self.proc = None
        self.lines = []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100",
                                          "-i", str(self.index)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append((time.time(), line.strip()))

    def stop(self, t0, t1):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm, mx, reasons = [], [], set()
        for t, line in self.lines:
            f = [x.strip() for x in line.split(",")]
            if len(f) < 9 or not (t0 - 0.05 <= t <= t1 + 0.15):
                continue
            try:
                sm.append(float(f[1])); mx.append(float(f[2]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no samples in the timed region"]}
        return {"sm_mhz": float(np.median(sm)), "sm_max_mhz": float(max(mx)), "reasons": sorted(reasons), "samples": len(sm)}


def host_cpu_info():
    """what the host side really has: visible CPUs, affinity, cgroup quota (a container can show 128 CPUs and be allowed a
    fraction of them) -- reported next to cpu_baseline.cores, which is the number of threads used"""
    info = {"visible": os.cpu_count(), "affinity": len(os.sched_getaffinity(0))}
    try:
        q = open("/sys/fs/cgroup/cpu.max").read().split()
        if q and q[0] != "max":
            info["cgroup_quota_cpus"] = round(int(q[0]) / int(q[1]), 2)
    except Exception:
        try:
            q = int(open("/sys/fs/cgroup/cpu/cpu.cfs_quota_us").read())
            per = int(open("/sys/fs/cgroup/cpu/cpu.cfs_period_us").read())
            if q > 0:
                info["cgroup_quota_cpus"] = round(q / per, 2)
        except Exception:
            pass
    return info


def usable_cpus():
    """CPUs this process can really use: visible CPUs, limited by the affinity mask and the cgroup CPU quota"""
    info = host_cpu_info()
    n = min(info["visible"] or 8, info["affinity"])
    if "cgroup_quota_cpus" in info:
        n = min(n, max(1, int(info["cgroup_quota_cpus"])))
    return max(1, n)


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md)"


def roofline_traffic():
    """dram bytes per launch of the sketch kernel from the committed ncu capture, if any"""
    p = os.path.join(ROOT, "profiles", "roofline_traffic.json")
    if os.path.exists(p):
        try:
            return json.load(open(p))
        except Exception:
            return {}
    return {}


def issue_peak():
    """measured INT32 issue rates (mashmap_b200/mm_issue_peak on this pool's B200), if committed"""
    p = os.path.join(ROOT, "profiles", "issue_peak.json")
    if os.path.exists(p):
        try:
            return json.load(open(p))
        except Exception:
            return None
    return None


def host_memory_info():
    """memory this process group may use: cgroup limit / current use, MemTotal / MemAvailable, the locked-memory ulimit"""
    info = {}
    for name, path in (("cgroup_max", "/sys/fs/cgroup/memory.max"), ("cgroup_current", "/sys/fs/cgroup/memory.current")):
        try:
            v = open(path).read().strip()
            info[name] = v if v == "max" else round(int(v) / 2**30, 1)
        except Exception:
            pass
    try:
        for line in open("/proc/meminfo"):
            f = line.split()
            if f[0] in ("MemTotal:", "MemAvailable:"):
                info[f[0][:-1]] = round(int(f[1]) / 2**20, 1)
    except Exception:
        pass
    return info


def rss_gb():
    try:
        for line in open("/proc/self/status"):
            if line.startswith("VmRSS:"):
                return round(int(line.split()[1]) / 2**20, 1)
    except Exception:
        pass
    return None


def keep_rank_stderr(rank):
    """every rank's stderr also goes to its own file (MM_BENCH_LOGDIR, default gpurun_out/ when that directory exists):
    torchrun only shows the tail of the merged stream, and a rank that dies with exit(1) must leave its reason behind"""
    d = os.environ.get("MM_BENCH_LOGDIR") or (os.path.join(ROOT, "gpurun_out") if os.path.isdir(os.path.join(ROOT, "gpurun_out")) else None)
    if not d:
        return
    try:
        os.makedirs(d, exist_ok=True)
        path = os.path.join(d, f"bench_rank{rank}.log")
        tee = subprocess.Popen(["tee", "-a", path], stdin=subprocess.PIPE, stdout=sys.stderr.fileno())
        os.dup2(tee.stdin.fileno(), 2)
    except Exception as e:  # never fatal
        print(f"[bench] rank {rank}: cannot keep a per-rank log: {e}", file=sys.stderr)


def _gpu_numa_node(pynvml, index):
    h = pynvml.nvmlDeviceGetHandleByIndex(index)
    node = None
    try:
        node = pynvml.nvmlDeviceGetNumaNodeId(h)
    except Exception:
        pass
    if node is None or node < 0:
        bus = pynvml.nvmlDeviceGetPciInfo(h).busId
        bus = bus.decode() if isinstance(bus, bytes) else bus
        node = int(open(f"/sys/bus/pci/devices/{bus[-12:].lower()}/numa_node").read())
    return node


def bind_to_gpu_numa_node(local_rank, world=1):
    """CPU affinity (and with it first-touch memory placement) of this rank = the NUMA node its GPU hangs off: the pinned
    batch buffer and the host tail then stay on the socket whose PCIe root the copies use. Returns (node, CPUs of the node
    this process may use, ranks of this job whose GPU hangs off the same node) or None."""
    try:
        import pynvml

        pynvml.nvmlInit()
        node = _gpu_numa_node(pynvml, local_rank)
        if node < 0:
            return None
        sharing = 0
        for r in range(world):  # one rank per GPU, rank r on GPU r of this node (torchrun's LOCAL_RANK)
            try:
                sharing += _gpu_numa_node(pynvml, r) == node
            except Exception:
                pass
        cpus = []
        for part in open(f"/sys/devices/system/node/node{node}/cpulist").read().strip().split(","):
            a, _, b = part.partition("-")
            cpus += list(range(int(a), int(b or a) + 1))
        cpus = sorted(set(cpus) & os.sched_getaffinity(0))
        if cpus:
            os.sched_setaffinity(0, cpus)
            return node, len(cpus), max(1, sharing)
    except Exception as e:
        log(f"NUMA binding skipped: {e}")
    return None


def host_threads_for_rank(world, numa):
    """host threads of one rank: its share of the CPUs it can really run on. Without a NUMA binding that is usable CPUs / ranks;
    with one, the node's CPUs are shared by the ranks bound to that node only (8 GPUs on two nodes of 64 CPUs under a 96-CPU
    quota: min(64 / 4, 96 / 8) = 12 per rank, not 64 / 8). More threads than CPUs only adds throttling."""
    info = host_cpu_info()
    share = usable_cpus() // max(1, world)
    if numa is not None:
        _, node_cpus, sharing = numa
        share = node_cpus // sharing
        if "cgroup_quota_cpus" in info:
            share = min(share, int(info["cgroup_quota_cpus"]) // max(1, world))
    return max(1, share)


def config_of(args):
    cfg = dict(CONFIGS[args.config])
    if cfg["kind"] == "reads":
        if args.reads:
            cfg["reads"] = args.reads
    else:  # assembly: the queries are the contigs of the second genome, cut to one common length
        contig_len = args.ref_bp // args.contigs
        cfg["reads"] = args.contigs
        cfg["read_len"] = contig_len - max(64, contig_len // 100)
    return cfg


def sketch_size_of(args, cfg):
    from mashmap_b200 import hostlib

    if args.sketch:
        return args.sketch
    if cfg["dense"]:  # parseCmdArgs.hpp:626-631
        return int(0.02 * (1 + (1 - cfg["pi"]) / 0.05) * (cfg["seg"] - K))
    # the reference's automatic choice for a file of this size (SURVEY 8(a) table: 220 / 20 / 70). A file >= 2 GiB would in
    # fact wrap the reference's int32 referenceSize (310 for this one, see DESIGN.md); --sketch 310 measures that variant.
    return int(hostlib.lib().skch_recommended_sketch_size(K, cfg["pi"], cfg["seg"], int(args.ref_bp * REF_FASTA_BYTES_PER_BASE) + 16 * args.contigs))


def workload_text(args, cfg, S):
    n, L = cfg["reads"], cfg["read_len"]
    if cfg["kind"] == "reads":
        q = f"{n} {cfg['what']} x {L} bp (err U[{cfg['err'][0] * 100:g}%,{cfg['err'][1] * 100:g}%])"
    else:
        q = (f"{n} contigs x {L} bp of a second assembly ({cfg['snp'] * 100:g}% SNPs, {cfg['indel'] * 100:g}% indels, "
             f"{cfg['inversions']} inversions, {cfg['translocations']} translocations)")
    opts = f"-s {cfg['seg']} --pi {int(cfg['pi'] * 100)}" + (" --dense" if cfg["dense"] else "") + (f" -f {cfg['filt']}" if cfg["filt"] != "map" else "")
    return (f"{q} vs {args.ref_bp / 1e9:.2f} Gbp uniform-random reference ({args.contigs} contigs), {opts}, k={K}, sketch={S} "
            f"(BASELINE.json {cfg['tag']})")


def make_queries(args, cfg, ref, seed_rank):
    """all queries of one step of this rank's workload as text on the device: [n, read_len] uint8 (+ truth for reads)"""
    from mashmap_b200 import synth_gpu

    if cfg["kind"] == "reads":
        return synth_gpu.simulate_reads(ref, cfg["reads"], cfg["read_len"], cfg["err"][0], cfg["err"][1], seed=2 + seed_rank, chunk=8192)
    q = synth_gpu.mutated_genome(ref, cfg["read_len"], cfg["snp"], cfg["indel"], cfg["inversions"], cfg["translocations"], seed=4)
    return q, None


def setup_workload(args, cfg, rank, world, device):
    """reference on the GPU -> host copy for the index builder (rank 0); this rank's queries generated on the GPU.
    weak scaling: every rank its own cfg.reads reads (seed 2 + rank); strong scaling: ONE set, rank r takes its block."""
    import torch

    from mashmap_b200 import dist as mdist
    from mashmap_b200 import synth_gpu

    contig_len = args.ref_bp // args.contigs
    t0 = time.time()
    ref = synth_gpu.random_reference(args.contigs, contig_len, seed=1, device=device)
    S = sketch_size_of(args, cfg)
    strong = cfg["scaling"] == "strong"
    seed_rank = 0 if strong else (args.as_rank if args.as_rank >= 0 else rank)
    q, truth = make_queries(args, cfg, ref, seed_rank)
    lo, hi = (mdist.shard_reads(cfg["reads"], rank, world) if strong else (0, cfg["reads"]))
    first_counter = lo if strong else rank * cfg["reads"]
    if device.type == "cuda":
        torch.cuda.synchronize()
    log(f"rank {rank}: reference {args.contigs} x {contig_len} bp and {cfg['reads']} queries x {cfg['read_len']} bp generated in "
        f"{time.time() - t0:.1f} s; sketch size {S}; this rank maps queries [{lo}, {hi})")
    t = None
    if truth is not None:
        t = tuple(truth[k].cpu().numpy() for k in ("contig", "start", "strand"))
    all_q = q  # strong scaling keeps the whole set on rank 0 for the single-GPU comparison
    return dict(ref_dev=ref if rank == 0 else None, contig_len=contig_len, sketch=S, queries=q[lo:hi], all_queries=all_q if (strong and rank == 0) else None,
                truth=t, lo=lo, hi=hi, first_counter=first_counter)


def build_index_on_device(args, cfg, wl, ctx, keep_lookup):
    """the reference index built on the GPU from the reference text that is already in device memory (mm_index_build)"""
    t0 = time.time()
    offs = np.arange(args.contigs + 1, dtype=np.uint64) * np.uint64(wl["contig_len"])
    st = ctx.index_build(None, offs, device_ptr=wl["ref_dev"].data_ptr(), keep_lookup=keep_lookup)
    log(f"device index: {st['n_minmers']} minmers ({st['n_minmers_before_filter']} before the frequent-seed filter), {st['n_keys']} keys, "
        f"{st['n_points']} points, freq threshold {st['freq_threshold']} in {time.time() - t0:.2f} s (window scan {st['ms_scan'] / 1e3:.2f} s over "
        f"{st['n_chunks']} chunks, {st['n_fixed_chunks']} re-scanned; records {st['ms_post'] / 1e3:.2f} s; lookup {st['ms_lookup'] / 1e3:.2f} s)")
    return st


def build_index_on_host(args, cfg, wl, threads):
    """--impl reference without a GPU: the host builder (the same window machine, one task per contig)"""
    from mashmap_b200 import hostlib

    t0 = time.time()
    offs = np.arange(args.contigs + 1, dtype=np.uint64) * np.uint64(wl["contig_len"])
    hi = hostlib.HostIndex.build(wl["ref_dev"].cpu().numpy().reshape(-1), offs, K, cfg["seg"], wl["sketch"], threads=threads)
    log(f"host index: {hi.n_minmers} minmers, {hi.n_keys} keys, {hi.n_points} points, freq threshold {hi.freq_threshold} "
        f"in {time.time() - t0:.1f} s ({threads} threads)")
    return hi


def text_segments(batch, read_len):
    """the batch's fragments with offsets into the plain text layout (read r at r * read_len) instead of the packed one"""
    seg = batch.segments.copy()
    stride = (read_len + 31) // 32 * 32  # reads sit at multiples of 32 bases in the packed batch
    rd = seg["offset"] // stride
    seg["offset"] = rd * read_len + (seg["offset"] - rd * stride)
    return seg


def gpu_arm(args):
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if world > 1:
        keep_rank_stderr(rank)
    numa = bind_to_gpu_numa_node(local_rank, world) if world > 1 else None
    import torch

    log(f"rank {rank}/{world}: host memory {host_memory_info()}, cpus {host_cpu_info()}, bound to NUMA node {numa}")
    dist = None
    if world > 1:
        import torch.distributed as dist

        dist.init_process_group("nccl", device_id=torch.device(f"cuda:{local_rank}"))
    torch.cuda.set_device(local_rank)
    device = torch.device(f"cuda:{local_rank}")
    from mashmap_b200 import capi, hostlib
    from mashmap_b200 import nccl as mnccl

    cfg = config_of(args)
    host_threads = host_threads_for_rank(world, numa)  # sized to the CPUs this rank can really use
    if world > 1:
        # several ranks share the host's CPU quota: the three pipeline threads of every rank sleep on blocking events instead
        # of spinning (measured on one rank: 8 threads 92 ms blocking vs 109 spinning per 400 k reads, 16 threads no difference),
        # and all of the rank's threads run the per-read tail
        os.environ.setdefault("MM_BLOCKING_WAIT", "1")
    if os.environ.get("BENCH_HOST_THREADS"):  # experiments: what one of N ranks gets on a host with few CPUs
        host_threads = max(1, int(os.environ["BENCH_HOST_THREADS"]))
    wl = setup_workload(args, cfg, rank, world, device)
    S, L, SEG, PI = wl["sketch"], cfg["read_len"], cfg["seg"], cfg["pi"]
    one_to_one = cfg["filt"] == "one-to-one"
    strong = cfg["scaling"] == "strong"

    # ---- index: built on the host by rank 0, uploaded; other ranks receive the device image with ONE NCCL broadcast ----
    comm = mnccl.create_with_torch(dist, rank, world, local_rank) if world > 1 else None  # the product's own communicator
    t_index = time.time()
    hi = hostlib.HostIndex.metadata_only(args.contigs, wl["contig_len"], K, SEG, S)  # contig names / lengths only: the index lives on the device
    bm = hostlib.BatchMapper(hi, pi=PI, device=local_rank, threads=host_threads, filter_mode=cfg["filt"])
    ctx = capi.Context.from_handle(bm.ctx_handle, S, device=local_rank)
    want_cpu = (not args.no_cpu_baseline) and world == 1
    cpu_real = want_cpu and args.cpu_kind != "port" and reference_library() is not None
    if want_cpu and args.cpu_kind == "reference" and not cpu_real:
        raise SystemExit("--cpu-kind reference: oracle/_ref/libmm_ref.so is not there (make -C oracle)")
    ref_session = None
    if cpu_real:  # the reference indexes the same contigs itself, from FASTA, while they are still at hand (not timed)
        ref_session, _ = real_reference_session(args, cfg, wl, S, usable_cpus())
        t_index = time.time()  # index_build_seconds is the product's side only
    want_port = want_cpu and not cpu_real
    ist = None
    if rank == 0:  # rank 0 builds the index on its GPU; the other ranks receive the image
        ist = build_index_on_device(args, cfg, wl, ctx, keep_lookup=want_port)
    host_index_arrays = ctx.index_download() if (rank == 0 and want_port) else None
    wl["ref_dev"] = None
    torch.cuda.empty_cache()
    if comm is not None:
        t0 = time.time()
        n = comm.index_broadcast(bm.ctx_handle, root=0)  # mm_index_broadcast (include/mashmap_b200_nccl.h)
        log(f"rank {rank}: index image {n / 1e9:.2f} GB received/sent in {time.time() - t0:.2f} s (includes waiting for rank 0's build)")
    index_seconds = time.time() - t_index

    # ---- the batch: pinned host copy (e2e) and device-resident copy (value) ----
    n_local = wl["hi"] - wl["lo"]
    ascii_reads = wl["queries"].reshape(-1).cpu().numpy()  # the queries as text (what the reference's path consumes)
    wl["queries"] = None
    torch.cuda.empty_cache()
    n_bases = n_local * L
    # e2e input: the pinned batch buffer of skch::BatchMapper, filled the way its FASTA reader fills it -- every read
    # packed to one nibble per base while it is copied in (outside the timed region, like parsing is)
    batch = bm.make_batch(n_local, L, first_seq_counter=wl["first_counter"])
    pack_seconds = batch.fill(ascii_reads, threads=host_threads)
    n_segs = len(batch.segments)
    # value input: the same reads resident in HBM as TEXT; the packing kernel (K0) is then part of every timed step
    seg_text = text_segments(batch, L)
    ctx.batch_upload(ascii_reads, seg_text)
    log(f"rank {rank}: batch resident ({n_local} queries, {n_segs} fragments), rss {rss_gb()} GB; host packing "
        f"{n_bases / max(pack_seconds, 1e-9) / 1e9:.1f} Gbases/s on {host_threads} threads")

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- value: resident inputs ----
    for _ in range(args.warmup):
        ctx.map_resident()
    sampler = ClockSampler(local_rank)
    sampler.start()
    time.sleep(0.3)
    barrier()
    t0 = time.time()
    launches0 = ctx.kernel_launches
    ev_ms, k_ms = 0.0, np.zeros(4)
    for _ in range(args.steps):
        nc, nl = ctx.map_resident()
        ms = ctx.stage_ms()
        ev_ms += ms[5]
        k_ms += np.array(ms[:3] + [ctx.pack_ms()])
    barrier()
    t1 = time.time()
    launches = ctx.kernel_launches - launches0
    clocks = sampler.stop(t0, t1)
    wall_ms = (t1 - t0) * 1e3
    seg_res, cands, loci = ctx.batch_fetch()
    diag = ctx.diag()
    log(f"rank {rank}: value phase done ({ev_ms / args.steps:.1f} ms/step), rare paths {diag}")

    # ---- e2e: host buffers -> C ABI -> records -> host tail -> (all-gather, one-to-one sweep) -> PAF text ----
    n_q_global = cfg["reads"] if strong else cfg["reads"] * world

    e2e_parts = {"map_s": 0.0, "records_s": 0.0, "allgather_s": 0.0, "one_to_one_s": 0.0}

    def e2e_step():
        ta = time.time()
        info = bm.map(batch)
        tb = time.time()
        e2e_parts["map_s"] += tb - ta
        gathered, final = 0, None
        if comm is not None or one_to_one:
            raw = bm.results_raw()
            tc = time.time()
            e2e_parts["records_s"] += tc - tb
            if comm is not None:  # all ranks' mapping records on every rank: mm_records_allgather (SURVEY 8(e))
                raw, counts = comm.records_allgather(raw)
                gathered = int(counts.sum())
            td = time.time()
            e2e_parts["allgather_s"] += td - tc
            if one_to_one and rank == 0:  # the run-wide reference-axis sweep + sort (computeMap.hpp:358-405) over ALL records
                kept, paf = bm.one_to_one(raw, n_q_global, L, copy=False)  # the text stays where the library wrote it
                final = (kept, len(paf))
            e2e_parts["one_to_one_s"] += time.time() - td
        return info, gathered, final

    for _ in range(min(args.warmup, 1)):
        e2e_step()
    for k_ in e2e_parts:
        e2e_parts[k_] = 0.0
    barrier()
    t0 = time.time()
    e2e_info, gathered, final = None, 0, None
    for _ in range(args.steps):
        e2e_info, gathered, final = e2e_step()
    barrier()
    e2e_ms = (time.time() - t0) * 1e3
    final_paf = bm.paf_final() if final is not None else None  # a copy of the last step's text, taken outside the timed region
    log(f"rank {rank}: e2e phase done ({e2e_ms / args.steps:.1f} ms/step), rss {rss_gb()} GB")
    h2d = batch.h2d_bytes + n_segs * capi.segment_dtype.itemsize
    d2h = n_segs * capi.segres_dtype.itemsize + len(cands) * capi.l1_dtype.itemsize + len(loci) * capi.l2_dtype.itemsize

    # ---- correctness of what was timed ----
    res = bm.results()
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, seg_res, cands, loci, res, wl["first_counter"], n_local)
    acc = _accuracy(res, wl["truth"], wl["contig_len"], wl["first_counter"], wl["lo"]) if wl["truth"] is not None else None
    sharded_check = None
    if strong and world > 1 and rank == 0 and one_to_one:
        # the same queries on this one GPU alone: the sharded run's final PAF must be the single-GPU PAF
        import hashlib

        full = bm.make_batch(cfg["reads"], L, first_seq_counter=0)
        full.fill(wl["all_queries"].reshape(-1).cpu().numpy(), threads=host_threads)
        bm.map(full)
        kept1, paf1 = bm.one_to_one(bm.results_raw(), cfg["reads"], L)
        full.close()
        sharded_check = {"paf_equal_to_single_gpu": bool(paf1 == final_paf), "mappings": int(final[0]), "single_gpu_mappings": int(kept1),
                         "paf_md5": hashlib.md5(final_paf).hexdigest()}
        bm.map(batch)  # results() below refer to this rank's own shard again

    # max over ranks
    times = torch.tensor([ev_ms, wall_ms, e2e_ms], dtype=torch.float64, device=device)
    if dist is not None:
        dist.all_reduce(times, op=dist.ReduceOp.MAX)
    ev_ms, wall_ms, e2e_ms = [float(x) for x in times.tolist()]
    total_bases = (cfg["reads"] * L if strong else n_bases * world) * args.steps

    if rank == 0:
        peak, peak_src = measured_peaks()
        b1 = SEG + 24 * S  # SURVEY 8(d): K1 algorithmic bytes per segment = L + 24 s
        k1_ms = k_ms[0] / args.steps
        achieved = b1 * n_segs / (k1_ms * 1e-3) / 1e9
        traffic = roofline_traffic()
        sm_count = torch.cuda.get_device_properties(local_rank).multi_processor_count
        out = {
            "metric": "mapped query Gbp/s", "value": total_bases / (ev_ms * 1e-3) / 1e9, "unit": "Gbp/s",
            "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ev_ms / args.steps,
            "higher_is_better": True, "scaling": cfg["scaling"], "vs_baseline": None, "dtype": "u64", "data": "synthetic",
            "config": {"workload": workload_text(args, cfg, S),
                       "segments_per_step": n_segs * world if not strong else int(cfg["reads"]) * (L // SEG + (1 if L % SEG else 0)),
                       "l2_policy": "inputs (reads + index) larger than L2, no flush",
                       "timing": "CUDA events on the launching stream, first kernel launch -> last kernel end, max over ranks",
                       "value_input": "reads resident in HBM as text (1 B/base); the packing kernel K0 runs inside every timed step",
                       "e2e_input": f"skch::BatchMapper's pinned batch buffer: one nibble per base, packed by the host reader at "
                                    f"ingest ({n_bases / max(pack_seconds, 1e-9) / 1e9:.1f} Gbases/s on {host_threads} threads, outside the timed region)",
                       "multi_gpu": (None if world == 1 else "one process per GPU; index image by ONE mm_index_broadcast (NCCL), reads "
                                     "sharded by rank, mapping records by mm_records_allgather every e2e step"
                                     + ("; run-wide one-to-one sweep + sort on rank 0" if one_to_one else "")),
                       "wall_ms_per_step": wall_ms / args.steps,
                       "index_build_seconds": index_seconds,  # contexts + pinned buffers + the build (index.build_s) + (with the CPU leg) the host copy of the index
                       "index": {"minmers": ist["n_minmers"], "keys": ist["n_keys"], "points": ist["n_points"], "built_on": "device (mm_index_build)",
                                 "build_s": ist["ms_total"] / 1e3, "window_scan_s": ist["ms_scan"] / 1e3, "records_s": ist["ms_post"] / 1e3, "lookup_s": ist["ms_lookup"] / 1e3,
                                 "chunks": ist["n_chunks"], "chunks_rescanned": ist["n_fixed_chunks"]},
                       "candidates": int(nc), "loci": int(nl), "host_threads": host_threads, "rare_paths": diag,
                       "mapped_read_fraction": None if acc is None else acc["mapped"],
                       "true_locus_fraction": None if acc is None else acc["correct"]},
            "clocks": clocks,
            "e2e": {"value": total_bases / (e2e_ms * 1e-3) / 1e9, "unit": "Gbp/s", "h2d_bytes_per_step": int(h2d),
                    "d2h_bytes_per_step": int(d2h), "ms_per_step": e2e_ms / args.steps,
                    "stage_seconds_last_step": {"device_call": e2e_info["sec_device"], "host_tail": e2e_info["sec_tail"]},
                    "paf_bytes_per_step": int(final[1] if final else e2e_info["paf_bytes"]), "records_gathered": int(gathered),
                    "rank0_seconds_per_step": {k_: v_ / args.steps for k_, v_ in e2e_parts.items()},
                    "efficiency_note": "e2e includes the all-gather" + (" and the run-wide one-to-one sweep" if one_to_one else "")},
            "gpu_launches": int(launches),
            "kernel_ms_per_step": {"pack": k_ms[3] / args.steps, "sketch": k_ms[0] / args.steps, "l1": k_ms[1] / args.steps,
                                   "l2": k_ms[2] / args.steps},
            "roofline": {"kernel": "k_sketch (K1)", "bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s",
                         "frac": achieved / peak,
                         "traffic": (traffic["k_sketch_dram_bytes_per_segment"] * n_segs if "k_sketch_dram_bytes_per_segment" in traffic else None),
                         "peak_source": peak_src, "algorithmic_bytes_per_segment": b1,
                         "instruction_roofline": _instruction_roofline(n_segs, SEG, k1_ms, clocks, sm_count),
                         "note": "bit-exact Murmur3 makes K1 INT-ALU bound (SURVEY 8(d)); see DESIGN.md for the instruction roofline"},
        }
        if world == 1:
            out["roofline"]["other_kernels"] = l1_l2_rooflines(ctx, seg_res, cands, loci, SEG, k_ms[1] / args.steps, k_ms[2] / args.steps, peak)
        if sharded_check is not None:
            out["sharded_check"] = sharded_check
        if want_cpu and cpu_real:
            # the unmodified reference on a bounded sample of the step, on all host threads; its mappings of those reads are
            # diffed against the product's (the timed result): parity against the reference itself at bench scale
            threads = usable_cpus()
            n_cpu = min(cpu_sample_reads(args, cfg, threads), n_local)
            cb, ref_rows = real_reference_step(ref_session, cfg, ascii_reads, n_cpu, threads, first_counter=wl["first_counter"], want_rows=True)
            ref_session.close()
            sel = (res[:, 0] - wl["first_counter"] < n_cpu) if len(res) else np.zeros(0, bool)
            d = _port_vs_reference(res[sel], ref_rows, cfg["seg"])
            out["parity"] = {"reads": int(n_cpu), "against": "the unmodified reference (oracle/_ref/libmm_ref.so, its own index)",
                             "stage": "per-read mappings (before the run-wide one-to-one sweep)" if one_to_one else "final mappings",
                             "mappings_gpu": d["mappings_port"], "mappings_reference": d["mappings_reference"],
                             "single_fragment_mappings_dropped_by_the_reference_uninitialised_n_merged":
                                 d["single_fragment_mappings_dropped_by_the_reference_uninitialised_n_merged"],
                             "mismatches": d["other_differences"], "max_identity_diff": d["max_identity_diff"]}
            out["cpu_baseline"] = cb
        elif want_cpu:
            cb = cpu_baseline(args, cfg, host_index_arrays, ascii_reads, S, gpu_rows=res, first_counter=wl["first_counter"])
            out["parity"] = cb.pop("parity")  # GPU mappings of the sampled reads == the CPU port's, at bench scale
            out["cpu_baseline"] = cb
        print(json.dumps(out), flush=True)
    if dist is not None:
        dist.barrier()
        if comm is not None:
            comm.close()
        dist.destroy_process_group()


DUMP_SEGMENTS = 65_536  # fragments sampled for --dump-outputs (of 2 M at the default size): ~14 MB of .npy in all
DUMP_READS = 32_768


def _ranges(first, count):
    """indices first[i] .. first[i] + count[i] - 1 of every i, concatenated, and the i each one belongs to"""
    count = count.astype(np.int64)
    owner = np.repeat(np.arange(len(count)), count)
    starts = np.repeat(first.astype(np.int64) - np.concatenate([[0], np.cumsum(count)[:-1]]), count)
    return starts + np.arange(int(count.sum())), owner


def dump_outputs(out_dir, seg_res, cands, loci, res, first_counter, n_reads):
    """What the last timed step handed its caller, as float64 .npy files that two builds can be compared on:
      segments.npy    value path (mm_map_resident), per sampled fragment: fragment index, sketch_max_hash >> 32,
                      sketch_max_hash & 0xffffffff, sketch_raw_count, sketch_size, n_points, minimum_hits, best_intersection,
                      n_candidates
      candidates.npy  the L1 candidates of those fragments in fragment order: fragment index, seqId, rangeStartPos, rangeEndPos,
                      intersectionSize, n_loci
      loci.npy        their L2 loci in the same order: fragment index, seqId, meanOptimalPos, optimalStart, optimalEnd,
                      sharedSketchSize, strand
      mappings.npy    e2e path (skch::BatchMapper): the mapping rows of a sample of the reads, as results() returns them
    The fragments' first_candidate / first_locus offsets are left out: they depend on the order the CTAs reserved their
    slices in, not on what was computed. The samples are drawn with a fixed seed from the fragment / read counts only."""
    os.makedirs(out_dir, exist_ok=True)
    rng = np.random.default_rng(12345)
    n = len(seg_res)
    pick = np.sort(rng.choice(n, min(n, DUMP_SEGMENTS), replace=False))
    sr = seg_res[pick]
    h = sr["sketch_max_hash"]
    np.save(os.path.join(out_dir, "segments.npy"), np.stack(
        [pick, h >> np.uint64(32), h & np.uint64(0xFFFFFFFF)] + [sr[f] for f in ("sketch_raw_count", "sketch_size", "n_points",
                                                                                  "minimum_hits", "best_intersection", "n_candidates")],
        axis=1).astype(np.float64))
    ci, owner = _ranges(sr["first_candidate"], sr["n_candidates"])
    c = cands[ci]
    np.save(os.path.join(out_dir, "candidates.npy"), np.stack(
        [pick[owner]] + [c[f] for f in ("seqId", "rangeStartPos", "rangeEndPos", "intersectionSize", "n_loci")], axis=1).astype(np.float64))
    li, lowner = _ranges(c["first_locus"], c["n_loci"])
    lc = loci[li]
    np.save(os.path.join(out_dir, "loci.npy"), np.stack(
        [pick[owner[lowner]]] + [lc[f] for f in ("seqId", "meanOptimalPos", "optimalStart", "optimalEnd", "sharedSketchSize", "strand")],
        axis=1).astype(np.float64))
    keep = np.sort(rng.choice(n_reads, min(n_reads, DUMP_READS), replace=False)) + first_counter
    np.save(os.path.join(out_dir, "mappings.npy"), res[np.isin(res[:, 0], keep)].astype(np.float64))
    log(f"outputs of the last step written to {out_dir}: {len(pick)} fragments, {len(c)} candidates, {len(lc)} loci, "
        f"mappings of {len(keep)} reads")


def algorithmic_bytes_l1_l2(seg_res, cands, loci, idx_seq, idx_wpos, seg_len):
    """SURVEY 8(d)'s algorithmic bytes of the L1 and L2 stages for one step, counted on the step's own records:
      B2 = 32 s_q (table probes) + 24 m (interval points) + 16 c (candidates out)           summed over the fragments
      B3 = 24 n_scan + 24 s_q + 24 c_out                                                     summed over the L1 candidates
    m = interval points of a fragment (segment result), c = its candidates, c_out = loci of a candidate, and n_scan = the
    minmerIndex entries between lower_bound((seqId, rangeStart - L - 1)) and the last entry with wpos <= rangeEnd
    (computeMap.hpp:1290-1340), counted against the index records themselves (idx_seq / idx_wpos, sorted by (seqId, wpos))."""
    s_q = seg_res["sketch_size"].astype(np.int64)
    b2 = 32 * int(s_q.sum()) + 24 * int(seg_res["n_points"].astype(np.int64).sum()) + 16 * int(len(cands))
    key = (idx_seq.astype(np.uint64) << np.uint64(32)) | idx_wpos.astype(np.uint32).astype(np.uint64)
    cseq = cands["seqId"].astype(np.uint64) << np.uint64(32)
    lo = np.maximum(cands["rangeStartPos"].astype(np.int64) - seg_len - 1, 0).astype(np.uint64)
    hi = np.maximum(cands["rangeEndPos"].astype(np.int64), 0).astype(np.uint64)
    first = np.searchsorted(key, cseq | lo, side="left")
    last = np.searchsorted(key, cseq | hi, side="right")
    n_scan = int(np.maximum(last.astype(np.int64) - first.astype(np.int64), 0).sum())
    b3 = 24 * n_scan + 24 * int(s_q[cands["segment"]].sum()) + 24 * int(len(loci))
    return {"B2_bytes": b2, "B3_bytes": b3, "interval_points": int(seg_res["n_points"].astype(np.int64).sum()), "candidates": int(len(cands)),
            "index_entries_scanned": n_scan, "loci": int(len(loci))}


def l1_l2_rooflines(ctx, seg_res, cands, loci, seg_len, k2_ms, k3_ms, peak):
    """roofline entries of K2 and K3 (VERDICT r1 weak 4): algorithmic bytes counted on the real configuration / stage time.
    Needs a host copy of the index records (6 GB at 3 Gbp, a few seconds, outside every timed region); any failure only
    drops the entries."""
    try:
        t0 = time.time()
        mi = ctx.index_minmers()
        counts = algorithmic_bytes_l1_l2(seg_res, cands, loci, mi["seqId"], mi["wpos"], seg_len)
        del mi
        n = max(1, len(seg_res))
        out = {}
        for name, b, ms in (("K2 (k_l1_probe + k_l1_warp + k_l1_cta)", counts["B2_bytes"], k2_ms), ("K3 (k_l2_ranges + k_l2_prep + k_l2_scan)", counts["B3_bytes"], k3_ms)):
            ach = b / (ms * 1e-3) / 1e9
            out[name] = {"bound": "hbm", "achieved": ach, "peak": peak, "unit": "GB/s", "frac": ach / peak, "algorithmic_bytes_per_segment": b / n}
        out["counts_per_step"] = counts
        out["counted_in_seconds"] = round(time.time() - t0, 1)
        return json.loads(json.dumps(out))  # plain Python numbers only: the JSON line must never fail on this extra
    except Exception as e:  # never fatal: the contract's roofline is K1's
        log(f"K2 / K3 roofline entries skipped: {type(e).__name__}: {e}")
        return None


def _instruction_roofline(n_segs, seg, k1_ms, clocks, sm_count):
    """K1 is bound by instruction issue, not by HBM: every k-mer position costs two bit-exact MurmurHash3_x64_128
    evaluations. Peak = the MEASURED rate at which this GPU runs that hash alone (mashmap_b200/mm_issue_peak: mm_hash.h's
    own device code on register-resident data, every lane busy, no memory, no selection; profiles/issue_peak.json), two
    hashes per position. What K1 loses against it is everything that is not hashing."""
    positions = n_segs * (seg - K + 1)
    achieved = positions / (k1_ms * 1e-3) / 1e9
    mhz = (clocks or {}).get("sm_mhz") or 1965.0
    ip = issue_peak() or {}
    per_clk = ip.get("hash19_per_clk_per_sm")
    if per_clk:
        peak = per_clk * sm_count * mhz * 1e6 * 32 / 2 / 1e9
        src = "measured: standalone Murmur3 (k=19) rate of mm_hash.h on this GPU (profiles/issue_peak.json), 2 hashes per position"
    else:  # no measurement committed: one instruction per clock per scheduler over the loop's SASS instruction count
        peak = sm_count * 4.0 * mhz * 1e6 * 32 / K1_INSTR_PER_POSITION / 1e9
        src = "nominal 1 instruction / clock / scheduler (no measurement committed)"
    return {"unit": "G k-mer positions/s", "achieved": achieved, "peak": peak, "frac": achieved / peak, "peak_source": src,
            "loop_instructions_per_position": K1_INSTR_PER_POSITION,
            "measured_issue_rates_per_sm_clk": {k: v for k, v in ip.items() if isinstance(v, float) and not k.startswith("hash19")} or None}


K1_INSTR_PER_POSITION = 170  # executed SASS instructions per k-mer position in k_sketch's loop (DESIGN.md section 3, scripts/sass_loops.py)


def _accuracy(res, truth, contig_len, first_counter, lo):
    contig_of, start_of, strand_of = truth
    if len(res) == 0:
        return {"mapped": 0.0, "correct": 0.0}
    q = res[:, 0] - first_counter + lo
    ok = (res[:, 3] == contig_of[q]) & (np.abs(res[:, 4].astype(np.int64) - start_of[q]) < 20_000) & (res[:, 6] == strand_of[q])
    mapped = len(np.unique(q)) / max(1, len(np.unique(np.arange(lo, lo + (res[:, 0].max() - first_counter + 1)))))
    return {"mapped": float(min(1.0, mapped)), "correct": float(ok.mean())}


def _parity_diff(cpu_rows, gpu_rows):
    """full-scale parity of what was timed: the mappings of the sampled reads from the CPU port of the reference path against
    the GPU product's (rows: query id, query start/end, ref id, ref start/end, strand, conserved sketches, block length,
    identity * 1e6). Coordinates / strand / counts exact, identity within 1e-4 (north_star)."""
    def order(r):
        return r[np.lexsort(tuple(r[:, c] for c in range(8, -1, -1)))] if len(r) else r

    a, b = order(cpu_rows), order(gpu_rows)
    out = {"mappings_cpu": int(len(a)), "mappings_gpu": int(len(b))}
    if len(a) == len(b) and np.array_equal(a[:, :9], b[:, :9]):
        d = np.abs(a[:, 9].astype(np.int64) - b[:, 9]) if len(a) else np.zeros(0, np.int64)
        out["mismatches"] = int((d > 100).sum())
        out["max_identity_diff"] = float(d.max() / 1e6) if len(d) else 0.0
    else:  # count rows (exact integer columns) present on one side only
        ka = {tuple(x) for x in a[:, :9].tolist()}
        kb = {tuple(x) for x in b[:, :9].tolist()}
        out["mismatches"] = len(ka ^ kb) + abs(len(a) - len(ka)) + abs(len(b) - len(kb))
        out["examples"] = [list(map(int, x)) for x in list(ka ^ kb)[:4]]
    return out


def _port_vs_reference(port_rows, ref_rows, seg):
    """the oracle port's mappings of a sample against the unmodified reference's. One known difference is classified, not
    hidden: a split read whose only mapping is a single fragment reaches filterWeakMappings with MappingResult::n_merged never
    written (computeMap.hpp:1227 / :429-430, undefined behaviour: the reference drops or keeps it depending on stack garbage);
    the port and the product define n_merged = 1 there and keep it (DESIGN.md section 4)."""
    def keyset(r):
        return {tuple(x) for x in r[:, :9].tolist()}

    a, b = keyset(port_rows), keyset(ref_rows)
    only_port, only_ref = a - b, b - a
    per_read = {}
    for x in port_rows[:, 0].tolist():
        per_read[x] = per_read.get(x, 0) + 1
    ub = {x for x in only_port if x[8] == seg and per_read.get(x[0], 0) == 1}
    ident = 0.0
    if len(port_rows) and len(ref_rows):
        common = {tuple(x[:9]): x[9] for x in ref_rows.tolist()}
        d = [abs(x[9] - common[tuple(x[:9])]) for x in port_rows.tolist() if tuple(x[:9]) in common]
        ident = max(d) / 1e6 if d else 0.0
    return {"mappings_port": int(len(port_rows)), "mappings_reference": int(len(ref_rows)),
            "single_fragment_mappings_dropped_by_the_reference_uninitialised_n_merged": len(ub),
            "other_differences": len(only_port - ub) + len(only_ref), "max_identity_diff": ident}


def cpu_sample_reads(args, cfg, threads):
    """queries per CPU sample: about 15 s of wall time (the port maps ~11 Mbp per second per CPU on configs[1]), at least one
    query per thread, at most the whole step"""
    if args.cpu_sample_reads:
        return min(cfg["reads"], args.cpu_sample_reads)
    want_bases = 170_000_000 * threads
    return int(min(cfg["reads"], max(threads, want_bases // cfg["read_len"])))


def cpu_baseline(args, cfg, index_arrays, ascii_reads, S, threads=None, n_reads=None, gpu_rows=None, first_counter=0, want_rows=False):
    """The oracle port of the reference path (oracle/libmm_oracle.so, mapModule per read, one task per read on
    all host threads) on a bounded sample of the same batch, with the same index content. With gpu_rows (the
    product's mappings of the whole batch) the port's mappings of the sampled reads are diffed against them."""
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import oracle_py

    threads = threads or usable_cpus()
    L = cfg["read_len"]
    mi, keys, offs, pts, fr = index_arrays  # host copies of the index the GPU arm maps against
    O = oracle_py.Oracle(K, cfg["seg"], S, cfg["pi"], filterMode={"map": 1, "one-to-one": 2, "none": 3}[cfg["filt"]])
    O.set_index(mi, keys, offs, pts, fr, np.full(args.contigs, args.ref_bp // args.contigs, dtype=np.int32))
    lib = oracle_py.lib()
    import ctypes as C

    lib.orc_map_reads_mt.restype = C.c_int64
    lib.orc_map_reads_mt.argtypes = [C.c_void_p, C.c_void_p, C.c_int64, C.c_int, C.c_int, C.c_int, C.POINTER(C.c_int64),
                                     C.c_void_p, C.c_int64]
    mapped = C.c_int64()
    n_reads = n_reads or cpu_sample_reads(args, cfg, threads)
    n_reads = min(n_reads, len(ascii_reads) // L)
    rows = np.zeros((64 * n_reads + 4096, 10), dtype=np.int32) if gpu_rows is not None else None
    t0 = time.time()
    c0 = os.times()
    n_map = lib.orc_map_reads_mt(O.h, ascii_reads.ctypes.data, n_reads, L, first_counter, threads, C.byref(mapped),
                                 rows.ctypes.data if rows is not None else None, len(rows) if rows is not None else 0)
    dt = time.time() - t0
    c1 = os.times()
    O.close()
    busy = ((c1.user - c0.user) + (c1.system - c0.system)) / max(dt, 1e-9)  # CPUs actually kept busy by the threads
    parity = None
    if gpu_rows is not None:
        sel = (gpu_rows[:, 0] - first_counter < n_reads) if len(gpu_rows) else np.zeros(0, bool)
        parity = {"reads": int(n_reads), "stage": "per-read mappings (before the run-wide one-to-one sweep)" if cfg["filt"] == "one-to-one" else "final mappings",
                  **_parity_diff(rows[: min(n_map, len(rows))], gpu_rows[sel])}
    return {**({"rows": rows[: min(n_map, len(rows))]} if want_rows else {}),
            "parity": parity, "value": n_reads * L / dt / 1e9, "unit": "Gbp/s", "cores": threads, "kind": "port",
            "cpus_busy": round(busy, 1), "host": host_cpu_info(),
            "note": "the port is a plain restatement kept for checking, slower than the program it restates: the unmodified reference "
                    "itself is timed by `bench.py --impl reference` (kind \"reference\")",
            "sample": f"first {n_reads} queries of the step ({n_reads * L / 1e6:.0f} Mbp), oracle/libmm_oracle.so mapModule per query "
                      f"on {threads} threads, {dt:.1f} s; {mapped.value} queries mapped, {n_map} mappings"}


def reference_library():
    """oracle/_ref/libmm_ref.so (the unmodified reference behind oracle/ref_harness.cpp), or None"""
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    try:
        import refh

        return refh if refh.available() else None
    except Exception:  # noqa: BLE001
        return None


def real_reference_session(args, cfg, wl, S, threads):
    """The reference's own Sketch + Map on the bench's reference: the contigs are written as FASTA, the reference parses
    them and builds its index itself (winSketch.hpp), exactly as `mashmap -r ref.fa` would. Returns (session, seconds)."""
    import shutil
    import tempfile

    import refh

    wd = tempfile.mkdtemp(prefix="mm_ref_arm_")
    path = os.path.join(wd, "ref.fa")
    t0 = time.time()
    ref = wl["ref_dev"].cpu().numpy()
    with open(path, "wb", buffering=1 << 24) as f:
        for i in range(ref.shape[0]):
            f.write(b">c%d\n" % i)
            f.write(ref[i].tobytes())
            f.write(b"\n")
    del ref
    t_fa = time.time() - t0
    t0 = time.time()
    try:
        R = refh.RefSession(["-r", path, "-q", path, "-s", str(cfg["seg"]), "--pi", f"{cfg['pi'] * 100:g}", "-J", str(S), "-t", str(threads),
                             "-f", cfg["filt"], "-k", str(K)])
    finally:
        shutil.rmtree(wd, ignore_errors=True)
    t_ix = time.time() - t0
    log(f"reference arm: FASTA written in {t_fa:.1f} s, the reference's own index built in {t_ix:.1f} s ({threads} threads)")
    return R, t_fa + t_ix


def real_reference_step(R, cfg, ascii_reads, n_reads, threads, first_counter=0, want_rows=False):
    """one bounded sample through the reference's own mapModule (oracle/ref_harness.cpp: refh_map_reads_mt)"""
    import ctypes as C

    import refh

    lib = refh.lib()
    lib.refh_map_reads_mt.restype = C.c_int64
    lib.refh_map_reads_mt.argtypes = [C.c_void_p, C.c_void_p, C.c_int64, C.c_int, C.c_int, C.c_int, C.POINTER(C.c_int64), C.c_void_p, C.c_int64]
    L = cfg["read_len"]
    mapped = C.c_int64()
    rows = np.zeros((64 * n_reads + 4096, 10), dtype=np.int32) if want_rows else None
    t0 = time.time()
    c0 = os.times()
    n_map = lib.refh_map_reads_mt(R.h, ascii_reads.ctypes.data, n_reads, L, first_counter, threads, C.byref(mapped),
                                  rows.ctypes.data if rows is not None else None, len(rows) if rows is not None else 0)
    dt = time.time() - t0
    c1 = os.times()
    busy = ((c1.user - c0.user) + (c1.system - c0.system)) / max(dt, 1e-9)
    out = {"value": n_reads * L / dt / 1e9, "unit": "Gbp/s", "cores": threads, "kind": "reference", "cpus_busy": round(busy, 1), "host": host_cpu_info(),
           "sample": f"first {n_reads} queries of the step ({n_reads * L / 1e6:.0f} Mbp), oracle/_ref/libmm_ref.so (the unmodified reference): "
                     f"skch::Map::mapModule per query on {threads} threads, {dt:.1f} s; {mapped.value} queries mapped, {n_map} mappings"}
    return out, (rows[: min(n_map, len(rows))] if rows is not None else None)


def cpu_arm(args):
    """--impl reference: the reference's CPU path on the host cores, every step a bounded sample of the arm's workload.
    kind "reference": the unmodified reference (oracle/_ref/libmm_ref.so) builds its own index from the FASTA of the bench's
    reference (set-up, minutes at 3 Gbp, not timed) and maps each sample with its own mapModule on all host threads; the
    oracle port runs the same sample once beside it (port_value, and the two sets of mappings are diffed).
    kind "port" (--ref-kind port, or no library): the oracle port on the index content the product built."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    import torch

    device = torch.device("cuda:0") if torch.cuda.is_available() else torch.device("cpu")
    threads = usable_cpus()
    cfg = config_of(args)
    sample = cpu_sample_reads(args, cfg, threads)
    if cfg["kind"] == "reads":
        cfg["reads"] = sample  # only the sample is generated
    wl = setup_workload(args, cfg, 0, 1, device)
    S = wl["sketch"]
    real = args.ref_kind != "port" and reference_library() is not None
    if args.ref_kind == "real" and not real:
        raise SystemExit("--ref-kind real: oracle/_ref/libmm_ref.so is not there (make -C oracle)")
    ascii_reads = np.ascontiguousarray(wl["queries"].reshape(-1).cpu().numpy())
    R, setup_s, extra = None, None, {}
    if real:
        R, setup_s = real_reference_session(args, cfg, wl, S, threads)
    if not real or cfg["kind"] == "reads":  # the port: the arm itself, or one sample beside the real reference
        if device.type == "cuda":  # the index content is the same either way (tests/test_gpu_index_build.py); the GPU builds it in seconds
            from mashmap_b200 import capi

            ctx = capi.Context(device=0, kmer_size=K, seg_length=cfg["seg"], sketch_size=S)
            build_index_on_device(args, cfg, wl, ctx, keep_lookup=True)
            arrays = ctx.index_download()
            ctx.close()
        else:
            arrays = build_index_on_host(args, cfg, wl, threads).arrays()
    wl["ref_dev"] = None
    times, last = [], None
    for i in range(args.warmup + args.steps):
        if real:
            last, _ = real_reference_step(R, cfg, ascii_reads, sample, threads)
        else:
            last = cpu_baseline(args, cfg, arrays, ascii_reads, S, threads=threads, n_reads=sample)
            last.pop("parity", None)
        if i >= args.warmup:
            times.append(sample * cfg["read_len"] / last["value"] / 1e9)
    if real and cfg["kind"] == "reads":  # the port on the same sample: speed beside the reference's, and the mappings diffed
        _, ref_rows = real_reference_step(R, cfg, ascii_reads, sample, threads, want_rows=True)
        port = cpu_baseline(args, cfg, arrays, ascii_reads, S, threads=threads, n_reads=sample, gpu_rows=ref_rows, want_rows=True)
        extra = {"port_value": port["value"], "port_vs_reference": _port_vs_reference(port.pop("rows"), ref_rows, cfg["seg"]), "setup_seconds": round(setup_s, 1)}
    if R is not None:
        R.close()
    dt = sum(times)
    val = sample * cfg["read_len"] * args.steps / dt / 1e9
    last["value"] = val
    last.update(extra)
    print(json.dumps({
        "impl": "reference", "metric": "mapped query Gbp/s", "value": val, "unit": "Gbp/s", "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": dt / args.steps * 1e3, "higher_is_better": True, "scaling": cfg["scaling"],
        "vs_baseline": None, "dtype": "u64", "data": "synthetic",
        "config": {"workload": f"bounded sample ({sample} queries per step) of: " + workload_text(args, config_of(args), S)},
        "cpu_baseline": last,
        "e2e": {"value": val, "unit": "Gbp/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }), flush=True)


if __name__ == "__main__":
    a = parse_args()
    if a.impl == "reference":
        cpu_arm(a)
    else:
        gpu_arm(a)
