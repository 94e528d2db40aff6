#!/usr/bin/env python
"""bench.py — POA windows/s (BASELINE.json metric) on B200, one process per GPU.

  python bench.py [--config 2|3|4|5] [--gpus N] [--steps K] [--warmup W]   our arm (sm_100a kernels via the C ABI)
  python bench.py --impl reference [--config ...] ...                      the reference's own CPU path (oracle/_ref)
  python bench.py ... --dump-outputs DIR     also write what the timed path returned in its last step (see dump_outputs)
  torchrun --nnodes=1 --nproc-per-node N ... bench.py --gpus N             one rank per GPU

Workloads (BASELINE.json `configs`; the default is config 2, the one the metric is quoted on at one GPU):
  2  synthetic 10k windows per GPU, w=500, 32 layers, 12 % ONT-like error, 3/-5/-4, full matrix   (weak scaling)
  3  synthetic 100k windows IN TOTAL, same shape, racon -b (banded), one stream cut into contiguous cost-balanced
     ranges, one per rank (SURVEY.md §8e)                                                          (strong scaling)
  4  Illumina mode: w=200, 60 pieces of 150-base reads per window (partial-span => Subgraph path), qualities, kNGS;
     50k windows per GPU                                                                           (weak scaling)
  5  fragment correction (-f): 10-kb reads against themselves: batched pre-alignment (rp_aln_*, edlib-identical) ->
     breaking points -> w=500 windows -> consensus; reports windows/s of the consensus stage and, under "aligner",
     pairs/s and GCUPS of the pre-alignment kernel                                                 (weak scaling)

A "step" = one pass of the hot path over the rank's batch.
  value      : windows/s with the batch resident in HBM (kernel launches only), CUDA-event timed, max over ranks
  e2e        : windows/s through the whole plugin call with HOST buffers: add windows (-> pinned staging), rp_poa_run
               (H2D + kernel + D2H), rp_poa_fetch_all; at N > 1 plus the NCCL gather of the consensus
  roofline   : algorithmic bytes (SURVEY.md §8d: 2 B x sum (L+1)[(N+1)+E], counted by the kernel's own device counters
               in a separate untimed launch) / isolated kernel time, against the measured HBM peak
  cpu_baseline: the unmodified reference (oracle/_ref) on the host cores, bounded sample (rank 0); its `gpu_reference`
               is the reference's own CUDA path (GenomeWorks cudapoa, unmodified) on the SAME number of GPUs
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

CONFIGS = {
    2: dict(workload="synthetic 10k windows, w=500, 32x ONT-error reads (12%), m/x/g=3/-5/-4, seed 42",
            metric="500-bp POA windows/sec at 32x coverage", banded=False, windows=10000, scaling="weak", wl=500,
            shape="ont"),
    3: dict(workload="synthetic 100k windows in total, w=500, 32x ONT-error reads (12%), m/x/g=3/-5/-4, seed 42, "
                     "--cuda-banded-alignment (-b), cost-balanced contiguous ranges per rank",
            metric="500-bp POA windows/sec at 32x coverage", banded=True, windows=100000, scaling="strong", wl=500,
            shape="ont"),
    4: dict(workload="Illumina mode: w=200, 60 pieces of 150-base reads per window (0.5% substitutions, Phred 30-40, "
                     "all partial-span), kNGS, m/x/g=3/-5/-4; 50k windows per GPU",
            metric="200-bp POA windows/sec at 60x short-read coverage", banded=False, windows=50000, scaling="weak",
            wl=200, shape="ngs"),
    5: dict(workload="fragment correction (-f): synthetic 10-kb reads (12% error) overlapped with themselves, "
                     "device pre-alignment + breaking points -> w=500 windows -> consensus",
            metric="500-bp POA windows/sec, fragment correction", banded=False, windows=0, scaling="weak", wl=500,
            shape="frag"),
}


def env_int(name, default):
    try:
        return int(os.environ.get(name, default))
    except ValueError:
        return default


def host_cores():
    try:
        return len(os.sched_getaffinity(0))
    except AttributeError:
        return os.cpu_count() or 1


def measured_hbm_peak():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    try:
        with open(path) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md)"


def ncu_traffic(cfg_id):
    """Per-launch DRAM bytes of the POA kernel from the committed ncu --set full capture of this config, if any."""
    path = os.path.join(ROOT, "profiles", "traffic.json")
    try:
        with open(path) as f:
            t = json.load(f)
        return t.get("config%d" % cfg_id, t if cfg_id == 2 else None)
    except Exception:
        return None


class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md recipe)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.gpu = gpu_index
        self.proc = None
        self.lines = []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.gpu), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "100"],
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
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1]))
                mx.append(float(f[2]))
            except ValueError:
                continue
            for name, val in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


# ---------------------------------------------------------------------------------------------------------------
# workloads
# ---------------------------------------------------------------------------------------------------------------
def make_windows(cfg_id, args, rank, world, sample=None):
    """The window set of this rank for a step (and, for config 5, the overlaps the windows come from)."""
    from racon_b200 import shard, windows
    cfg = CONFIGS[cfg_id]
    n = args.windows or cfg["windows"]
    if cfg["shape"] == "ont" and cfg["scaling"] == "weak":
        if sample is not None:
            n = min(n, sample)
        state = 42
        for _ in range(rank):  # every rank draws ITS OWN stretch of the generator's stream
            _, state = windows.synth_windows(n, err=0.12, state=state)
        ws, _ = windows.synth_windows(n, err=0.12, state=state)
        return ws, {"windows_total": n * world}
    if cfg["shape"] == "ont":  # one stream for everybody, contiguous cost-balanced ranges (SURVEY.md §8e)
        if sample is not None:
            ws, _ = windows.synth_windows(min(n, sample), err=0.12, state=42)
            return ws, {"windows_total": n}
        full, _ = windows.synth_windows(n, err=0.12, state=42)
        lo, hi = shard.shard_bounds_by_cost(windows.window_costs(full), rank, world)
        return windows.slice_windows(full, lo, hi), {"windows_total": n, "range": [lo, hi]}
    if cfg["shape"] == "ngs":
        if sample is not None:
            n = min(n, sample)
        ws, _ = windows.synth_ngs_windows(n, state=4242 + 1000003 * rank)
        return ws, {"windows_total": n * world}
    raise SystemExit("bench.py: config %d has its own driver" % cfg_id)


def config_key(cfg, args, banded=None):
    """`config` of the JSON line: names the workload and nothing else, identical in both arms (`--impl reference` included) so
    that the driver compares like with like; what THIS run did beyond that (window counts, batch objects, host binding,
    checksums ...) goes into the line's `run` object."""
    return {"workload": cfg["workload"], "baseline_config": args.config,
            "l2": "GPU arm: a step's inputs (hundreds of MB) + DP scratch (tens of GB) exceed the 126 MB L2, no explicit flush; "
                  "reference arm: host cores, bounded sample of the same windows"}


def run_reference(args, rank, world):
    """The reference's own CPU implementation (Window::generate_consensus over spoa, compiled unmodified into
    oracle/_ref) on all host threads.  Each step = a bounded sample of the same workload."""
    if rank != 0:
        return
    from oracle import bindings as ob
    cfg = CONFIGS[args.config]
    cores = host_cores()
    if not ob.have_ref():
        print(json.dumps({"impl": "reference", "unavailable": "oracle/_ref/libracon_ref.so not built"}))
        return
    if cfg["shape"] == "frag":
        ws = frag_workload(args, 0, sample_reads=min(24, args.frag_reads))["windows"]
    else:
        ws, _ = make_windows(args.config, args, 0, 1, sample=(200 if cfg["shape"] == "ont" else 1500) * cores)
    n_sample = ws.n_windows
    # the reference scales poorly past the physical cores (allocator contention in spoa::Graph): give it the
    # better of "all hardware threads" and "half of them", decided on an untimed probe
    threads = cores
    from racon_b200 import windows
    if cores >= 4:
        probe = windows.slice_windows(ws, 0, min(n_sample, 16 * cores))
        t_all = ob.ref_consensus(probe, threads=cores)[2]
        t_half = ob.ref_consensus(probe, threads=cores // 2)[2]
        threads = cores if t_all <= t_half else cores // 2
    for _ in range(args.warmup):
        ob.ref_consensus(ws, threads=threads)
    t0 = time.perf_counter()
    secs = 0.0
    for _ in range(args.steps):
        _, _, s = ob.ref_consensus(ws, threads=threads)
        secs += s
    wall = time.perf_counter() - t0
    value = n_sample * args.steps / secs
    sample = "%d of the workload's windows per step, %d host threads (of %d hardware threads; best of all/half), " \
             "consensus loop only" % (n_sample, threads, cores)
    line = {
        "impl": "reference", "metric": cfg["metric"], "value": value, "unit": "windows/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * secs / args.steps,
        "higher_is_better": True, "scaling": cfg["scaling"], "vs_baseline": None, "dtype": "int16", "data": "synthetic",
        "config": config_key(cfg, args), "run": {"sample": sample, "wall_s": wall},
        "cpu_baseline": {"value": value, "unit": "windows/s", "cores": threads, "kind": "reference", "sample": sample},
        "e2e": {"value": value, "unit": "windows/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line))


# ---------------------------------------------------------------------------------------------------------------
# config 5: fragment correction — synthetic reads, overlaps, device pre-alignment, windows
# ---------------------------------------------------------------------------------------------------------------
def frag_workload(args, rank, sample_reads=None):
    """Synthetic -f input: `frag_reads` reads of ~10 kb drawn from a random genome at ~30x (12 % error, forward strand),
    every pair of reads whose genome intervals share >= 2 kb is an overlap (both directions: dual PAF), overlap
    coordinates derived from the true genome coordinates like a mapper would report them.  Returns the sequences, the
    overlap table and — built by the device pre-alignment + breaking points + racon's window assembly (host mirror of
    polisher.cpp:383-461) — the window set."""
    import numpy as np
    from racon_b200 import api
    from tests import util  # mutate(): the numpy window maker's error model
    n_reads = sample_reads or args.frag_reads
    rlen = args.frag_read_len
    rng = np.random.default_rng(777 + rank)
    cov = 30
    glen = max(rlen * 2, n_reads * rlen // cov)
    genome = bytes(b"ACGT"[i] for i in rng.integers(4, size=glen))
    starts = np.sort(rng.integers(0, glen - rlen, size=n_reads))
    reads, spans = [], []
    for s in starts:
        r = util.mutate(rng, genome[s:s + rlen], 0.12)
        reads.append(r)
        spans.append((int(s), int(s) + rlen))
    seq_off = np.zeros(n_reads + 1, np.uint64)
    seq_off[1:] = np.cumsum([len(r) for r in reads])
    bases = np.frombuffer(b"".join(reads), np.uint8).copy()
    quals = np.full(bases.size, ord("5"), np.uint8)
    ov = []
    for i in range(n_reads):
        for j in range(i + 1, n_reads):
            if spans[j][0] >= spans[i][1]:
                break
            lo, hi = max(spans[i][0], spans[j][0]), min(spans[i][1], spans[j][1])
            if hi - lo < 2000:
                continue

            def coords(k):
                a = int((lo - spans[k][0]) * len(reads[k]) / rlen)
                b = int((hi - spans[k][0]) * len(reads[k]) / rlen)
                return a, min(b, len(reads[k]))
            qi, qj = coords(i), coords(j)
            # overlap row: q_id, t_id, strand, q_begin, q_end, q_length, t_begin, t_end, t_length
            ov.append((i, j, 0, qi[0], qi[1], len(reads[i]), qj[0], qj[1], len(reads[j])))
            ov.append((j, i, 0, qj[0], qj[1], len(reads[j]), qi[0], qi[1], len(reads[i])))
    ov = np.asarray(ov, np.uint32).reshape(-1, 9)
    t0 = time.perf_counter()
    pol = api.MirrorPolisher(bases.tobytes(), quals.tobytes(), seq_off, np.zeros(n_reads, np.uint8), n_reads, ov,
                             window_length=500, fragment_correction=True)
    init_s = time.perf_counter() - t0
    ex = pol.export()
    pol.close()
    from racon_b200 import windows
    ws = windows.WindowSet(bases=ex["bases"], quals=None, seq_off=ex["seq_off"], seq_has_qual=None,
                           seq_begin=ex["seq_begin"], seq_end=ex["seq_end"], win_first=ex["win_first"],
                           win_type=ex["win_type"])
    pairs = [(bytes(bases[int(seq_off[o[0]]) + int(o[3]):int(seq_off[o[0]]) + int(o[4])]),
              bytes(bases[int(seq_off[o[1]]) + int(o[6]):int(seq_off[o[1]]) + int(o[7])])) for o in ov]
    return {"windows": ws, "pairs": pairs, "reads": n_reads, "overlaps": len(ov), "init_s": init_s}


def time_aligner(pairs, local, steps, warmup):
    """rp_aln_* over the overlaps' spans, resident: CUDA events around rp_aln_launch."""
    import torch
    from racon_b200 import api
    b = api.AlnBatch(device=local)
    st = torch.cuda.current_stream()
    b.set_stream(st.cuda_stream)
    taken = 0
    for q, t in pairs:
        if not b.add(q, t):
            break
        taken += 1
    cells = float(sum(len(q) * len(t) for q, t in pairs[:taken]))
    b.upload()
    for _ in range(max(1, warmup)):
        b.launch()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(st)
    for _ in range(steps):
        b.launch()
    e1.record(st)
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / steps
    b.download()
    b.sync()
    results = [b.fetch(k) for k in range(taken)]
    bad = sum(1 for r in results if r[2] != 0)
    b.close()
    return results, {"pairs": taken, "pairs_per_s": taken / (ms * 1e-3), "gcups_full_matrix_equivalent": cells / (ms * 1e-3) / 1e9,
            "ms_per_launch": ms, "soft_failures": bad, "kernel": "rp_aln_kernel",
            "bound": "integer issue (bit-vector words in registers; HBM sees only sequences and the stored leaf words)"}


# ---------------------------------------------------------------------------------------------------------------
DUMP_CONSENSUS_BYTES = 46 << 20   # consensus rows; with the aligner's sample and the per-item arrays a dump stays < 64 MB
DUMP_ALIGNER_PAIRS = 300          # config 5: CIGARs of at most this many overlaps (~10 kb spans: < 12 MB as float32)


def dump_outputs(path, out, lens, pol, st):
    """--dump-outputs: what the last timed end-to-end step handed back to its caller (rp_poa_fetch_all of every batch
    object: consensus bytes, their lengths, the polished flags, the window statuses) as DIR/<name>.npy, so that two builds
    run with the same arguments (hence the same seeded windows) can be compared output for output.  Consensus rows are the
    bytes' codes as float32, zero past each window's length.  When the consensus rows would exceed DUMP_CONSENSUS_BYTES, a
    fixed seeded sample of windows is written; window_index.npy lists the windows written either way.  The windows are
    rank 0's; the by-reference leg (e2e.by_reference) computes the same consensus and is not dumped."""
    import numpy as np
    n, stride = out.shape
    keep = min(n, DUMP_CONSENSUS_BYTES // (4 * stride))
    idx = np.arange(n) if keep == n else np.sort(np.random.default_rng(0).choice(n, keep, replace=False))
    cons = out[idx].astype(np.float32)
    cons[np.arange(stride)[None, :] >= lens[idx][:, None]] = 0
    os.makedirs(path, exist_ok=True)
    for name, a in (("consensus", cons), ("consensus_length", lens[idx].astype(np.float32)),
                    ("polished", pol[idx].astype(np.float32)), ("status", st[idx].astype(np.float32)),
                    ("window_index", idx.astype(np.float64))):
        np.save(os.path.join(path, name + ".npy"), a)


def dump_aligner_outputs(path, results):
    """config 5, --dump-outputs: what the last timed aligner launch handed back (rp_aln_fetch_cigar per overlap) for a
    fixed seeded sample of DUMP_ALIGNER_PAIRS overlaps (all of them when there are fewer), listed in aln_index.npy:
    aln_edit_distance.npy and aln_status.npy per overlap, the CIGAR strings' byte codes concatenated in aln_cigar.npy
    (float32) with aln_cigar_offset.npy marking where each one starts and ends."""
    import numpy as np
    n = len(results)
    idx = np.arange(n) if n <= DUMP_ALIGNER_PAIRS else np.sort(
        np.random.default_rng(0).choice(n, DUMP_ALIGNER_PAIRS, replace=False))
    cigars = [results[i][0] for i in idx]
    offset = np.zeros(len(idx) + 1, np.float64)
    offset[1:] = np.cumsum([len(c) for c in cigars])
    os.makedirs(path, exist_ok=True)
    for name, a in (("aln_cigar", np.frombuffer(b"".join(cigars), np.uint8).astype(np.float32)),
                    ("aln_cigar_offset", offset),
                    ("aln_edit_distance", np.asarray([results[i][1] for i in idx], np.float32)),
                    ("aln_status", np.asarray([results[i][2] for i in idx], np.float32)),
                    ("aln_index", idx.astype(np.float64))):
        np.save(os.path.join(path, name + ".npy"), a)


# ---------------------------------------------------------------------------------------------------------------
def parse_cpulist(text):
    cpus = set()
    for part in text.strip().split(","):
        if not part:
            continue
        a, _, b = part.partition("-")
        cpus.update(range(int(a), int(b or a) + 1))
    return cpus


_AFFINITY_BEFORE_BINDING = []   # bind_near_gpu() notes what it narrowed; the CPU baselines get the whole host back


def bind_near_gpu(props):
    """Multi-rank runs: keep this rank's host threads (and with them its pinned staging buffers, first touched after this
    call) on the CPUs of the socket its GPU hangs off (sysfs local_cpulist of the PCI device), as `numactl` would on a
    production node; without it, 8 ranks' packers and H2D/D2H staging wander across both sockets.  Returns a short
    description for the JSON line; any failure leaves the affinity untouched."""
    if os.environ.get("RP_BENCH_NO_BIND"):
        return "off (RP_BENCH_NO_BIND)"
    try:
        dev = "%04x:%02x:%02x.0" % (props.pci_domain_id, props.pci_bus_id, props.pci_device_id)
        with open("/sys/bus/pci/devices/%s/local_cpulist" % dev) as f:
            near = parse_cpulist(f.read())
        have = os.sched_getaffinity(0)
        use = near & have
        if not use or use == have:
            return "none needed (%d cpus, all local to %s)" % (len(have), dev)
        os.sched_setaffinity(0, use)
        _AFFINITY_BEFORE_BINDING.append(have)
        return "%d of %d cpus, local to %s" % (len(use), len(have), dev)
    except Exception as e:  # noqa: BLE001 — sysfs layout differs between boxes; the run is valid without the binding
        return "unavailable (%s)" % type(e).__name__


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", type=int, default=2, choices=sorted(CONFIGS))
    ap.add_argument("--windows", type=int, default=0, help="override the config's window count")
    ap.add_argument("--banded", type=int, default=-1, help="override the config's -b flag (0/1)")
    ap.add_argument("--frag-reads", type=int, default=400, help="config 5: reads per GPU")
    ap.add_argument("--frag-read-len", type=int, default=10000)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--internal-by-reference", action="store_true", help=argparse.SUPPRESS)
    ap.add_argument("--e2e-batches", type=int, default=2,
                    help="batch objects the end-to-end arm cycles through (racon's -c/--cudapoa-batches)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write what the last timed end-to-end step (and, config 5, the last aligner launch) returned as "
                         "DIR/<name>.npy (rank 0's windows)")
    args = ap.parse_args()
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes what this project's timed path computed: not available with --impl reference")
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup

    rank = env_int("RANK", 0)
    world = env_int("WORLD_SIZE", 1)
    local = env_int("LOCAL_RANK", 0)
    if args.impl == "reference":
        run_reference(args, rank, world)
        return

    import numpy as np
    import torch
    import torch.distributed as dist
    from racon_b200 import api, shard, windows

    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device — the POA hot path has no CPU fallback")
    torch.cuda.set_device(local)
    distributed = world > 1
    host_binding = bind_near_gpu(torch.cuda.get_device_properties(local)) if distributed else "single rank: not bound"
    if distributed:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        # The POA kernel is persistent and fills every SM's shared memory: a collective's kernel only gets on the GPU where a
        # POA block retires.  On a high-priority stream it takes those slots ahead of the next POA launch already waiting for
        # them (the per-step consensus gather then completes inside the running step instead of behind the next kernel).
        os.environ.setdefault("TORCH_NCCL_HIGH_PRIORITY", "1")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))

    cfg = CONFIGS[args.config]
    banded = cfg["banded"] if args.banded < 0 else bool(args.banded)
    wl = cfg["wl"]
    aligner = aln_results = None
    meta = {}
    if cfg["shape"] == "frag":
        fw = frag_workload(args, rank)
        ws = fw["windows"]
        aln_results, aligner = time_aligner(fw["pairs"], local, args.steps, args.warmup)
        meta = {"reads_per_gpu": fw["reads"], "overlaps_per_gpu": fw["overlaps"], "windows_total": ws.n_windows * world,
                "window_build_s": fw["init_s"]}
    else:
        ws, meta = make_windows(args.config, args, rank, world)
    n = ws.n_windows
    n_total = meta.get("windows_total", n * world)
    mem = int(os.environ.get("RP_BENCH_MEM", 40e9))     # device-memory budget per batch object (several are alive)
    if args.internal_by_reference:
        res = by_reference_leg(args, api, windows, torch, ws, local, wl, banded, mem, dist if distributed else None, n_total)
        if rank == 0:
            res["host_cpu_binding"] = host_binding
            print(json.dumps(res))
        if distributed:
            dist.destroy_process_group()
        return

    def new_batch():
        return api.PoaBatch(device=local, window_length=wl, banded=banded, mem_bytes=mem)

    batch = new_batch()
    stream = torch.cuda.current_stream()
    batch.set_stream(stream.cuda_stream)
    t_pack0 = time.perf_counter()
    took = batch.add_window_set(ws)
    pack_ms = 1e3 * (time.perf_counter() - t_pack0)
    assert took == n, "batch object could not hold the workload (%d of %d windows)" % (took, n)
    lens_in = np.diff(ws.seq_off.astype(np.int64))
    stride = int(2 * lens_in.max() + 64)

    def barrier():
        if distributed:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- counters launch (untimed): algorithmic bytes of this batch + a correctness probe ----------
    batch.enable_counters(True)
    batch.run()
    batch.sync()
    info = batch.info()
    band_info = batch.band_info()
    out, lens, pol, st = batch.fetch_all(stride)
    if (st != 0).any():
        raise SystemExit("bench.py: %d windows hit a device limit" % int((st != 0).sum()))
    checksum = "%016x" % windows.fnv1a64([out[i, :lens[i]].tobytes() for i in range(min(n, 200))])
    if cfg["shape"] == "ont" and rank == 0 and n >= 200 and checksum != "50f18d884e3254d2":
        raise SystemExit("bench.py: consensus checksum %s != the reference's known answer 50f18d884e3254d2" % checksum)
    alg_bytes = 2.0 * (info["dp_cells"] + info["pred_cells"])
    batch.enable_counters(False)

    # ---- kernel-only arm: inputs resident in HBM --------------------------------------------------
    # (1) the kernel alone: isolated launches on one stream, CUDA events around each -> roofline.kernel_ms
    batch.upload()
    for _ in range(args.warmup):
        batch.launch()
    barrier()
    iso = [torch.cuda.Event(enable_timing=True) for _ in range(4)]
    iso[0].record(stream)
    for k in range(3):
        batch.launch()
        iso[k + 1].record(stream)
    barrier()
    kern_ms = [iso[k].elapsed_time(iso[k + 1]) for k in range(3)]
    # (2) the K timed steps: one launch per step over the resident batch, steps alternating between two batch objects
    # on two streams (both hold the whole batch in HBM), so that the tail of one step — the last windows of a launch
    # leave most SMs idle — is filled by the head of the next, as it is in a real multi-batch run
    batch2 = new_batch()
    stream2 = torch.cuda.Stream()
    batch2.set_stream(stream2.cuda_stream)
    assert batch2.add_window_set(ws) == n
    batch2.upload()
    batch2.launch()
    barrier()
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    ev0, ev1, evb = (torch.cuda.Event(enable_timing=True) for _ in range(3))
    launches0 = batch.info()["launches"] + batch2.info()["launches"]
    ev0.record(stream)
    stream2.wait_event(ev0)
    for k in range(args.steps):
        (batch if k % 2 == 0 else batch2).launch()
    evb.record(stream2)
    stream.wait_event(evb)
    ev1.record(stream)
    barrier()
    clocks = sampler.stop() if rank == 0 else None
    total_ms = ev0.elapsed_time(ev1)
    gpu_launches = batch.info()["launches"] + batch2.info()["launches"] - launches0
    batch2.close()
    forced = None
    if banded:
        # A banded object (racon -b) picks the kernel by window length: the band layout from 768 bases on, the full matrix
        # below — same results, the faster of the two (DESIGN.md §3b).  Everything above measured THAT.  The band layout
        # itself, asked for explicitly on the same windows: isolated launches + how many band results the device refused.
        saved = os.environ.get("RP_POA_BAND_K")
        os.environ["RP_POA_BAND_K"] = "8"
        bf = api.PoaBatch(device=local, window_length=wl, banded=True, mem_bytes=mem)
        bf.set_stream(stream.cuda_stream)
        assert bf.add_window_set(ws) == n
        bf.run()
        bf.sync()
        fo, fl, _, fst = bf.fetch_all(stride)
        f_ck = "%016x" % windows.fnv1a64([fo[i, :fl[i]].tobytes() for i in range(min(n, 200))])
        fbi = bf.band_info()
        bf.upload()
        bf.launch()
        barrier()
        f0, f1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        f0.record(stream)
        bf.launch()
        bf.launch()
        f1.record(stream)
        barrier()
        forced = {"ms": f0.elapsed_time(f1) / 2, "tried": fbi["band_alignments"], "redone": fbi["band_redone_full"],
                  "width": fbi["band_width"], "same_consensus": f_ck == checksum and not (fst != 0).any()}
        bf.close()
        if saved is None:
            os.environ.pop("RP_POA_BAND_K", None)
        else:
            os.environ["RP_POA_BAND_K"] = saved

    # ---- end-to-end arm: C-ABI call with host buffers (H2D + kernel + D2H + fetch) ------------------
    # what racon's CUDAPolisher does with `-c K` batch objects (cudapolisher.cpp:254-276): each object, on its own
    # stream, is reset, filled from host buffers (copied into pinned staging), run (H2D + kernel + D2H, asynchronous)
    # and read back; while one object's kernel runs, the host fills the next one.
    nb = max(1, args.e2e_batches)
    objs = [new_batch() for _ in range(nb)]
    bounds = [n * k // nb for k in range(nb + 1)]
    last = {}

    # the one exchange step of the path: the final consensus gather over NCCL (SURVEY.md §8e), once per step, asynchronous:
    # a step's gather is queued when its last object is read back and finished before the next one is queued (and before
    # the timed region ends), so no rank waits for another rank in the middle of its step
    gather = shard.RowGather(n, stride, device="cuda", dst=0) if distributed else None

    def finalize(parts):
        out, lens, pol, st = (np.concatenate([p[i] for p in parts]) for i in range(4))
        if gather is not None:
            got = gather.finish(block=False)   # schedules the read-back of the previous step's gather, never waits
            if got is not None:
                last["gathered"] = got
            gather.start(out, lens)
        last["out"], last["lens"], last["pol"], last["st"] = out, lens, pol, st

    # where the host spends a step (wall clock of this rank's calling thread, summed over the timed steps): filling the
    # objects, queueing H2D + kernel + D2H, waiting for a kernel to finish, reading results back, the consensus gather
    phase = {"add": 0.0, "run": 0.0, "wait": 0.0, "fetch": 0.0, "gather": 0.0}
    clock = time.perf_counter

    def plugin_steps(n_steps):
        pending = [None] * nb
        parts = {}

        def collect(k):
            t_a = clock()
            objs[k].sync()
            t_b = clock()
            s_done = pending[k]
            parts[s_done][k] = objs[k].fetch_all(stride)
            t_c = clock()
            pending[k] = None
            if all(x is not None for x in parts[s_done]):
                finalize(parts.pop(s_done))
            phase["wait"] += t_b - t_a
            phase["fetch"] += t_c - t_b
            phase["gather"] += clock() - t_c

        for s_i in range(n_steps):
            parts[s_i] = [None] * nb
            for k, b in enumerate(objs):
                if pending[k] is not None:
                    collect(k)
                t_a = clock()
                b.reset()
                cnt = bounds[k + 1] - bounds[k]
                assert b.add_window_set(ws, first=bounds[k], count=cnt) == cnt
                t_b = clock()
                b.run()
                phase["add"] += t_b - t_a
                phase["run"] += clock() - t_b
                pending[k] = s_i
        for k in range(nb):
            if pending[k] is not None:
                collect(k)
        t_a = clock()
        if gather is not None:
            got = gather.finish()
            if got is not None:
                last["gathered"] = got
        phase["gather"] += clock() - t_a

    plugin_steps(2)
    barrier()
    for key in phase:
        phase[key] = 0.0
    t0 = time.perf_counter()
    plugin_steps(args.steps)
    barrier()
    out, lens = last["out"], last["lens"]
    e2e_ms = 1e3 * (time.perf_counter() - t0)
    if windows.fnv1a64([out[i, :lens[i]].tobytes() for i in range(min(n, 200))]) != int(checksum, 16):
        raise SystemExit("bench.py: end-to-end arm produced a different consensus than the kernel-only arm")
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, out, lens, last["pol"], last["st"])
        if aln_results is not None:
            dump_aligner_outputs(args.dump_outputs, aln_results)
    io = objs[0].info()
    io["h2d_bytes"] = sum(b.info()["h2d_bytes"] for b in objs)
    io["d2h_bytes"] = sum(b.info()["d2h_bytes"] for b in objs)
    for b in objs + [batch]:
        b.close()
    torch.cuda.empty_cache()

    # ---- max over ranks ---------------------------------------------------------------------------
    tt = torch.tensor([total_ms, e2e_ms, float(forced["tried"] if forced else 0), float(forced["redone"] if forced else 0),
                       float(forced["ms"] if forced else 0.0)], dtype=torch.float64, device="cuda")
    if distributed:
        t2 = tt.clone()
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        dist.all_reduce(t2, op=dist.ReduceOp.SUM)
        band_tot = (float(t2[2]), float(t2[3]))
    else:
        band_tot = (float(tt[2]), float(tt[3]))
    total_ms, e2e_ms, forced_ms = float(tt[0]), float(tt[1]), float(tt[4])

    if rank == 0:
        peak, peak_src = measured_hbm_peak()
        ms_per_step = total_ms / args.steps
        value = n_total / (ms_per_step * 1e-3)
        kern_avg_ms = sum(kern_ms) / len(kern_ms)
        achieved = alg_bytes / (kern_avg_ms * 1e-3) / 1e9
        traffic = ncu_traffic(args.config)
        line = {
            "metric": cfg["metric"], "value": value, "unit": "windows/s", "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": cfg["scaling"],
            "vs_baseline": None, "dtype": "int16", "data": "synthetic",
            "config": config_key(cfg, args),
            "run": dict({"windows_rank0": n,
                            "window_len": wl, "banded": banded,
                            "parallelism": "windows sharded across %d GPU(s), no data-path collective" % world,
                            "l2": "inputs (%.0f MB) + per-step DP scratch (>> 126 MB) exceed L2; no explicit flush"
                                  % (io["h2d_bytes"] / 1e6),
                            "steps_overlap": "timed steps alternate between two resident batch objects on two streams; "
                                             "roofline.kernel_ms is an isolated launch",
                            "workers_windows_in_flight": io["workers"], "first_pack_ms": pack_ms,
                            "host_cpu_binding": host_binding,
                            "consensus_fnv_first200": checksum}, **meta),
            "e2e": {"value": n_total * args.steps / (e2e_ms * 1e-3), "unit": "windows/s",
                    "h2d_bytes_per_step": io["h2d_bytes"], "d2h_bytes_per_step": io["d2h_bytes"],
                    "batch_objects": nb,
                    "host_ms_per_step_rank0": {k2: round(1e3 * v / args.steps, 2) for k2, v in phase.items()},
                    "includes": "every step, per batch object: rp_poa_reset + rp_poa_add_window_set (host buffers -> pinned "
                                "staging) + rp_poa_run (H2D, kernel, D2H) + rp_poa_sync + rp_poa_fetch_all; the objects stay "
                                "in flight across steps (as CUDAPolisher keeps its batches busy), timed from the first add "
                                "to the last fetch"
                                + ("; + one NCCL all_gather of the step's consensus per step, queued asynchronously and "
                                   "finished inside the timed region" if distributed else "")},
            "gpu_launches": int(gpu_launches),
            "clocks": clocks,
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s",
                         "frac": achieved / peak, "traffic": (traffic or {}).get("dram_bytes_per_launch"),
                         "traffic_source": (traffic or {}).get("source"),
                         "kernel": "rp_poa_kernel", "kernel_ms": kern_avg_ms,
                         "achieved_overlapped": alg_bytes / (ms_per_step * 1e-3) / 1e9 * (n / max(1, n_total / world)),
                         "algorithmic_bytes_per_launch": alg_bytes,
                         "algorithmic_bytes_per_window": alg_bytes / n, "peak_source": peak_src,
                         "note": "algorithmic bytes count the cells the accepted DP computed: the full rows, or with -b "
                                 "the band's columns per row"},
        }
        if banded:
            line["band"] = {
                "policy": "a banded object uses the band layout for windows of >= 768 bases and the full-matrix kernel below "
                          "(same results; the faster kernel either way): value / e2e / roofline above are what -b runs for "
                          "this window length",
                "layout_in_use_here": bool(band_info["band_layout_in_use"]),
                "band_layout_forced": {
                    "width_columns": forced["width"], "alignments_tried_in_band": int(band_tot[0]),
                    "redone_with_full_matrix_on_device": int(band_tot[1]),
                    "same_consensus_as_default": bool(forced["same_consensus"]),
                    "kernel_ms_isolated": forced_ms, "value_isolated": n_total / (forced_ms * 1e-3),
                    "value_default_isolated": n / (kern_avg_ms * 1e-3) * (n_total / n)}}
        if aligner:
            line["aligner"] = aligner
        if cfg["shape"] != "frag" and not os.environ.get("RP_BENCH_NO_BY_REFERENCE"):
            br = by_reference(args, world)
            if "consensus_fnv_first200" in br:
                br["same_consensus_as_by_pointer"] = br["consensus_fnv_first200"] == checksum
            line["e2e"]["by_reference"] = br
        if not args.no_cpu_baseline:
            line["cpu_baseline"] = cpu_baseline(args, cfg, banded, world, ws)
        print(json.dumps(line))
    if distributed:
        # The other ranks wait for rank 0's baselines on the HOST (rendezvous store), not in an NCCL barrier: a pending
        # NCCL collective is a spinning kernel on every GPU, and the reference's GPU path is being timed on those GPUs.
        import datetime
        store = dist.distributed_c10d._get_default_store()
        if rank == 0:
            store.set("bench_baselines_done", "1")
            time.sleep(1.0)   # let the waiters read the key before the process that may host the store goes away
        else:
            store.wait(["bench_baselines_done"], datetime.timedelta(minutes=20))
        dist.destroy_process_group()


def run_group(cmd, timeout, **kw):
    """subprocess.run with a time limit that takes the child's whole process group down (a torchrun child has workers of its
    own: killing only the launcher would leave them on the GPUs).  Returns (returncode, stdout, stderr)."""
    import signal
    p = subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=kw.pop("stderr", subprocess.PIPE), text=True,
                         start_new_session=True, **kw)
    try:
        out, err = p.communicate(timeout=timeout)
        return p.returncode, out, err or ""
    except subprocess.TimeoutExpired:
        try:
            os.killpg(p.pid, signal.SIGKILL)   # the session we started: nothing else is in it
        except ProcessLookupError:
            pass
        p.communicate()
        raise


def by_reference(args, world):
    """The end-to-end arm once more with the windows added BY REFERENCE into a device-resident read store (SURVEY §8 f2;
    rp_reads_create + rp_poa_add_window_set_refs): the sequences are uploaded once, before the timed region — in a racon run
    every read belongs to the run, not to a batch —, a step then moves descriptors only and the layers are extracted on the
    device.  Reported beside `e2e`, which stays the by-pointer call of the reference's own interface.  Own process with a
    time limit, like the reference's GPU path: the newest code path must not be able to take the bench line down."""
    here = os.path.dirname(os.path.abspath(__file__))
    cmd = [sys.executable]
    env = dict(os.environ)
    if world > 1:
        # the same ranks once more, as a job of its own: one process per GPU under torchrun, on another port
        import socket
        with socket.socket() as sk:
            sk.bind(("127.0.0.1", 0))
            port = sk.getsockname()[1]
        for key in list(env):
            if key in ("RANK", "LOCAL_RANK", "WORLD_SIZE", "LOCAL_WORLD_SIZE", "GROUP_RANK", "GROUP_WORLD_SIZE",
                       "MASTER_ADDR", "MASTER_PORT", "ROLE_RANK", "ROLE_NAME", "ROLE_WORLD_SIZE") or \
                    key.startswith("TORCHELASTIC_"):
                del env[key]
        cmd += ["-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", str(world), "--master-addr", "127.0.0.1",
                "--master-port", str(port)]
    cmd += [os.path.join(here, "bench.py"), "--internal-by-reference", "--gpus", str(world), "--config", str(args.config),
            "--steps", str(args.steps), "--warmup", str(args.warmup), "--e2e-batches", str(args.e2e_batches)]
    if args.windows:
        cmd += ["--windows", str(args.windows)]
    if args.banded >= 0:
        cmd += ["--banded", str(args.banded)]
    try:
        rc, out, err = run_group(cmd, 300, cwd=here, env=env)
        lines = [l for l in out.splitlines() if l.startswith("{")]
        if lines:
            return json.loads(lines[-1])
        return {"unavailable": "no output (exit %d): %s" % (rc, err.strip().splitlines()[-1:] or "")}
    except Exception as e:  # noqa: BLE001 - reported, never fatal
        return {"unavailable": "%s" % e}


def by_reference_leg(args, api, windows, torch, ws, local, wl, banded, mem, dist=None, n_total=None):
    """child process(es) of by_reference(): K timed steps, each = per batch object reset + add-by-reference + run
    (descriptor H2D, gather kernel, POA kernel, D2H) + sync + fetch_all, two objects in flight; host clock between device
    syncs (+ a barrier on both sides and the max over ranks when there are several)"""
    import numpy as np
    n = ws.n_windows
    n_total = n_total or n

    def fence():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    stride = int(2 * np.diff(ws.seq_off.astype(np.int64)).max() + 64)
    t0 = time.perf_counter()
    store = api.ReadStore.from_flat(ws.bases, ws.seq_off, ws.quals, ws.seq_has_qual, device=local)
    torch.cuda.synchronize()
    store_ms = 1e3 * (time.perf_counter() - t0)
    refs = windows.as_refs(ws)
    nb = max(1, args.e2e_batches)
    objs = [api.PoaBatch(device=local, window_length=wl, banded=banded, mem_bytes=mem) for _ in range(nb)]
    bounds = [n * k // nb for k in range(nb + 1)]
    last = {}

    def steps(n_steps):
        pending = [None] * nb
        parts = {}

        def collect(k):
            objs[k].sync()
            s_done = pending[k]
            parts[s_done][k] = objs[k].fetch_all(stride)
            pending[k] = None
            if all(x is not None for x in parts[s_done]):
                done = parts.pop(s_done)
                last["out"], last["lens"], _, last["st"] = (np.concatenate([d[i] for d in done]) for i in range(4))

        for s_i in range(n_steps):
            parts[s_i] = [None] * nb
            for k, b in enumerate(objs):
                if pending[k] is not None:
                    collect(k)
                b.reset()
                cnt = bounds[k + 1] - bounds[k]
                assert b.add_window_set_refs(store, refs, first=bounds[k], count=cnt) == cnt
                b.run()
                pending[k] = s_i
        for k in range(nb):
            if pending[k] is not None:
                collect(k)

    steps(2)
    fence()
    t0 = time.perf_counter()
    steps(args.steps)
    fence()
    ms = 1e3 * (time.perf_counter() - t0)
    if dist is not None:
        t = torch.tensor([ms], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = float(t[0])
    out, lens = last["out"], last["lens"]
    res = {"value": n_total * args.steps / (ms * 1e-3), "unit": "windows/s", "ms_per_step": ms / args.steps,
           "h2d_bytes_per_step": sum(b.info()["h2d_bytes"] for b in objs),
           "d2h_bytes_per_step": sum(b.info()["d2h_bytes"] for b in objs),
           "per_rank": dist is not None, "store_device_bytes": store.device_bytes(), "store_upload_ms_once": store_ms,
           "device_limit_windows": int((last["st"] != 0).sum()),
           "consensus_fnv_first200": "%016x" % windows.fnv1a64([out[i, :lens[i]].tobytes() for i in range(min(n, 200))]),
           "includes": "per step and batch object: rp_poa_reset + rp_poa_add_window_set_refs (metadata only) + rp_poa_run "
                       "(descriptor H2D, layer-extraction kernel, POA kernel, D2H) + rp_poa_sync + rp_poa_fetch_all; the "
                       "sequences were uploaded once before the timed region (store_upload_ms_once)"
                       + ("; one process per GPU, barrier on both sides, max over ranks, no consensus gather"
                          if dist is not None else "")}
    for b in objs:
        b.close()
    store.close()
    return res


def cpu_baseline(args, cfg, banded, world, ws):
    """oracle/_ref (the unmodified reference) on the box's host cores, bounded sample (~10-30 s of CPU work)."""
    from oracle import bindings as ob
    from racon_b200 import windows
    if _AFFINITY_BEFORE_BINDING:   # the timed GPU arms are over: the reference runs on every core of the host, not on the
        try:                       # socket this rank was bound to
            os.sched_setaffinity(0, _AFFINITY_BEFORE_BINDING[0])
        except OSError:
            pass
    cores = host_cores()
    if ob.have_ref():
        kind, fn = "reference", ob.ref_consensus
    else:
        kind, fn = "port", ob.oracle_consensus
    per_core = 300 if cfg["shape"] in ("ont", "frag") else 2500
    n_sample = min(ws.n_windows, max(64, per_core * cores))
    sample_ws = windows.slice_windows(ws, 0, n_sample)
    threads = cores
    if cores >= 4:  # see run_reference(): best of all hardware threads / half of them
        probe = windows.slice_windows(sample_ws, 0, min(n_sample, 16 * cores))
        threads = cores if fn(probe, threads=cores)[2] <= fn(probe, threads=cores // 2)[2] else cores // 2
    secs = fn(sample_ws, threads=threads)[2]
    res = {"value": n_sample / secs, "unit": "windows/s", "cores": threads, "kind": kind,
           "sample": "first %d windows of rank 0's workload, %d host threads (of %d hardware threads), consensus loop "
                     "only (%.1f s)" % (n_sample, threads, cores, secs)}
    if cfg["shape"] == "ont":
        res["gpu_reference"] = gpu_reference(args, cfg, banded, world)
    elif cfg["shape"] == "ngs":
        res["gpu_reference"] = {"note": "the reference's CUDA path marks every kNGS window failed and re-runs it on the CPU "
                                        "(src/cuda/cudabatch.cpp:229-256): its throughput on this workload is the "
                                        "cpu_baseline above"}
    return res


def gpu_reference(args, cfg, banded, world):
    """The reference's OWN GPU path (GenomeWorks cudapoa, unmodified, oracle/_ref/libref_cudapoa.so) on the same workload,
    the same box and the SAME number of GPUs, driven like CUDAPolisher::polish drives it (two batch objects per GPU, one
    host thread each) — SURVEY §8(d)'s GPU baseline.  Separate process with a time limit: a failure inside the reference
    library must not take the bench line down.  Timing only (cudapoa's consensus is not spoa's)."""
    here = os.path.dirname(os.path.abspath(__file__))
    n = args.windows or cfg["windows"]
    total = n if cfg["scaling"] == "strong" else n * world
    cmd = [sys.executable, "-m", "oracle.cudapoa_time", "--windows", str(total), "--devices", str(world), "--batches", "2"]
    if banded:
        cmd.append("--banded")
    try:
        rc, out, _ = run_group(cmd, 240, cwd=here, stderr=subprocess.DEVNULL)
        lines = [l for l in out.splitlines() if l.startswith("{")]
        return json.loads(lines[-1]) if lines else {"unavailable": "no output (exit %d)" % rc}
    except Exception as e:  # noqa: BLE001 - reported, never fatal
        return {"unavailable": "%s" % e}


if __name__ == "__main__":
    main()
