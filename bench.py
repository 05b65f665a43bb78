#!/usr/bin/env python3
"""bench.py -- throughput of the motif-scan hot path on B200, next to the reference CPU path.

    python bench.py [--gpus N] [--steps K] [--warmup W]            our arm (CUDA, C ABI)
    python bench.py --impl reference [--gpus N] [--steps K] ...    the reference's CPU extension

Metric (BASELINE.json): motif*bp scored per second, both strands.

Headline workload = BASELINE.json configs[3], north_star's target: the genome-wide 2-strand scan of a
synthetic hg19-shaped genome (25 chromosomes, 3.1 Gbp, ~7 % N) with a JASPAR-2020-vertebrates-shaped set
of 750 PWMs (length 6-30), cutoffs at p = 1e-4.  STRONG scaling: the same genome at every N; the packed
genome's position space is cut into N contiguous shares, rank r scans share r (one process per GPU), and the
only cross-rank step is the final host-side gather of the per-motif site counts (750 int64 per rank sent to
rank 0 over gloo -- no NCCL on this path), which sits INSIDE every timed step.

One "step" = one pass over the whole genome:
  value        the rank's share already resident in HBM (2-bit codes + N mask); prefilter + exact fp64
               re-score + ordering of the sites + count gather.  CUDA events on the launch stream.
  e2e          host buffers in, host buffers out, through the product API (`GenomeScanner.scan`, i.e. the C-ABI
               calls msb_seqs_from_packed / msb_scan_ranges / msb_result_*): every step uploads the share's
               packed planes from pinned host memory (0.375 B/bp), scans it unit by unit and copies ALL sites
               (score + packed position and strand: 12 B each, MSB_SCAN_COMPACT) to pinned host memory, upload and download
               overlapping the scan of the neighbouring unit; then the count gather.  Wall clock between
               synchronisations, max over ranks.  `e2e.variants.counts_out` is the same with only the
               per-motif counts coming back (MSB_SCAN_COUNTS).
  secondary    BASELINE.json configs[1] (750 PWMs x 50,000 1 kb peaks per GPU, weak-scaled as in round 1),
               device-resident and end to end, in the `configs1` block of the same JSON line.
Prints ONE JSON line on rank 0.

`--dump-outputs DIR` (rank 0) writes, after the timed steps, what the last timed step of each path returned, as
float64 .npy files: `genome_counts` (per-motif site counts of the genome-wide scan, gathered over the ranks),
`genome_sites_{motif,chrom,start,score,strand}` (a fixed, seeded sample of DUMP_SITES sites of rank 0's share,
from the end-to-end leg, in site order), `configs1_counts` (rank 0's per-motif counts of the secondary block's
device-resident leg) and `configs1_sites_{motif,region,start,score,strand}` (the same kind of sample of rank 0's
sites from the secondary block's end-to-end leg; `start` is relative to the peak `region`).  The inputs are
seeded, so two builds run with the same arguments can be compared file for file.
"""
import argparse
import hashlib
import json
import os
import statistics
import subprocess
import sys
import tempfile
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

METRIC = "motif_bp_scored_per_sec_both_strands"
UNIT = "motif*bp/s"
N_MOTIFS = 750
P_VALUE = "1e-4"
N_BACKGROUND = 100000
GENOME_SEED = 19
N_FRACTION = 0.07
UNIT_BP = 1 << 26                 # largest unit; a share is cut into at least 8 units so that the first upload and the
MIN_UNIT_BP = 1 << 24             # last download (the only copies nothing hides) stay small next to the share
# secondary block (configs[1])
N_REGIONS = 50000
REGION_BP = 1000
DUMP_SITES = 1 << 19              # --dump-outputs: 2 samples of 5 float64 arrays of this many sites, 40 MB


def genome_shape(scale=1.0):
    from motifscan_b200.synth import HG19_NAMES, HG19_SIZES
    return HG19_NAMES, [max(int(s * scale), 64) for s in HG19_SIZES]


def workload_name(scale=1.0):
    names, sizes = genome_shape(scale)
    return (f"configs[3]: genome-wide scan of a synthetic hg19-shaped genome ({len(sizes)} chromosomes, {sum(sizes)} bp, "
            f"{int(100 * N_FRACTION)} % N) x {N_MOTIFS} JASPAR-2020-vertebrates-shaped PWMs (len 6-30), both strands, "
            f"cutoffs p={P_VALUE}; position space sharded over the ranks")


def load_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as fh:
            return json.load(fh), "measured (MEASURED_PEAKS.json)"
    return {"hbm_gbs": 6650.0, "sm_max_mhz": 1965.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1590.0}, \
        "fallback (B200_PROFILING.md)"


class ClockSampler:
    """SM clock, power and throttle reasons of one GPU sampled through NVML every ~2 ms on a thread for
    the whole timed region; falls back to `nvidia-smi -lms` when the NVML binding is missing."""
    FIELDS = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
              "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
              "clocks_event_reasons.sw_power_cap")

    def __init__(self, index, uuid=None, period_s=0.005):
        self.index = index
        self.uuid = uuid
        self.period_s = period_s
        self.proc = None
        self.path = None
        self.thread = None
        self.stop_flag = threading.Event()
        self.samples = []          # (sm_mhz, power_w, reasons bitmask)
        self.max_mhz = None
        self.nvml = None

    def _nvml_loop(self, handle):
        nv = self.nvml
        get_reasons = getattr(nv, "nvmlDeviceGetCurrentClocksEventReasons", None) or nv.nvmlDeviceGetCurrentClocksThrottleReasons
        while not self.stop_flag.is_set():
            try:
                self.samples.append((nv.nvmlDeviceGetClockInfo(handle, nv.NVML_CLOCK_SM),
                                     nv.nvmlDeviceGetPowerUsage(handle) / 1e3, int(get_reasons(handle))))
            except Exception:
                break
            time.sleep(self.period_s)

    def start(self):
        try:
            import pynvml as nv
            nv.nvmlInit()
            handle = None
            if self.uuid:   # CUDA_VISIBLE_DEVICES may renumber the devices: find ours by UUID
                name = self.uuid if str(self.uuid).startswith("GPU-") else f"GPU-{self.uuid}"
                for cand in (name, name.encode()):
                    try:
                        handle = nv.nvmlDeviceGetHandleByUUID(cand)
                        break
                    except Exception:
                        handle = None
            if handle is None:
                handle = nv.nvmlDeviceGetHandleByIndex(self.index)
            self.nvml = nv
            self.max_mhz = nv.nvmlDeviceGetMaxClockInfo(handle, nv.NVML_CLOCK_SM)
            self.thread = threading.Thread(target=self._nvml_loop, args=(handle,), daemon=True)
            self.thread.start()
            return
        except Exception:
            self.nvml = None
        try:
            fd, self.path = tempfile.mkstemp(suffix=".csv")
            os.close(fd)
            self.proc = subprocess.Popen(
                ["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.FIELDS}",
                 "--format=csv,noheader,nounits", "-lms", "20"],
                stdout=open(self.path, "w"), stderr=subprocess.DEVNULL)
        except Exception:
            self.proc = None

    def stop(self):
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        if self.thread is not None:
            self.stop_flag.set()
            self.thread.join(timeout=2)
            nv = self.nvml
            names = {"hw_slowdown": "HwSlowdown", "hw_thermal_slowdown": "HwThermalSlowdown",
                     "sw_thermal_slowdown": "SwThermalSlowdown", "sw_power_cap": "SwPowerCap"}
            bits = {}
            for key, suffix in names.items():
                for prefix in ("nvmlClocksEventReason", "nvmlClocksThrottleReason"):
                    if hasattr(nv, prefix + suffix):
                        bits[key] = getattr(nv, prefix + suffix)
                        break
            if self.samples:
                mask = 0
                for _, _, r in self.samples:
                    mask |= r
                busy = [x for x in self.samples if x[1] > 0.5 * max(y[1] for y in self.samples)] or self.samples
                out.update(sm_mhz=statistics.median(x[0] for x in busy), sm_max_mhz=self.max_mhz,
                           sm_min_mhz=min(x[0] for x in self.samples), power_w_max=max(x[1] for x in self.samples),
                           reasons=sorted(k for k, b in bits.items() if mask & b), samples=len(self.samples),
                           source="NVML, 5 ms period; median over the samples above half the peak power (under load)")
            return out
        if self.proc is None:
            return out
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap")
        try:
            for line in open(self.path):
                parts = [p.strip() for p in line.split(",")]
                if len(parts) < 7:
                    continue
                try:
                    sm.append(float(parts[0]))
                    mx.append(float(parts[1]))
                except ValueError:
                    continue
                for name, flag in zip(names, parts[3:7]):
                    if flag.lower().startswith("active"):
                        reasons.add(name)
            os.unlink(self.path)
        except Exception:
            pass
        if sm:
            out.update(sm_mhz=statistics.median(sm), sm_max_mhz=max(mx), reasons=sorted(reasons),
                       samples=len(sm), source="nvidia-smi -lms 20")
        return out


# ------------------------------------------------------------------------------------------------
# workload
# ------------------------------------------------------------------------------------------------
def n_runs(n, rng):
    """N runs of one synthetic chromosome of n bases (start, length): 10 kb telomeres, one centromere-like
    block and a handful of assembly gaps -- about N_FRACTION of the chromosome in total."""
    edge = max(1, min(10000, n // 50))
    runs = [(0, edge), (n - edge, edge)]
    budget = int(n * N_FRACTION) - 2 * edge
    if budget > 0 and n > 4 * edge:
        big = int(budget * 0.8)
        runs.append((n // 3, big))
        gaps = 8
        for k in range(gaps):
            ln = max((budget - big) // gaps, 1)
            a = int(rng.integers(edge, max(n - edge - ln, edge + 1)))
            runs.append((a, ln))
    return runs


def make_genome(device, scale=1.0):
    """The synthetic genome as a host `PackedGenome` (pinned planes), generated on the GPU with torch
    (seeded, so every rank holds the same genome) -- torch is plumbing here, not the scan path."""
    import torch
    from motifscan_b200.genome import PackedGenome
    names, sizes = genome_shape(scale)
    order = sorted(range(len(names)), key=lambda i: names[i])          # Genome.chroms is sorted (genome/__init__.py:99)
    chroms = [names[i] for i in order]
    n_blocks = sum((sizes[i] + 31) // 32 for i in order)
    codes, nmask, pin = PackedGenome._alloc(n_blocks, True)
    dev = torch.device("cuda", device)
    gen = torch.Generator(device=dev)
    gen.manual_seed(GENOME_SEED)
    rng = np.random.default_rng(GENOME_SEED)
    sh2 = (2 * torch.arange(16, device=dev, dtype=torch.int64))[None, :]
    sh1 = torch.arange(32, device=dev, dtype=torch.int64)[None, :]
    at = 0
    for i in order:
        n = sizes[i]
        nb = (n + 31) // 32
        u = torch.randint(0, 256, (nb * 32,), dtype=torch.uint8, device=dev, generator=gen)
        # composition A/T 0.297, C/G 0.203 (synth.BG up to 1/256)
        code = (u >= 76).to(torch.int64) + (u >= 128).to(torch.int64) + (u >= 180).to(torch.int64)
        del u
        isn = torch.zeros(nb * 32, dtype=torch.bool, device=dev)
        for a, ln in n_runs(n, rng):
            isn[a:a + ln] = True
        isn[n:] = False
        code[isn] = 0
        code[n:] = 0
        cw = (code.view(-1, 16) << sh2).sum(dim=1).to(torch.int32)
        mw = (isn.view(-1, 32).to(torch.int64) << sh1).sum(dim=1).to(torch.int32)
        del code, isn
        codes[2 * at:2 * (at + nb)] = cw.cpu().numpy().view(np.uint32)
        nmask[at:at + nb] = mw.cpu().numpy().view(np.uint32)
        del cw, mw
        at += nb
    torch.cuda.synchronize(dev)
    torch.cuda.empty_cache()
    return PackedGenome(chroms, {names[i]: sizes[i] for i in order}, codes, nmask, name="synthetic-hg19", _pin=pin)


def motif_workload():
    from motifscan_b200 import synth
    _, pwms, _ = synth.motif_set(N_MOTIFS, seed=2020)
    return pwms


def cutoff_cache_path(pwms):
    h = hashlib.sha1()
    for p in pwms:
        h.update(np.ascontiguousarray(p).tobytes())
    h.update(f"{N_BACKGROUND}:{P_VALUE}".encode())
    return os.path.join(tempfile.gettempdir(), f"msb200_bench_cutoffs_{h.hexdigest()[:16]}.npy")


def background():
    from motifscan_b200 import synth
    return synth.background_samples(N_BACKGROUND, 30, seed=1)


def cutoffs_gpu(engine, ctx, pwms):
    """motif --build arithmetic (cli/motif.py:129-153) on the device: background samples of the longest
    motif's length, strand 3, order statistic int(n * 1e-4) - 1, rounded to 8 decimals."""
    blob, off = background()
    motifs = engine.MotifSet(ctx, pwms)
    bg = engine.SequenceSet(ctx, blob=blob, seq_off=off)
    rank = int(N_BACKGROUND * 0.1 ** 4) - 1
    cut = engine.score_select(ctx, motifs, bg, 3, [rank])[:, 0]
    bg.close(), motifs.close()
    return np.around(cut, 8)


def cutoffs_cpu(pwms):
    """The same on the CPU with the reference's extension (or the oracle port): c_score + sort."""
    import oracle
    blob, off = background()
    raw = blob.tobytes()
    seqs = [raw[off[i]:off[i + 1]].decode("ascii") for i in range(N_BACKGROUND)]
    ref = oracle.load_reference_cscore()
    if ref is not None:
        sc = np.array(ref.c_score([p.tolist() for p in pwms], seqs, 3, os.cpu_count() or 1))
    else:
        sc = oracle.score_arrays([p.tolist() for p in pwms], seqs, 3)
    rank = int(N_BACKGROUND * 0.1 ** 4) - 1
    return np.around(-np.sort(-sc, axis=1)[:, rank], 8)


def scan_cutoffs(built):
    """Cutoffs the scans use.  A few synthetic motifs get a non-positive p = 1e-4 cutoff on the iid background;
    by the reference's rule (N adds 0, cscore.c:346) every all-N window would then be a site (2e8 gap positions
    x those motifs x 2 strands).  Motif sets built on real genomes have positive cutoffs, so both arms floor
    them at 1e-6."""
    return np.maximum(built, 1e-6)


def shared_cutoffs(pwms, build):
    """Both arms scan with the SAME cutoffs: whoever runs first builds them (the GPU arm on the device, the
    reference arm on the CPU -- bit-identical by the parity tests) and leaves them in a cache file."""
    path = cutoff_cache_path(pwms)
    if os.path.exists(path):
        try:
            cut = np.load(path)
            if cut.shape == (len(pwms),):
                return cut, "cache file written by the other arm"
        except Exception:
            pass
    cut = build()
    try:
        tmp = path + f".{os.getpid()}.tmp.npy"
        np.save(tmp, cut)
        os.replace(tmp, path)
    except OSError:
        pass
    return cut, "built by this arm"


def algorithmic_adds(pwm_lens, seq_lens):
    """SURVEY.md section 8(d): OPS = 2 * sum_seqs sum_m max(len_i - L_m + 1, 0) * L_m -- one add per PWM
    column per strand per window, the reference's inner loop (cscore.c:344-354)."""
    total = 0
    for length in seq_lens:
        w = np.maximum(int(length) - pwm_lens + 1, 0)
        total += 2 * int((w * pwm_lens).sum())
    return total


# ------------------------------------------------------------------------------------------------
# CPU side: the reference's own extension (oracle/_ref) or, if it never compiled, the oracle port.
# ------------------------------------------------------------------------------------------------
def cpu_scanner():
    import oracle
    ref = oracle.load_reference_cscore()
    if ref is not None:
        return "reference", ref.c_scan_motif
    return "port", oracle.c_scan_motif


def genome_samples(pg, n_pieces, piece_bp):
    """`n_pieces` windows of `piece_bp` bases spread over the genome (one across an N run), as
    (chromosome, start, string) -- the bounded sample of the workload the CPU legs scan."""
    out = []
    big = [c for c in pg.chroms if pg.chrom_sizes[c] > 4 * piece_bp] or pg.chroms
    for k in range(n_pieces):
        c = big[(k * 7) % len(big)]
        n = pg.chrom_sizes[c]
        if k == 0:
            a = max(n // 3 - piece_bp // 2, 0)          # straddles the start of the centromere-like N block
        else:
            a = int((0.05 + 0.9 * ((k * 0.37) % 1.0)) * max(n - piece_bp, 1))
        out.append((c, a, pg.decode_bytes(c, a, a + piece_bp).decode("ascii")))
    return out


def flatten_ref_sites(ref_sites):
    """Per-motif lists of [seq, start, score, strand] -> (counts, seq, start, score, strand) arrays."""
    counts = np.array([len(r) for r in ref_sites], dtype=np.int64)
    flat = [s for r in ref_sites for s in r]
    if not flat:
        return counts, np.zeros(0, np.int64), np.zeros(0, np.int64), np.zeros(0), np.zeros(0, np.int8)
    arr = np.array(flat, dtype=np.float64)
    return (counts, arr[:, 0].astype(np.int64), arr[:, 1].astype(np.int64), np.ascontiguousarray(arr[:, 2]),
            arr[:, 3].astype(np.int8))


def run_reference(args, rank, world):
    if rank != 0:
        return 0
    pwms = motif_workload()
    kind, fn = cpu_scanner()
    n_threads = os.cpu_count() or 1
    matrices = [p.tolist() for p in pwms]
    built, cut_src = shared_cutoffs(pwms, lambda: cutoffs_cpu(pwms))
    cutoffs = scan_cutoffs(built).tolist()
    names, sizes = genome_shape(args.scale)
    # The reference cannot hold the genome-wide result (2.6e8 sites x ~250 B of Python objects), so every
    # step scans a bounded sample: pieces of a synthetic chromosome of the same composition, generated on the
    # host (the reference arm touches no GPU code).  Throughput per bp does not depend on the sample size.
    from motifscan_b200 import synth
    rng = np.random.default_rng(GENOME_SEED)
    piece_bp = 1 << 20
    budget_s = 150.0
    per_step = max(budget_s / (args.steps + args.warmup), 2.0)
    probe = [bytes(synth.random_bases(rng, piece_bp, lower_frac=0.0)).decode()]
    t0 = time.perf_counter()
    fn(matrices, cutoffs, probe, 3, n_threads)
    rate = piece_bp / max(time.perf_counter() - t0, 1e-6)
    n_pieces = int(max(1, min(64, rate * per_step / piece_bp)))
    seqs = [bytes(synth.random_bases(rng, piece_bp, lower_frac=0.0)).decode() for _ in range(n_pieces)]
    k = len(seqs[0]) // 3
    seqs[0] = seqs[0][:k] + "N" * int(piece_bp * N_FRACTION) + seqs[0][k + int(piece_bp * N_FRACTION):]
    units = N_MOTIFS * sum(len(s) for s in seqs)
    for _ in range(args.warmup):
        fn(matrices, cutoffs, seqs, 3, n_threads)
    times = []
    for _ in range(args.steps):
        t0 = time.perf_counter()
        fn(matrices, cutoffs, seqs, 3, n_threads)
        times.append(time.perf_counter() - t0)
    ms = 1e3 * sum(times) / len(times)
    value = units / (ms / 1e3)
    sample = (f"{n_pieces} x {piece_bp} bp of synthetic chromosome of the workload's composition x all {N_MOTIFS} motifs per step "
              f"(the full genome is {sum(sizes)} bp: extrapolated linearly in motif*bp)")
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True,
        "scaling": "strong", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": workload_name(args.scale), "sample": sample, "n_threads": n_threads,
                   "cutoffs": f"p={P_VALUE} from {N_BACKGROUND} background samples, floored at 1e-6 ({cut_src})"},
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": n_threads, "kind": kind, "sample": sample},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line))
    return 0


# ------------------------------------------------------------------------------------------------
def measure_fp8_peak():
    """Dense e4m3 x e4m3 -> f16 tcgen05 peak of this GPU, measured live by bench_micro/fp8_peak (one CTA per
    SM, M = 128, N = 256, K = 32 MMAs back to back from shared memory, no epilogue): {"burst", "sustained"}."""
    exe = os.path.join(ROOT, "bench_micro", "fp8_peak")
    if not os.path.exists(exe):
        return None
    try:
        out = subprocess.run([exe], capture_output=True, text=True, timeout=120).stdout
        for line in out.splitlines():
            if line.startswith("{"):
                return json.loads(line)
    except Exception:
        return None
    return None


def compare_window(res, ref_sites):
    """GPU result of a window scan vs the CPU extension's per-motif lists: sites compared, motifs that differ."""
    counts, seq, start, score, strand = flatten_ref_sites(ref_sites)
    off = res.offsets
    bad = 0
    at = 0
    for m, c in enumerate(counts):
        a, b = off[m], off[m + 1]
        ok = (b - a == c and np.array_equal(res.seq_idx[a:b], seq[at:at + c]) and np.array_equal(res.start[a:b], start[at:at + c])
              and np.array_equal(res.strand[a:b], strand[at:at + c])
              and np.array_equal(np.ascontiguousarray(res.score[a:b]).view(np.uint64), score[at:at + c].view(np.uint64)))
        bad += 0 if ok else 1
        at += c
    return int(counts.sum()), bad


def site_sample(prefix, offsets, arrays, n=DUMP_SITES, seed=0):
    """A seeded sample of `n` sites of a motif-major result (all of them when there are fewer), in site order:
    `<prefix>_motif` from the per-motif `offsets`, and `<prefix>_<name>` for every per-site array of `arrays`."""
    total = int(offsets[-1])
    idx = np.sort(np.random.default_rng(seed).choice(total, size=min(n, total), replace=False))
    out = {prefix + "_motif": np.searchsorted(offsets, idx, side="right") - 1}
    out.update({f"{prefix}_{name}": a[idx] for name, a in arrays.items()})
    return out


def write_outputs(out_dir, arrays):
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), np.asarray(a, dtype=np.float64))


def run_ours(args, rank, local_rank, world):
    import torch
    from motifscan_b200 import _lib, engine
    from motifscan_b200.genome_scan import GenomeScanner
    from motifscan_b200.shard import gather_counts

    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device -- the scan path has no CPU fallback")
    torch.cuda.set_device(local_rank)
    dist = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("gloo")          # host-side barrier / gather only: NCCL is not on this path

    def barrier():
        torch.cuda.synchronize()
        if dist is not None:
            dist.barrier()

    def max_over_ranks(x):
        if dist is None:
            return float(x)
        t = torch.tensor([float(x)], dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t[0])

    def sum_over_ranks(x):
        if dist is None:
            return int(x)
        t = torch.tensor([int(x)], dtype=torch.int64)
        dist.all_reduce(t)
        return int(t[0])

    cpus = _lib.bind_thread_near(local_rank)     # before any pinned allocation: stay on this GPU's side of the host
    stream = torch.cuda.Stream()                 # the context launches on a stream torch can put events on
    ctx = engine.Context(local_rank, stream=stream.cuda_stream)
    pwms = motif_workload()
    pwm_lens = np.array([p.shape[1] for p in pwms], dtype=np.int64)
    if rank == 0:
        built, cut_src = shared_cutoffs(pwms, lambda: cutoffs_gpu(engine, ctx, pwms))
    else:
        built, cut_src = None, ""
    if dist is not None:
        t = torch.from_numpy(built.copy()) if rank == 0 else torch.zeros(N_MOTIFS, dtype=torch.float64)
        dist.broadcast(t, 0)
        built = t.numpy()
    cutoffs = scan_cutoffs(built)

    t0 = time.perf_counter()
    pg = make_genome(local_rank, args.scale)
    gen_s = time.perf_counter() - t0
    sizes = [pg.chrom_sizes[c] for c in pg.chroms]
    genome_bp = int(sum(sizes))
    units_total = N_MOTIFS * genome_bp                       # motif*bp per step, whole job
    adds_total = algorithmic_adds(pwm_lens, sizes)

    try:
        gpu_uuid = str(torch.cuda.get_device_properties(local_rank).uuid)
    except Exception:
        gpu_uuid = None
    fp8 = measure_fp8_peak() if rank == 0 else None

    # ---- leg 1: device-resident -------------------------------------------------------------------------
    unit_bp = int(min(UNIT_BP, max(MIN_UNIT_BP, genome_bp // world // 8)))
    gs = GenomeScanner(pg, pwms, cutoffs=cutoffs, contexts=[ctx], world=world, rank=rank, unit_bp=unit_bp, resident=True)
    share_bp = sum(u.owned_bp for u in gs.shares[0])
    gs_blocks = (gs.shares[0][0].block0, gs.shares[0][-1].block1)

    gather_ms = []

    def gather(counts):
        """The final host-side gather of the per-motif counts (on rank 0), inside every timed step."""
        t0 = time.perf_counter()
        total = gather_counts(counts, dist, dst=0)
        gather_ms.append(1e3 * (time.perf_counter() - t0))
        return total

    def resident_step():
        out = gs.scan(collect_sites=False, order_sites=True)
        return out, gather(out.counts)

    for _ in range(args.warmup):
        out, total_counts = resident_step()
    # rank 0 samples its GPU (NVML takes driver-wide locks: eight ranks polling at once slow each other's CUDA calls)
    sampler = ClockSampler(local_rank, gpu_uuid) if rank == 0 else None
    step_ms, phases, launches = [], {"prefilter": [], "exact": [], "order": []}, 0
    pre_launches = 0
    barrier()
    if sampler is not None:
        sampler.start()
    t_wall0 = time.perf_counter()
    for _ in range(args.steps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        out, total_counts = resident_step()
        e1.record(stream)
        e1.synchronize()
        step_ms.append(e0.elapsed_time(e1))
        st = gs.last_stats[0]
        for k in phases:
            phases[k].append(st[k])
        launches += st["launches"]
        pre_launches = st["prefilter_launches"]
    barrier()
    wall_ms = 1e3 * (time.perf_counter() - t_wall0) / args.steps
    # per-rank kernel time of a pass (the count gather makes every rank's step as long as the slowest rank's)
    mine = [sum(phases[k]) / len(phases[k]) for k in ("prefilter", "exact", "order")] + [float(share_bp)]
    if dist is not None:
        every = [torch.zeros(4, dtype=torch.float64) for _ in range(world)]
        dist.all_gather(every, torch.tensor(mine, dtype=torch.float64))
        per_rank = [[round(float(x), 3) for x in t] for t in every]
    else:
        per_rank = [[round(x, 3) for x in mine]]
    candidates = gs.last_stats[0]["candidates"]
    n_units = gs.last_stats[0]["units"]
    ms_per_step = max_over_ranks(sum(step_ms) / len(step_ms))
    wall_ms = max_over_ranks(wall_ms)
    n_sites_total = int(total_counts.sum()) if rank == 0 else 0
    gather_resident_ms = sum(gather_ms[-args.steps:]) / args.steps
    gs.close()

    # ---- leg 2: end to end (host planes in, host sites / counts out) -----------------------------------------
    gs = GenomeScanner(pg, pwms, cutoffs=cutoffs, contexts=[ctx], world=world, rank=rank, unit_bp=unit_bp, resident=False)
    h2d_bytes = sum(12 * (u.upload1 - u.block0) for u in gs.shares[0])

    e2e_phases = []

    def e2e_leg(collect_sites):
        sites_here, keep = 0, None
        for _ in range(min(args.warmup, 3)):
            out = gs.scan(collect_sites=collect_sites)
            gather(out.counts)
            out.close()
        barrier()
        t0 = time.perf_counter()
        for k in range(args.steps):
            out = gs.scan(collect_sites=collect_sites)        # returns when every unit's sites are in host memory
            total = gather(out.counts)
            sites_here = int(out.counts.sum())
            if k + 1 < args.steps or not collect_sites:
                out.close()
            else:
                keep = out
        barrier()
        ms = max_over_ranks(1e3 * (time.perf_counter() - t0) / args.steps)
        e2e_phases.append({k: gs.last_stats[0][k] for k in ("prefilter", "exact", "order")})
        return ms, sites_here, total, keep

    counts_ms, _, total_b, _ = e2e_leg(False)
    sites_ms, sites_here, total_c, kept = e2e_leg(True)
    clocks = sampler.stop() if sampler is not None else None
    d2h_sites = 12 * sites_here + 8 * (N_MOTIFS + 1) * len(gs.shares[0])
    d2h_counts = 8 * N_MOTIFS * len(gs.shares[0])
    if rank == 0:
        assert np.array_equal(total_b, total_counts) and np.array_equal(total_c, total_counts), "legs disagree on the per-motif counts"
    merge_ms = None
    outputs = {"genome_counts": total_counts} if rank == 0 else {}
    if kept is not None:
        t0 = time.perf_counter()
        n_merged = len(kept.start)                            # the lazy host-side gather of the site arrays
        merge_ms = 1e3 * (time.perf_counter() - t0)
        assert n_merged == sites_here
        if rank == 0 and args.dump_outputs:
            outputs.update(site_sample("genome_sites", kept.offsets, {"chrom": kept.chrom_idx, "start": kept.start,
                                                                     "score": kept.score, "strand": kept.strand}))
        kept.close()
    gs.close()
    h2d_all, d2h_all = sum_over_ranks(h2d_bytes), sum_over_ranks(d2h_sites)

    # ---- secondary block: configs[1] -------------------------------------------------------------------------
    c1 = configs1_block(args, engine, ctx, pg, pwms, cutoffs, torch, barrier, max_over_ranks, rank, world, local_rank)
    launches += c1.pop("_launches")
    outputs["configs1_counts"] = c1.pop("_counts")
    outputs.update(c1.pop("_sample"))
    launches_all = sum_over_ranks(launches)

    if rank == 0:
        peaks, peaks_src = load_peaks()
        pre_ms = sum(phases["prefilter"]) / len(phases["prefilter"])
        n_pre = max(pre_launches, 1)
        adds_rank = adds_total * share_bp / genome_bp          # this rank's share of the algorithmic work
        alg_flops = 8.0 * adds_rank                            # 4 L MACs per strand and window, 2 flop per MAC
        achieved = alg_flops / (pre_ms / 1e3) / 1e12
        bf16_sus = peaks.get("bf16_tflops_sustained") or peaks.get("bf16_tflops", 1590.0)
        peak_2bf16 = 2.0 * bf16_sus
        peak_fp8 = (fp8 or {}).get("sustained_tflops")
        peak = peak_fp8 or peak_2bf16
        sm_count = torch.cuda.get_device_properties(local_rank).multi_processor_count
        issue_peak = sm_count * 128 * peaks.get("sm_max_mhz", 1965.0) * 1e6 / 1e12
        traffic = None
        tpath = os.path.join(ROOT, "profiles", "prefilter_traffic.json")
        if os.path.exists(tpath):
            try:
                traffic = json.load(open(tpath)).get("dram_bytes_per_launch")
            except Exception:
                traffic = None
        # MMA work actually issued (mirrors ensure_tc_tables / prefilter_tc_kernel): motifs sorted by length, 128 per
        # 256-column tile, K steps of 32 = 8 bases up to the tile's longest motif; every 512-base position tile that
        # holds a live window runs 4 shifted 128-row MMAs per tile and K step (tiles inside N runs are skipped)
        lens_sorted = np.sort(pwm_lens)
        ksteps = sum(int(-(-int(lens_sorted[i:i + 128].max()) // 8)) for i in range(0, len(lens_sorted), 128))
        w = pg.work_prefix()
        u0, u1 = gs_blocks
        live_bases = float(w[u1] - w[u0]) - float(u1 - u0)
        issued = live_bases / 512.0 * 4 * ksteps * (2.0 * 128 * 256 * 32) / (pre_ms / 1e3) / 1e12
        roofline = {
            "bound": "tensor", "kernel": "prefilter_tc_kernel", "achieved": achieved, "peak": peak, "unit": "TFLOP/s",
            "issued": {"tflops": issued, "frac_of_peak": issued / peak, "k_steps_issued": ksteps,
                       "k_steps_needed": float(np.ceil(pwm_lens).sum() / 8.0 / 128.0),
                       "note": "MMA work issued on this rank's non-N bases: K padded to 8 bases per step, 256-column tiles"},
            "frac": achieved / peak,
            "peak_source": ("dense e4m3 tcgen05 peak measured live by bench_micro/fp8_peak (sustained over ~1 s)" if peak_fp8 else
                            f"2 x bf16_tflops_sustained from {peaks_src} (bench_micro/fp8_peak not built)"),
            "peak_measured_fp8": fp8, "peak_2x_bf16_sustained": peak_2bf16, "frac_of_2x_bf16_sustained": achieved / peak_2bf16,
            "algorithmic_flops_per_launch": alg_flops / n_pre, "launches_per_step": n_pre, "launch_ms": pre_ms / n_pre,
            "traffic": traffic,
            "note": "achieved = 8 x the reference's adds (unpadded one-hot x PWM contraction: 4 L MACs per strand and window, "
                    "2 flop per MAC) of this rank's share / summed prefilter launch time (CUDA events on the launch stream); "
                    "N windows are skipped on the device but counted as work, as the reference does them",
            "cuda_core_view": {"adds_per_s_T": adds_rank / (pre_ms / 1e3) / 1e12, "issue_peak_T": issue_peak},
            "hbm": {"algorithmic_bytes_per_step": 0.375 * share_bp + 16.0 * candidates,
                    "achieved_gbs": (0.375 * share_bp + 16.0 * candidates) / (pre_ms / 1e3) / 1e9,
                    "peak_gbs": peaks.get("hbm_gbs"), "note": "not the binding resource"},
        }
        cpu = None
        if world == 1 and not args.no_cpu:
            cpu = cpu_legs(engine, ctx, pg, pwms, cutoffs)
        line = {
            "metric": METRIC, "value": units_total / (ms_per_step / 1e3), "unit": UNIT, "n_gpus": world,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_per_step,
            "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
            "dtype": "e4m3 x e4m3 -> f16 tensor-core prefilter + f64 exact", "data": "synthetic",
            "config": {"workload": workload_name(args.scale), "n_motifs": N_MOTIFS, "genome_bp": genome_bp,
                       "strand": "both", "p_value": P_VALUE,
                       "cutoffs": f"p={P_VALUE} from {N_BACKGROUND} background samples, floored at 1e-6 ({cut_src})",
                       "l2": "inputs larger than L2 (0.375 B/bp packed genome share, >= 145 MB per rank, streamed once per step)",
                       "parallelism": f"position space cut into {world} contiguous share(s), one process per GPU, units of "
                                      f"{unit_bp} bp; gather = {N_MOTIFS} int64 counts per rank sent to rank 0 over gloo inside every step",
                       "genome_generation_s": gen_s,
                       "host_cores_rank0": f"{len(cpus)} NUMA-local cores" if cpus else "unbound"},
            "phase_ms": {k: sum(v) / len(v) for k, v in phases.items()},
            "wall_ms_per_step": wall_ms, "units_per_step_rank0": n_units, "count_gather_ms_rank0": gather_resident_ms,
            "per_rank_kernel_ms": {"columns": ["prefilter", "exact", "order", "share_bp"], "rows": per_rank},
            "sites_per_step": n_sites_total, "candidates_per_step_rank0": candidates,
            "e2e": {"value": units_total / (sites_ms / 1e3), "unit": UNIT, "ms_per_step": sites_ms, "steps": args.steps,
                    "h2d_bytes_per_step": h2d_all, "d2h_bytes_per_step": d2h_all,
                    "what": "GenomeScanner.scan: packed planes up from pinned host memory, ALL sites down to pinned host memory "
                            "(per-unit motif-major blocks), per-motif counts gathered over the ranks",
                    "host_merge_ms_rank0": merge_ms,
                    "kernel_phase_ms_rank0": {"counts_out": e2e_phases[0], "sites_out": e2e_phases[1]},
                    "variants": {
                        "sites_out": {"value": units_total / (sites_ms / 1e3), "ms_per_step": sites_ms, "d2h_bytes_per_step": d2h_all},
                        "counts_out": {"value": units_total / (counts_ms / 1e3), "ms_per_step": counts_ms,
                                       "d2h_bytes_per_step": sum_over_ranks_cached(d2h_counts, world)}}},
            "gpu_launches": int(launches_all),
            "gpu_launches_note": "own kernels over all timed steps (both workloads); a CUB sort / scan is counted as one launch",
            "roofline": roofline, "clocks": clocks, "configs1": c1,
        }
        if cpu is not None:
            line["cpu_baseline"] = cpu["all_cores"]
            line["cpu_baseline_1thread"] = cpu["one_thread"]
        if args.dump_outputs:
            write_outputs(args.dump_outputs, outputs)
        print(json.dumps(line))
    else:
        pass
    if dist is not None:
        dist.barrier()
        dist.destroy_process_group()
    return 0


def sum_over_ranks_cached(x, world):
    return int(x) * int(world)       # the same on every rank (one count vector per unit)


def cpu_legs(engine, ctx, pg, pwms, cutoffs):
    """cpu_baseline (reference extension, all host threads) and the 1-thread figure, on bounded samples of the
    genome; the GPU result of the same windows is compared site for site."""
    kind, fn = cpu_scanner()
    n_threads = os.cpu_count() or 1
    matrices = [p.tolist() for p in pwms]
    cut = cutoffs.tolist()
    piece_bp = 1 << 20
    probe = genome_samples(pg, 1, piece_bp)
    t0 = time.perf_counter()
    fn(matrices, cut, [probe[0][2]], 3, n_threads)
    rate = piece_bp / max(time.perf_counter() - t0, 1e-6)
    n_pieces = int(max(2, min(48, rate * 15.0 / piece_bp)))
    samples = genome_samples(pg, n_pieces, piece_bp)
    seqs = [s for _, _, s in samples]
    t0 = time.perf_counter()
    ref_sites = fn(matrices, cut, seqs, 3, n_threads)
    dt = time.perf_counter() - t0
    motifs = engine.MotifSet(ctx, pwms, cutoffs)
    sset = engine.SequenceSet(ctx, seqs)
    res = engine.scan(ctx, motifs, sset, 3)
    total, bad = compare_window(res, ref_sites)
    res.close(), sset.close(), motifs.close()
    bp = sum(len(s) for s in seqs)
    out = {"all_cores": {"value": N_MOTIFS * bp / dt, "unit": UNIT, "cores": n_threads, "kind": kind,
                         "sample": f"{n_pieces} windows of {piece_bp} bp of the genome (one across an N run) x all {N_MOTIFS} motifs, {dt:.1f} s",
                         "parity": {"sites_compared": total, "motifs_with_any_difference": bad,
                                    "bar": "identical (seq, start, strand) lists and bit-identical scores"}}}
    one = samples[1][2][:1 << 18]
    t0 = time.perf_counter()
    fn(matrices, cut, [one], 3, 1)
    dt1 = time.perf_counter() - t0
    out["one_thread"] = {"value": N_MOTIFS * len(one) / dt1, "unit": UNIT, "cores": 1, "kind": kind,
                         "sample": f"{len(one)} bp x all {N_MOTIFS} motifs, {dt1:.1f} s"}
    return out


def configs1_regions(pg, rank):
    """A rank's configs[1] peaks: the largest chromosome and the sorted starts of its REGION_BP-base windows."""
    chrom = max(pg.chroms, key=lambda c: pg.chrom_sizes[c])
    size = pg.chrom_sizes[chrom]
    rng = np.random.default_rng(50 + rank)
    n_regions = min(N_REGIONS, max(size // (2 * REGION_BP), 1))
    return chrom, np.sort(rng.integers(0, max(size - REGION_BP, 1), size=n_regions)).astype(np.int64)


def configs1_block(args, engine, ctx, pg, pwms, cutoffs, torch, barrier, max_over_ranks, rank, world, local_rank):
    """BASELINE.json configs[1] per GPU (weak-scaled, as in round 1): 50,000 peaks of 1 kb x 750 PWMs.
    `value`: the peaks' packed windows resident in HBM.  `e2e`: the product's resident-genome scanner path --
    region descriptors (20 B each) up, windows cut out of the resident chromosome on the device
    (msb_seqs_extract), scan, all sites down; consecutive steps are pipelined (MSB_SCAN_ASYNC: the copy of step
    k's sites overlaps step k + 1) and the timed region ends when the last step's sites are on the host."""
    import oracle  # noqa: F401  (CPU legs only, below)
    from motifscan_b200.genome import DeviceGenome
    chrom, starts = configs1_regions(pg, rank)
    size = pg.chrom_sizes[chrom]
    n_regions = len(starts)

    class One:                      # the largest chromosome, resident on this rank's GPU
        chroms, chrom_sizes = [chrom], {chrom: size}
    b0 = int(pg.block_off[pg.chrom_index[chrom]])
    nb = (size + 31) // 32
    resident = engine.SequenceSet.from_packed(ctx, [size], *pg.planes(b0, b0 + nb))
    idx = np.zeros(n_regions, dtype=np.int32)
    motifs = engine.MotifSet(ctx, pwms, cutoffs)
    units = N_MOTIFS * n_regions * REGION_BP
    windows = resident.extract(idx, starts, starts + REGION_BP)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")
    for _ in range(args.warmup):
        engine.scan_device(ctx, motifs, windows, 3)
    step_ms, launches = [], 0
    phase = {"prefilter": [], "exact": [], "order": []}
    barrier()
    for _ in range(args.steps):
        flush.fill_(1)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        n_sites = engine.scan_device(ctx, motifs, windows, 3)
        step_ms.append(1e3 * (time.perf_counter() - t0))
        t = ctx.timings()
        for k in phase:
            phase[k].append(t[k])
        launches += ctx.counters()["launches"]
    dev_ms = [phase["prefilter"][i] + phase["exact"][i] + phase["order"][i] for i in range(args.steps)]
    ms = max_over_ranks(sum(dev_ms) / len(dev_ms))
    counts = ctx.site_counts(N_MOTIFS)
    windows.close()

    # end to end: two scanner workers on this GPU -- two host threads, each with its own context (stream), motif set
    # and resident chromosome -- so that while one is on the host side of its step (descriptor upload, count read-backs,
    # result bookkeeping) the other one's kernels keep the device busy; within a worker consecutive steps are pipelined
    # with MSB_SCAN_ASYNC.  Every step is a complete scan of the 50,000 peaks from descriptors to host sites.
    n_workers = 2
    workers = [(ctx, motifs, resident)]
    for _ in range(n_workers - 1):
        c2 = engine.Context(local_rank)
        workers.append((c2, engine.MotifSet(c2, pwms, cutoffs), engine.SequenceSet.from_packed(c2, [size], *pg.planes(b0, b0 + nb))))

    def run_worker(k, n_steps, out, keep):
        c, mo, res_genome = workers[k]
        prev, n_launch = None, 0
        for _ in range(n_steps):
            w = res_genome.extract(idx, starts, starts + REGION_BP)
            res = engine.scan(c, mo, w, 3, async_=True, compact=True)
            n_launch += c.counters()["launches"] + 1
            w.close()
            if prev is not None:
                prev.wait()
                prev.close()
            prev = res
        prev.wait()
        out[k] = (prev.n_sites, n_launch, prev if keep else None)
        if not keep:
            prev.close()

    def run_all(n_steps, keep_last=False):
        """`keep_last`: worker 0 returns its last result unclosed (for --dump-outputs)."""
        per = [n_steps // n_workers + (1 if k < n_steps % n_workers else 0) for k in range(n_workers)]
        out = [None] * n_workers
        threads = [threading.Thread(target=run_worker, args=(k, per[k], out, keep_last and k == 0)) for k in range(n_workers) if per[k]]
        for t in threads:
            t.start()
        for t in threads:
            t.join()
        return [o for o in out if o is not None]
    run_all(2 * min(args.warmup, 3))
    barrier()
    e2e_steps = args.steps
    t0 = time.perf_counter()
    done = run_all(e2e_steps, keep_last=bool(args.dump_outputs) and rank == 0)
    e2e_ms = 1e3 * (time.perf_counter() - t0) / e2e_steps
    sites = done[0][0]
    launches += sum(o[1] for o in done)
    barrier()
    e2e_ms = max_over_ranks(e2e_ms)
    sample, last = {}, done[0][2]
    if last is not None:
        sample = site_sample("configs1_sites", last.offsets, {"region": last.seq_idx, "start": last.start,
                                                              "score": last.score, "strand": last.strand})
        last.close()
    for c2, mo2, rs2 in workers[1:]:
        mo2.close(), rs2.close(), c2.close()
    block = {
        "workload": f"configs[1]: {N_MOTIFS} PWMs x {n_regions} synthetic {REGION_BP} bp peaks per GPU (windows of the resident "
                    f"{chrom}), both strands, cutoffs p={P_VALUE}; weak-scaled over {world} GPU(s)",
        "value": world * units / (ms / 1e3), "unit": UNIT, "ms_per_step": ms,
        "timing": "sum of the three phases' CUDA-event times per step (prefilter + exact + order), L2 flushed between steps",
        "phase_ms": {k: sum(v) / len(v) for k, v in phase.items()}, "sites_per_step_rank0": int(n_sites),
        "e2e": {"value": world * units / (e2e_ms / 1e3), "unit": UNIT, "ms_per_step": e2e_ms,
                "h2d_bytes_per_step": world * 20 * n_regions, "d2h_bytes_per_step": world * (12 * int(sites) + 8 * (N_MOTIFS + 1)),
                "what": "region descriptors up, windows cut from the resident chromosome on the device, scan, all sites down (12 B each: "
                        "score + packed position and strand, MSB_SCAN_COMPACT); "
                        f"{len(done)} scanner worker(s) (host thread + context each) on the GPU, a worker's consecutive steps "
                        "pipelined with MSB_SCAN_ASYNC; "
                        "wall clock over all steps until the last sites are on the host", "steps": e2e_steps},
        "_launches": launches, "_counts": counts, "_sample": sample,
    }
    if world == 1 and not args.no_cpu:
        # Scanner-level CPU baseline (BASELINE.md section 3): the reference's Scanner.scan_motifs =
        # c_scan_motif + make_motif_sites + deduplicate_motif_sites (scanner.py:125-131), all host threads
        kind, fn = cpu_scanner()
        import oracle as orc
        n = 2000
        seqs = [pg.decode_bytes(chrom, int(a), int(a) + REGION_BP).decode() for a in starts[:n]]
        matrices = [p.tolist() for p in pwms]
        t0 = time.perf_counter()
        raw = fn(matrices, cutoffs.tolist(), seqs, 3, os.cpu_count() or 1)
        t_ext = time.perf_counter() - t0
        nested = orc.deduplicate_motif_sites(orc.make_motif_sites(raw, [int(a) for a in starts[:n]]), [p.shape[1] for p in pwms])
        t_all = time.perf_counter() - t0
        block["cpu_baseline_scanner_level"] = {
            "value": N_MOTIFS * n * REGION_BP / t_all, "extension_call_only": N_MOTIFS * n * REGION_BP / t_ext, "unit": UNIT,
            "cores": os.cpu_count() or 1, "kind": kind,
            "sample": f"first {n} peaks x all motifs: c_scan_motif {t_ext:.1f} s + make_motif_sites + deduplicate_motif_sites "
                      f"(the reference's Python, restated in oracle/) {t_all - t_ext:.1f} s",
            "sites_after_dedup": int(sum(len(c) for per in nested for c in per))}
    motifs.close()
    resident.close()
    return block


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline legs")
    ap.add_argument("--scale", type=float, default=1.0, help="shrink every chromosome by this factor (development only)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the last timed step's results to DIR/<name>.npy (float64)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the results of --impl ours")
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.impl == "reference":
        return run_reference(args, rank, world)
    return run_ours(args, rank, local_rank, world)


if __name__ == "__main__":
    sys.exit(main())
