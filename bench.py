#!/usr/bin/env python
"""bench.py -- headline benchmark of the depletion hot path (BASELINE.json: reads/s & FASTQ GB/s depleted at 1/2/4/8 B200).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--config c4|c2] [--pairs P] [--split]
                    [--dump-outputs DIR]

Default workload = BASELINE.json configs[3] (C4, the configuration the metric is quoted on; it fits one GPU):
100 M 2x150 pairs (2 x 33.1 GB of FASTQ) against a 50 M-id depletion set delivered as a one-column id list.
`--gpus N` is STRONG scaling: the SAME input is cut into N byte ranges per file (shards), one per rank.  One step =

    evidence   every rank turns ITS byte range of the id list into slot images grouped by table page (parse, hash,
    set_build  partition: done once per key across the box), one barrier, then every rank assembles the whole table from
               all ranks' lists, read over NVLink out of symmetric memory            -> the same exact id set in every HBM
               (--setbuild replicated: the id list itself is replicated -- peer pull or NCCL all-gather -- and
               ReadAlignment::from_txt runs on every rank over the whole list)
    filter     R1 and R2 shards: ONE pass of the fused parse -> probe -> compact kernel each, line phase speculated
    exchange   one all-gather of a few integers per file (own-range newline counts that prove the speculation, output
               sizes -> write offsets of the concatenation) and an all-reduce of the report counters

all of it inside the timed region, on device buffers (nothing goes through host `bytes`).  `phases_ms` breaks a step
down (CUDA events on the stream, max over ranks).  `--config c2` is round 1's workload (classifier, 10 M pairs per GPU,
weak scaling).

`value`  : reads/s with every input already resident in HBM (CUDA events on the launching stream).
`e2e`    : the same metric through the host-buffer C ABI calls (pinned host memory; H2D + D2H inside).
`roofline`: the fused kernel's algorithmic bytes (input + output bytes, SURVEY 8d) / its CUDA-event time.
`cpu_baseline`: the CPU oracle (a port structured like the reference: 1 thread for evidence, one thread per
            mate file) on a bounded sample, timed on this box's host cores.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True  # the benchmark leaves the tree it runs from as it found it

METRIC = "reads_per_s_depleted"
UNIT = "reads/s"
WORKLOAD_C2 = "classifier: synthetic 10M 2x150 pairs + Kraken2 reads/report, -T Chordata -D 9606, deplete"
WORKLOAD_C4 = "C4: 100M 2x150 pairs (66.2 GB FASTQ) with a 50M-id depletion set (TXT id list), sharded by byte range"


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            return json.load(f).get("hbm_gbs", 6650.0), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


class ClockSampler:
    """SM clock and throttle reasons sampled through NVML DURING the timed region (a thread polling every
    millisecond: the timed region of the device arm is only tens of milliseconds long)"""

    def __init__(self, device: int):
        self.device = device
        self.sm, self.reasons = [], set()
        self.mx = None
        self._stop = threading.Event()
        self._armed = threading.Event()
        self.th = None
        self.err = None

    def _run(self, nv, h):
        bits = {"hw_slowdown": nv.nvmlClocksEventReasonHwSlowdown,
                "hw_thermal_slowdown": nv.nvmlClocksEventReasonHwThermalSlowdown,
                "sw_thermal_slowdown": nv.nvmlClocksEventReasonSwThermalSlowdown,
                "sw_power_cap": nv.nvmlClocksEventReasonSwPowerCap}
        while True:
            try:
                sm = float(nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM))
                r = nv.nvmlDeviceGetCurrentClocksEventReasons(h)
                if self._armed.is_set():  # only samples of the timed region count
                    self.sm.append(sm)
                    for k, b in bits.items():
                        if r & b:
                            self.reasons.add(k)
            except Exception as e:  # noqa: BLE001
                self.err = repr(e)
                return
            if self._stop.wait(0.001):
                return

    def start(self):
        try:
            import pynvml as nv

            nv.nvmlInit()
            # NVML indexes physical devices: honour CUDA_VISIBLE_DEVICES when it is a plain index list
            vis = os.environ.get("CUDA_VISIBLE_DEVICES", "")
            idx = self.device
            if vis and all(x.strip().isdigit() for x in vis.split(",")):
                idx = int(vis.split(",")[self.device])
            h = nv.nvmlDeviceGetHandleByIndex(idx)
            self.mx = float(nv.nvmlDeviceGetMaxClockInfo(h, nv.NVML_CLOCK_SM))
            self.th = threading.Thread(target=self._run, args=(nv, h), daemon=True)
            self.th.start()
        except Exception as e:  # noqa: BLE001
            self.err = repr(e)

    def arm(self):
        """the timed region starts: NVML is initialised and the thread is polling already (start() costs tens of
        milliseconds on some ranks -- inside the timed region that skew lands in the first step's exchange)"""
        self._armed.set()

    def stop(self) -> dict:
        self._stop.set()
        if self.th:
            self.th.join(timeout=2)
        if not self.sm:
            return {"sm_mhz": None, "sm_max_mhz": self.mx, "reasons": [f"nvml unavailable: {self.err}"], "samples": 0}
        return {"sm_mhz": statistics.median(self.sm), "sm_max_mhz": self.mx, "reasons": sorted(self.reasons),
                "samples": len(self.sm)}


def bind_to_gpu_numa_node(device: int):
    """Best effort: run this rank on the CPUs next to its GPU (sysfs local_cpulist of the PCI device) so that
    the pinned host buffers of the end-to-end arm are allocated on the GPU's NUMA node.  Returns the cpulist."""
    try:
        import pynvml as nv

        nv.nvmlInit()
        vis = os.environ.get("CUDA_VISIBLE_DEVICES", "")
        idx = device
        if vis and all(x.strip().isdigit() for x in vis.split(",")):
            idx = int(vis.split(",")[device])
        bus = nv.nvmlDeviceGetPciInfo(nv.nvmlDeviceGetHandleByIndex(idx)).busId
        bus = bus.decode() if isinstance(bus, bytes) else bus
        dom, rest = bus.split(":", 1)
        path = f"/sys/bus/pci/devices/{dom[-4:].lower()}:{rest.lower()}/local_cpulist"
        cpulist = open(path).read().strip()
        cpus = set()
        for part in cpulist.split(","):
            a, _, b = part.partition("-")
            cpus.update(range(int(a), int(b or a) + 1))
        if cpus:
            os.sched_setaffinity(0, cpus)
        return cpulist
    except Exception as e:  # noqa: BLE001
        return f"unbound ({type(e).__name__})"


def mem_available_gb() -> float:
    """host memory this job may still take: MemAvailable, capped by the container's cgroup limit when there is one"""
    avail = 0.0
    try:
        with open("/proc/meminfo") as f:
            for line in f:
                if line.startswith("MemAvailable:"):
                    avail = int(line.split()[1]) / 1e6
    except OSError:
        pass
    for lim, cur in (("/sys/fs/cgroup/memory.max", "/sys/fs/cgroup/memory.current"),
                     ("/sys/fs/cgroup/memory/memory.limit_in_bytes", "/sys/fs/cgroup/memory/memory.usage_in_bytes")):
        try:
            v = open(lim).read().strip()
            if v != "max" and int(v) < (1 << 60):
                left = (int(v) - int(open(cur).read().strip())) / 1e9
                avail = min(avail, left) if avail else left
        except (OSError, ValueError):
            pass
    return avail


def taxids_for_config():
    """host stage: report -> taxid strings (-T Chordata -D 9606), the C++ state machine"""
    from scrubby_b200 import hostlib, synth

    return hostlib.get_taxids_from_report(synth.gen_kraken_report(5000), ["Chordata"], ["9606"])


# ------------------------------------------------------------------------------------------------ CPU arm
_CPU_SAMPLE = {}


def cpu_sample_run(pairs: int, config: str):
    """the CPU oracle on `pairs` pairs: evidence -> set on 1 thread, the two mate files on 2 threads
    (cleaner.rs:238-248).  Inputs are generated once (untimed).  Returns (seconds, reads, fastq_bytes)."""
    from oracle import oracle as orc
    from scrubby_b200 import synth

    key = (pairs, config)
    if key not in _CPU_SAMPLE:
        ev = synth.gen_kraken_reads(pairs).numpy() if config == "c2" else synth.gen_txt_ids(pairs).numpy()
        _CPU_SAMPLE[key] = (synth.gen_kraken_report(5000), ev, [synth.gen_fastq(pairs, m).numpy() for m in (1, 2)])
    rep, ev, fq = _CPU_SAMPLE[key]
    orc.lib()
    t0 = time.perf_counter()
    if config == "c2":
        tax = orc.taxids_from_report(rep, ["Chordata"], ["9606"])
        ids = orc.set_from_reads(ev, 0, tax)
    else:
        ids = orc.set_from_txt(ev)
    res = [None, None]

    def one(i):
        res[i] = orc.clean_fastq(fq[i], ids, False, want_bytes=False)

    th = [threading.Thread(target=one, args=(i,)) for i in range(2)]
    for t in th:
        t.start()
    for t in th:
        t.join()
    dt = time.perf_counter() - t0
    reads = res[0].reads_in + res[1].reads_in
    return dt, reads, int(fq[0].size + fq[1].size)


def cpu_sample_loop(pairs: int, config: str, min_seconds: float, max_reps: int = 200):
    """repeats the bounded sample until `min_seconds` of CPU work have been timed; returns the totals"""
    tot_t, tot_reads, tot_bytes, reps = 0.0, 0, 0, 0
    while reps < max_reps and (tot_t < min_seconds or reps == 0):
        dt, reads, nbytes = cpu_sample_run(pairs, config)
        tot_t += dt
        tot_reads += reads
        tot_bytes += nbytes
        reps += 1
    return tot_t, tot_reads, tot_bytes, reps


def cpu_sample_text(pairs: int, config: str, reps: int, nbytes: int) -> str:
    ev = f"{pairs} Kraken2 lines" if config == "c2" else f"the id list of its {pairs // 2} host reads"
    return (f"{reps} x ({pairs} pairs + {ev}) = {nbytes / 1e9:.2f} GB FASTQ; C oracle structured like the reference "
            "(evidence on 1 thread, one thread per mate file, SipHash-1-3 string set); the Rust reference itself "
            "cannot be built here (no cargo/rustc)")


def fused_traffic(config: str, n_gpus: int, split: bool):
    """DRAM bytes per launch of the fused kernel from the committed `ncu --set full` capture of this workload
    (profiles/fused_traffic.json, written by tools/ncu_summary.py); None when no capture matches."""
    p = os.path.join(ROOT, "profiles", "fused_traffic.json")
    try:
        with open(p) as f:
            j = json.load(f)
        if j.get("config") == config and j.get("n_gpus", 1) == n_gpus and bool(j.get("split")) == bool(split):
            return j["dram_bytes_read"] + j["dram_bytes_write"]
    except Exception:
        pass
    return None


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    sample = args.cpu_pairs
    times = []
    reps = 1
    for i in range(args.warmup + args.steps):
        # one step = the bounded sample repeated for about args.cpu_step_seconds of CPU work
        dt, reads, nbytes, reps = cpu_sample_loop(sample, args.config, args.cpu_step_seconds if i >= args.warmup else 0.0)
        if i >= args.warmup:
            times.append(dt)
    t = sum(times) / len(times)
    value = reads / t
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": t * 1e3, "higher_is_better": True,
        "scaling": "strong" if args.config == "c4" else "weak",
        "vs_baseline": None, "dtype": "u8", "data": "synthetic",
        "config": {"workload": WORKLOAD_C4 if args.config == "c4" else WORKLOAD_C2, "sample_pairs_per_step": sample * reps,
                   "outputs": "kept (reference-equivalent single output)", "fastq_gb_per_s": nbytes / t / 1e9},
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": 2, "kind": "port",
                         "sample": cpu_sample_text(sample, args.config, reps, nbytes) + " per step",
                         "cores_available": os.cpu_count()},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line))


# ------------------------------------------------------------------------------------------------ helpers
def fastq_record_at(offset: int, start: int = 0, read_len: int = 150):
    """(index of the record that holds byte `offset`, byte offset of that record's first byte) in the synthetic
    file whose first record is syn.{start}"""
    from scrubby_b200 import synth

    lo, hi = 0, 1
    while synth.fastq_size(hi, start, read_len) <= offset:
        hi *= 2
    while lo < hi:  # largest n with fastq_size(n) <= offset
        mid = (lo + hi + 1) // 2
        if synth.fastq_size(mid, start, read_len) <= offset:
            lo = mid
        else:
            hi = mid - 1
    return lo, synth.fastq_size(lo, start, read_len)


def gen_fastq_range(pairs: int, mate: int, a: int, b: int, device):
    """bytes [a, b) of the synthetic mate file of `pairs` records, as a device tensor padded by 16 readable bytes.
    The base / quality bytes of a record depend on the chunking of the generator, so a shard is not a byte-exact view
    of the single-GPU file -- ids, framing and sizes are (membership and record lengths only depend on the index)."""
    import torch

    from scrubby_b200 import synth

    i0, o0 = fastq_record_at(a)
    i1, _ = fastq_record_at(b - 1)
    i1 = min(pairs, i1 + 1)
    size = synth.fastq_size(i1 - i0, i0)
    buf = torch.empty(size + 16, dtype=torch.uint8, device=device)
    synth.gen_fastq(i1 - i0, mate, device=device, start=i0, out=buf)
    lo = a - o0
    if lo == 0:
        out = buf
    else:  # re-base so that the shard's first byte is 16-byte aligned (shard cuts are multiples of 16)
        out = torch.empty(b - a + 16, dtype=torch.uint8, device=device)
        out[: b - a] = buf[lo: lo + (b - a)]
        del buf
    out[b - a: b - a + 16] = 0
    return out


def gen_txt_full(pairs: int, device, chunk: int = 25_000_000):
    import torch

    from scrubby_b200 import synth

    parts = [synth.gen_txt_ids(min(chunk, pairs - s), device=device, start=s) for s in range(0, pairs, chunk)]
    return torch.cat(parts) if len(parts) > 1 else parts[0]


DUMP_WINDOWS, DUMP_WINDOW_BYTES, DUMP_BLOCK_BYTES, DUMP_SEED = 1024, 2048, 1 << 24, 0x5C2B


def dump_outputs(out_dir: str, torch, res, d_out, d_oth):
    """Writes what the last timed step handed its caller to `out_dir`, so that two builds can be compared output for
    output (the inputs depend only on the arguments):
      counts.npy                   float64 [file, (reads_in, reads_out, bytes kept, bytes removed)]
      kept_r{1,2}.npy              float32 [DUMP_WINDOWS, DUMP_WINDOW_BYTES]: the kept FASTQ bytes of windows at fixed,
                                   seeded offsets (the whole output is ~16.5 GB per file at the default size)
      kept_r{1,2}_block_sums.npy   float64: the byte sum of every DUMP_BLOCK_BYTES block of the kept output, so that every
                                   byte takes part in the comparison
      removed_r{1,2}*.npy          the same for the removed records (--split)
    At most four 8 MiB sample arrays plus the block sums: well below 64 MB."""
    import numpy as np

    os.makedirs(out_dir, exist_ok=True)

    def save(name, a):
        np.save(os.path.join(out_dir, name + ".npy"), a)

    save("counts", np.array([[r.reads_in, r.reads_out, r.n_written, r.n_other] for r in res], dtype=np.float64))
    for i, r in enumerate(res):
        for j, (kind, buf, n) in enumerate((("kept", d_out[i], r.n_written), ("removed", d_oth[i], r.n_other))):
            if buf is None:
                continue
            x = buf[:n]
            w = min(DUMP_WINDOW_BYTES, n)
            g = torch.Generator().manual_seed(DUMP_SEED + 2 * i + j)
            starts = torch.randint(0, n - w + 1, (DUMP_WINDOWS,), generator=g).sort().values
            save(f"{kind}_r{i + 1}", x[(starts[:, None] + torch.arange(w)).to(x.device)].float().cpu().numpy())
            # block by block: a sum with an int64 accumulator copies its input to int64 first
            sums = [x[a: a + DUMP_BLOCK_BYTES].sum(dtype=torch.int64) for a in range(0, n, DUMP_BLOCK_BYTES)]
            save(f"{kind}_r{i + 1}_block_sums", torch.stack(sums).double().cpu().numpy() if sums else np.zeros(0))


class Phases:
    """CUDA events on the launching stream at the phase boundaries of every timed step"""

    def __init__(self, torch, names):
        self.torch, self.names = torch, names
        self.steps = []
        self.cur = None

    def begin(self):
        self.cur = [self._ev()]

    def mark(self):
        self.cur.append(self._ev())

    def end(self):
        self.steps.append(self.cur)

    def _ev(self):
        e = self.torch.cuda.Event(enable_timing=True)
        e.record()
        return e

    def each_ms(self):
        return [[round(s[k].elapsed_time(s[k + 1]), 3) for k in range(len(self.names))] for s in self.steps]

    def mean_ms(self):
        out = {}
        for k, name in enumerate(self.names):
            out[name] = sum(s[k].elapsed_time(s[k + 1]) for s in self.steps) / max(1, len(self.steps))
        return out


# ------------------------------------------------------------------------------------------------ our arm
def run_ours(args):
    import torch
    import torch.distributed as dist

    from scrubby_b200 import api, synth
    from scrubby_b200 import dist as sdist

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    assert torch.cuda.is_available(), "bench.py needs a CUDA device (there is no CPU fallback)"
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    cpulist = bind_to_gpu_numa_node(local) if not args.no_bind else "unbound (--no-bind)"
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    D = dist if world > 1 else None

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    c4 = args.config == "c4"
    pairs = args.pairs or (100_000_000 if c4 else 10_000_000)
    ctx = api.Context(local)  # enqueues on torch's current stream
    t_setup = time.perf_counter()
    if c4:
        # ---- strong scaling: every file is ONE input cut into `world` byte ranges
        sizes = [synth.fastq_size(pairs)] * 2
        shards = [sdist.plan_shards(sz, world, halo=args.halo)[rank] for sz in sizes]
        d_r = [gen_fastq_range(pairs, m + 1, sh.start, sh.start + sh.buf_len, dev) for m, sh in enumerate(shards)]
        n_r = [sh.buf_len for sh in shards]
        own_bytes = sum(sh.own_len for sh in shards)
        ev_full = gen_txt_full(pairs, dev)
        ev_total = int(ev_full.numel())
        per = sdist.evidence_shard_len(ev_total, world)
        d_ev = torch.zeros(per + 16, dtype=torch.uint8, device=dev)
        mine = ev_full[rank * per: min(ev_total, (rank + 1) * per)]
        d_ev[: mine.numel()] = mine
        del mine
        # sharded set build (N > 1): this rank's byte range + a halo; every rank parses / hashes / partitions only its own
        # range, the page-sorted slot images are read over NVLink, every rank assembles the whole table
        sharded = None
        if world > 1 and args.setbuild in ("auto", "sharded"):
            try:
                evs = sdist.evidence_shard_with_halo(ev_full, rank, world, per)
                sharded = sdist.ShardedTxtSet(api, ctx, dist, ev_total, per, dev, direct=not args.pull_lists)
            except Exception as e:  # noqa: BLE001
                sys.stderr.write(f"[bench] rank {rank}: sharded set build unavailable ({type(e).__name__}: {e})\n")
                sharded = None
        d_ev_all = torch.empty(world * per + 16, dtype=torch.uint8, device=dev) if world > 1 else None
        # the evidence shards live in symmetric memory: every rank pulls the others' ranges over NVLink (no rendezvous
        # per step); --gather nccl keeps the NCCL all-gather
        peer_ev = None
        gather_how = "nccl all-gather"
        if world > 1 and args.gather == "pull" and (sharded is None or args.setbuild == "auto"):
            try:
                peer_ev = sdist.PeerFile(per, dist, dev)
                peer_ev.local[: per + 16].copy_(d_ev)
                peer_ev.publish(dist)
                gather_how = "peer pull (symmetric memory, NVLink P2P copies)"
            except Exception as e:  # noqa: BLE001
                sys.stderr.write(f"[bench] rank {rank}: symmetric memory unavailable ({type(e).__name__}: {e}); NCCL all-gather\n")
                peer_ev = None
        del ev_full
        # --setbuild auto (N > 1): the three ways to get the same set onto every rank are timed during setup (device
        # events, max over ranks, so every rank picks the same one) and the fastest runs in the timed steps:
        #   direct     sharded build, the page kernel reads the peers' lists in place over NVLink
        #   pulled     sharded build, the peers' lists are first copied over NVLink in bulk
        #   replicated the id list itself is replicated and every rank builds the whole set alone
        tuned = None
        if world > 1 and args.setbuild == "auto" and sharded is not None:
            def one_build(mode):
                if mode == "replicated":
                    ev = peer_ev.pull(ev_total, d_ev_all) if peer_ev is not None else \
                        sdist.replicate_file_dev(d_ev, per, ev_total, D, d_ev_all)
                    api.IdSet.from_txt(ctx, ev).free()
                else:
                    sharded.direct = mode == "direct"
                    got = sharded.build(*evs)
                    assert got is not None, "the id list of this workload takes the sharded build"
                    got.free()
            tuned = {}
            for mode in ("direct", "pulled", "replicated"):
                for _ in range(2):
                    one_build(mode)
                barrier()
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                for _ in range(3):
                    one_build(mode)
                e1.record()
                torch.cuda.synchronize()
                t_m = torch.tensor([e0.elapsed_time(e1) / 3], dtype=torch.float64, device=dev)
                dist.all_reduce(t_m, op=dist.ReduceOp.MAX)
                tuned[mode] = round(float(t_m[0]), 3)
            best = min(tuned, key=tuned.get)
            sys.stderr.write(f"[bench] rank {rank}: set build candidates (ms, max over ranks) {tuned} -> {best}\n")
            if best == "replicated":
                sharded = None
            else:
                sharded.direct = best == "direct"
        if sharded is not None:
            gather_how = ("sharded set build: page-sorted slot images " +
                          ("read from peer memory by the page kernel" if sharded.direct else "pulled over NVLink"))
        taxids = None
        n_k = per if world > 1 else ev_total
        # a depleted file is smaller than its input: the outputs are sized for the expected kept fraction + slack
        cap = [int(sh.buf_len * (1.0 if args.split else 0.56)) + (1 << 20) for sh in shards]
    else:
        # ---- weak scaling (round 1's workload): every rank owns its own 10M-pair shard and its Kraken2 lines
        start = rank * pairs
        taxids = taxids_for_config()
        d_r = [synth.gen_fastq(pairs, m, device=dev, start=start) for m in (1, 2)]
        d_ev = synth.gen_kraken_reads(pairs, device=dev, start=start)
        n_r = [int(t.numel()) for t in d_r]
        own_bytes = sum(n_r)
        n_k = int(d_ev.numel())
        shards = None
        cap = [n + 64 for n in n_r]
    d_out = [torch.empty(c, dtype=torch.uint8, device=dev) for c in cap]
    d_oth = [torch.empty(c, dtype=torch.uint8, device=dev) for c in cap] if args.split else [None, None]
    torch.cuda.synchronize()
    t_setup = time.perf_counter() - t_setup

    names = ["evidence", "set_build", "filter", "exchange"] if c4 else ["set_build", "filter"]
    ph = Phases(torch, names)

    def step_dev(timed=False):
        """-> ((reads_in, reads_out, bytes written) of the WHOLE job, paths, one_pass, this rank's result per file)"""
        if timed:
            ph.begin()
        if c4:
            ids = None
            if sharded is not None:  # evidence = partition of the own range + barrier + offset tables; set_build = assembly
                ids = sharded.build(*evs, mark=ph.mark if timed else None)
                assert ids is not None, "the id list of this workload takes the sharded build"
            else:  # evidence = replication of the id list; set_build = from_txt over the whole list
                if peer_ev is not None:
                    ev = peer_ev.pull(ev_total, d_ev_all)
                else:
                    ev = sdist.replicate_file_dev(d_ev, per, ev_total, D, d_ev_all)
                if timed:
                    ph.mark()
                ids = api.IdSet.from_txt(ctx, ev)
            if timed:
                ph.mark()
            if world == 1:
                r = [api.clean_fastq_dev(ctx, ids, d_r[i], n_r[i], d_out[i], d_oth[i]) for i in range(2)]
                if timed:
                    ph.mark()
                tot = [sum(x.reads_in for x in r), sum(x.reads_out for x in r), sum(x.n_written for x in r)]
                paths = [x.path for x in r]
                one_pass = True
            else:
                jobs = [(d_r[i], shards[i], d_out[i], d_oth[i]) for i in range(2)]
                r = rs = sdist.clean_files_sharded_dev(api, ctx, ids, jobs, D)
                if timed:
                    ph.mark()
                # report counters: NCCL all-reduce (the all-gather above already carries them; this is the
                # reduction the report writer consumes)
                cnt = torch.tensor([sum(x.n_written for x in rs), 0, 0], dtype=torch.int64, device=dev)
                dist.all_reduce(cnt, op=dist.ReduceOp.SUM)
                tot = [sum(x.reads_in for x in rs), sum(x.reads_out for x in rs), int(cnt[0])]
                paths = [x.path for x in rs]
                one_pass = all(x.one_pass for x in rs)
            if timed:
                ph.mark()
        else:
            ids = api.IdSet.from_reads(ctx, d_ev, 0, taxids)
            if timed:
                ph.mark()
            r = [api.clean_fastq_dev(ctx, ids, d_r[i], n_r[i], d_out[i], d_oth[i]) for i in range(2)]
            if timed:
                ph.mark()
            tot = [sum(x.reads_in for x in r), sum(x.reads_out for x in r), sum(x.n_written for x in r)]
            paths = [x.path for x in r]
            one_pass = True
        ids.free()
        if timed:
            ph.end()
        return tot, paths, one_pass, r

    # ---- device-resident arm
    ctx.set_profiling(False)
    for _ in range(args.warmup):
        tot, paths, one_pass, _ = step_dev()
    assert all(p == 1 for p in paths), "the fused kernel must be the path that runs"
    assert one_pass, "the one-pass (speculated line phase) protocol must hold on canonical input"
    ctx.set_profiling(True)
    ctx.fused_stats()
    sampler = ClockSampler(local)
    if not os.environ.get("SGPU_BENCH_NOSAMPLER"):
        sampler.start()
    barrier()
    sampler.arm()
    l0 = ctx.launches
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.profiler.start()  # `ncu --profile-from-start off` lists exactly the timed launches
    e0.record()
    for _ in range(args.steps):
        tot, paths, one_pass, res = step_dev(True)
    e1.record()
    barrier()
    torch.cuda.profiler.stop()
    clocks = sampler.stop()
    ms = e0.elapsed_time(e1) / args.steps
    launches = (ctx.launches - l0)
    f_ms, f_n, f_bytes = ctx.fused_stats()
    ctx.set_profiling(False)
    if args.dump_outputs:  # before the end-to-end arm, which frees the output buffers
        dump_outputs(args.dump_outputs, torch, res, d_out, d_oth)
    phases = ph.mean_ms()
    sys.stderr.write(f"[bench] rank {rank}: phases of every timed step (ms; {', '.join(names)}) {ph.each_ms()}\n")
    if c4:
        reads_job, kept_job, written_job = tot  # whole job (summed over ranks by the exchange)
    else:
        reads_job, kept_job, written_job = tot  # this rank; summed below
    assert (reads_job == 2 * pairs) if (c4 or world == 1) else True

    # ---- end-to-end arm: pinned host buffers through the host-pointer C ABI (H2D + D2H inside)
    if args.e2e_steps > 0:
        e2e = run_e2e(args, torch, dist, D, api, sdist, ctx, dev, world, rank, c4, pairs, shards, d_r, n_r, d_ev, n_k,
                      taxids, cap, barrier, (per, ev_total) if c4 else None, written_job, d_out, d_oth,
                      (sharded, evs) if (c4 and sharded is not None) else None)
    else:
        e2e = {"t": float("nan"), "h2d": 0, "d2h": 0, "steps": 0, "each": [], "warm": [], "pairs": 0, "scale": 1.0,
               "mem_gb": round(mem_available_gb(), 1), "note": "skipped (--e2e-steps 0)", "h2d_rank": 0, "d2h_rank": 0}

    # ---- max over ranks
    ms_t = torch.tensor([ms, e2e["t"] * 1e3 if e2e["steps"] else 0.0, f_ms / max(f_n, 1)] + [phases[n] for n in names], dtype=torch.float64,
                        device=dev)
    cnt = torch.tensor([reads_job, kept_job, own_bytes, launches], dtype=torch.int64, device=dev)
    fmin = torch.tensor([f_bytes / (f_ms * 1e-3) / 1e9 if f_ms > 0 else 0.0], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(ms_t, op=dist.ReduceOp.MAX)
        dist.all_reduce(fmin, op=dist.ReduceOp.MIN)
        dist.all_reduce(cnt, op=dist.ReduceOp.SUM)  # report counters, NCCL allreduce
    ms, e2e_ms, f_avg_max = float(ms_t[0]), float(ms_t[1]), float(ms_t[2])
    phases_max = {n: round(float(ms_t[3 + k]), 4) for k, n in enumerate(names)}
    if c4:
        reads_all, kept_all = reads_job, kept_job
    else:
        reads_all, kept_all = int(cnt[0]), int(cnt[1])
    bytes_all, launches_all = int(cnt[2]), int(cnt[3])

    if rank == 0:
        peak, peak_src = peaks()
        achieved = f_bytes / (f_ms * 1e-3) / 1e9 if f_ms > 0 else 0.0
        cpu_sample_run(args.cpu_pairs, args.config)  # warm the page cache / allocator
        dt, creads, cbytes, reps = cpu_sample_loop(args.cpu_pairs, args.config, args.cpu_seconds)
        cpu = {"value": creads / dt, "unit": UNIT, "cores": 2, "kind": "port",
               "sample": cpu_sample_text(args.cpu_pairs, args.config, reps, cbytes) + f", {dt:.2f} s",
               "cores_available": os.cpu_count(), "fastq_gb_per_s": cbytes / dt / 1e9}
        if c4:
            workload = WORKLOAD_C4 if pairs == 100_000_000 else f"C4 shape at {pairs} 2x150 pairs + the id list of its host reads"
        else:
            workload = WORKLOAD_C2 if pairs == 10_000_000 else f"classifier: synthetic {pairs} 2x150 pairs + Kraken2 reads/report"
        line = {
            "metric": METRIC, "value": reads_all / (ms * 1e-3), "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True, "scaling": "strong" if c4 else "weak",
            "vs_baseline": None, "dtype": "u8", "data": "synthetic",
            "config": {
                "workload": workload, "pairs_total": pairs if c4 else pairs * world,
                "fastq_bytes_total": bytes_all, "evidence_bytes": ev_total if c4 else n_k * world,
                "outputs": "kept+removed" if args.split else "kept (reference-equivalent single output)",
                "fraction_kept": kept_all / reads_all,
                "parallelism": (f"byte-range shards x{world}; " +
                                ("id set built once on the GPU; " if world == 1 else
                                 f"{gather_how}, the whole table assembled on every rank; " if sharded is not None else
                                 f"id list replicated by {gather_how}, set built on every rank; ") +
                                "one-pass filter with speculated line phase; counters all-reduced (NCCL)") if c4
                else f"chunk-sharded x{world} (co-partitioned evidence, no collective in the step)",
                "setbuild_candidates_ms": tuned if c4 else None,
                "host_cpus_rank0": cpulist, "setup_s_rank0": round(t_setup, 1),
                "l2": "inputs (>= 8 GB per GPU) are far larger than the 126 MB L2; no explicit flush",
                "fastq_gb_per_s": bytes_all / (ms * 1e-3) / 1e9,
            },
            "phases_ms": phases_max,
            "e2e": {"value": (reads_all / (e2e_ms * 1e-3) * e2e["scale"]) if e2e["steps"] else None, "unit": UNIT, "h2d_bytes_per_step": e2e["h2d"],
                    "d2h_bytes_per_step": e2e["d2h"], "ms_per_step": e2e_ms, "steps": e2e["steps"],
                    "ms_each_rank0": e2e["each"], "warmup_ms_each_rank0": e2e["warm"], "pairs": e2e["pairs"],
                    "h2d_gb_per_s_rank0": (e2e["h2d_rank"] / e2e["t"] / 1e9) if e2e["steps"] else None,
                    "d2h_gb_per_s_rank0": (e2e["d2h_rank"] / e2e["t"] / 1e9) if e2e["steps"] else None,
                    "host_mem_available_gb": e2e["mem_gb"], "note": e2e["note"],
                    "host_copy_ceiling_all_ranks": e2e.get("ceiling"),
                    "timing": "host wall clock around the host-buffer C ABI calls of one step on pinned host "
                              "buffers (evidence upload + set build + both mate files), stream synchronised, max over ranks"},
            "gpu_launches": launches_all,
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s",
                         "frac": achieved / peak if peak else None, "traffic": fused_traffic(args.config, world, args.split),
                         "kernel": "fastq_fused_kernel", "launches": f_n, "avg_ms": f_ms / f_n if f_n else None,
                         "algorithmic_bytes_per_launch": f_bytes / f_n if f_n else None, "peak_source": peak_src,
                         "share_of_step": f_ms / (ms * args.steps) if ms else None,
                         "achieved_min_over_ranks": float(fmin[0]), "avg_ms_max_over_ranks": f_avg_max},
            "cpu_baseline": cpu,
            "clocks": clocks,
        }
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


def host_copy_ceiling(torch, dist, dev, world, h_src, h_dst, n_bytes: int, reps: int = 3):
    """aggregate pinned-memory copy rate of the box with every rank copying at once (GB/s: H2D alone, D2H alone, both
    directions together) -- the ceiling of the end-to-end arm, whatever the kernels do"""
    n = min(n_bytes, int(h_src.numel()), int(h_dst.numel()), 4 << 30)
    d = torch.empty(n, dtype=torch.uint8, device=dev)
    s2 = torch.cuda.Stream(device=dev)
    out = []
    for mode in ("h2d", "d2h", "both"):
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        t0 = time.perf_counter()
        for _ in range(reps):
            if mode in ("h2d", "both"):
                d.copy_(h_src[:n], non_blocking=True)
            if mode in ("d2h", "both"):
                with torch.cuda.stream(s2):
                    h_dst[:n].copy_(d, non_blocking=True)
        torch.cuda.synchronize()
        dt = time.perf_counter() - t0
        t = torch.tensor([dt], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        moved = n * reps * (2 if mode == "both" else 1) * world
        out.append(round(moved / float(t[0]) / 1e9, 1))
    del d
    return {"h2d_gb_per_s": out[0], "d2h_gb_per_s": out[1], "both_gb_per_s": out[2], "bytes_per_rank_and_copy": n}


def run_e2e(args, torch, dist, D, api, sdist, ctx, dev, world, rank, c4, pairs, shards, d_r, n_r, d_ev, n_k, taxids, cap,
            barrier, evinfo, written_job, d_out, d_oth, sharded_ev=None):
    """the step through HOST buffers: inputs in pinned host memory, outputs into pinned host memory"""
    # the pinned copies of every rank's inputs and outputs must fit the host (with room to spare: pinned pages cannot be
    # reclaimed and an exhausted box kills the job).  A single-GPU run that does not fit runs on a prefix of whole
    # records (a rate is still a rate; `pairs` / `note` say so); a multi-GPU run that does not fit is not run.
    need_gb = (sum(n_r) + sum(cap) + n_k) / 1e9
    avail = mem_available_gb()
    if world > 1:
        a_t = torch.tensor([avail], dtype=torch.float64, device=dev)
        dist.all_reduce(a_t, op=dist.ReduceOp.MIN)
        avail = float(a_t[0])
    sys.stderr.write(f"[bench] rank {rank}: e2e needs {need_gb:.1f} GB of pinned host memory per rank x {world}, "
                     f"{avail:.0f} GB available\n")
    note = "full workload"
    frac = 1.0
    if avail and need_gb * world > 0.55 * avail:
        if world > 1:
            return {"t": float("nan"), "h2d": 0, "d2h": 0, "steps": 0, "each": [], "warm": [], "pairs": 0, "scale": 1.0,
                    "mem_gb": round(avail, 1), "h2d_rank": 0, "d2h_rank": 0,
                    "note": f"not run: {need_gb * world:.0f} GB of pinned host memory needed, {avail:.0f} GB available"}
        frac = max(0.05, 0.55 * avail / need_gb)
        note = f"host memory: {avail:.0f} GB available, {need_gb:.0f} GB needed -> the first {frac:.2f} of every file"
    e_n = []
    for i in range(2):
        if frac >= 1.0:
            e_n.append(n_r[i])
        else:  # cut at a record boundary: a prefix of whole records is a valid file
            k = int(n_r[i] * frac)
            tail = bytes(d_r[i][k: k + 4096].cpu().numpy())
            at = tail.find(b"\n@syn.")
            e_n.append(k + at + 1)
    h_r = [torch.empty(n + 16, dtype=torch.uint8, pin_memory=True) for n in e_n]
    h_k = torch.empty(n_k + 16, dtype=torch.uint8, pin_memory=True)
    for i in range(2):
        h_r[i][: e_n[i]].copy_(d_r[i][: e_n[i]])
    h_k[:n_k].copy_(d_ev[:n_k])
    # the device-resident arm is over: its buffers go back to the driver (the host-buffer path stages on the device)
    d_r.clear()
    d_out.clear()
    d_oth.clear()
    if not (c4 and world > 1):
        del d_ev
    torch.cuda.empty_cache()
    e_cap = [int(c * min(1.0, frac * 1.05)) + (1 << 20) for c in cap]
    h_out = [torch.empty(c, dtype=torch.uint8, pin_memory=True) for c in e_cap]
    h_oth = [torch.empty(c, dtype=torch.uint8, pin_memory=True) for c in e_cap] if args.split else [None, None]
    torch.cuda.synchronize()
    sys.stderr.write(f"[bench] rank {rank}: pinned buffers ready, {mem_available_gb():.0f} GB of host memory left\n")
    if c4 and world > 1:
        per, ev_total = evinfo
        d_ev2 = torch.empty(per + 16, dtype=torch.uint8, device=dev)
        d_ev_all = torch.empty(world * per + 16, dtype=torch.uint8, device=dev)
        if sharded_ev is not None:  # the rank's id-list range + halo from pinned host memory, then the sharded build
            sharded, evs = sharded_ev
            h_evs = torch.empty(evs[0].numel(), dtype=torch.uint8, pin_memory=True)
            h_evs.copy_(evs[0])
            d_evs = torch.empty_like(evs[0])

    dbg = os.environ.get("SGPU_BENCH_DEBUG")

    def step_host():
        if dbg:
            sys.stderr.write(f"[bench] rank {rank}: host step, {mem_available_gb():.0f} GB of host memory left\n")
        if c4 and world > 1 and sharded_ev is not None:
            d_evs.copy_(h_evs, non_blocking=True)
            ids = sharded.build(d_evs, *evs[1:])
            assert ids is not None, "the synthetic id list is inline-only: the sharded build must not decline it"
        elif c4 and world > 1:
            d_ev2[:per].copy_(h_k[:per], non_blocking=True)
            ev = sdist.replicate_file_dev(d_ev2, per, ev_total, D, d_ev_all)
            ids = api.IdSet.from_txt(ctx, ev)
        elif c4:
            ids = api.IdSet.from_txt(ctx, h_k[:n_k])
            r = [api.clean_fastq_host(ctx, ids, h_r[i], e_n[i], h_out[i], h_oth[i]) for i in range(2)]
        else:
            ids = api.IdSet.from_reads(ctx, h_k[:n_k], 0, taxids)
            r = [api.clean_fastq_host(ctx, ids, h_r[i], e_n[i], h_out[i], h_oth[i]) for i in range(2)]
        if c4 and world > 1:
            r = sdist.clean_files_sharded_host(api, ctx, ids, [(h_r[i], shards[i], h_out[i], h_oth[i]) for i in range(2)], D)
            assert all(x.one_pass for x in r), "speculated line phase refuted on canonical input"
        ids.free()
        return r

    e2e_steps = max(1, min(args.steps, args.e2e_steps))
    # warm-up: first touches of the pinned buffers, the chunk buffers of the pipeline, the memory pool.  The host side
    # settles by TIME rather than by step count: at least three steps, then until a step is within 15 % of the fastest
    # seen, at most eight
    warm_each = []
    while len(warm_each) < 8:
        t0 = time.perf_counter()
        rh = step_host()
        torch.cuda.synchronize()
        warm_each.append(time.perf_counter() - t0)
        if len(warm_each) >= 3 and warm_each[-1] <= 1.15 * min(warm_each) and warm_each[-2] <= 1.15 * min(warm_each):
            break
    if world > 1:  # every rank leaves the warm-up together
        w_t = torch.tensor([len(warm_each)], dtype=torch.int64, device=dev)
        dist.all_reduce(w_t, op=dist.ReduceOp.MAX)
        for _ in range(int(w_t) - len(warm_each)):
            rh = step_host()
    barrier()
    e2e_each = []
    for _ in range(e2e_steps):
        t0 = time.perf_counter()
        rh = step_host()
        torch.cuda.synchronize()
        e2e_each.append(time.perf_counter() - t0)
    t_e2e = sum(e2e_each) / e2e_steps
    d2h = sum(r.n_written + r.n_other for r in rh)
    h2d = sum(e_n) + n_k
    reads_e2e = sum(r.reads_in for r in rh)
    tot = torch.tensor([reads_e2e], dtype=torch.int64, device=dev)
    if world > 1 and not c4:  # (the sharded C4 results already carry the whole file's counters)
        dist.all_reduce(tot, op=dist.ReduceOp.SUM)
    io = torch.tensor([h2d, d2h], dtype=torch.int64, device=dev)
    if world > 1:
        dist.all_reduce(io, op=dist.ReduceOp.SUM)  # bytes of the whole job per step (every rank moves its own shard)
    h2d_rank, d2h_rank = h2d, d2h
    h2d, d2h = int(io[0]), int(io[1])
    total_reads = 2 * pairs if c4 else 2 * pairs * world
    scale = int(tot[0]) / total_reads  # 1.0 unless the arm ran on a prefix
    if frac >= 1.0 and world == 1:
        assert sum(r.n_written for r in rh) == written_job, "host and device arms disagree"
    ceiling = host_copy_ceiling(torch, dist, dev, world, h_r[0], h_out[0], int(h_out[0].numel()))
    return {"ceiling": ceiling, "t": t_e2e, "h2d": h2d, "d2h": d2h, "steps": e2e_steps, "each": [round(x * 1e3, 2) for x in e2e_each],
            "warm": [round(x * 1e3, 2) for x in warm_each], "pairs": int(tot[0]) // 2, "scale": scale,
            "mem_gb": round(avail, 1), "note": note, "h2d_rank": h2d_rank, "d2h_rank": d2h_rank}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10, help="timed steps (at least 1)")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", default="c4", choices=["c4", "c2"],
                    help="c4: 100M pairs + 50M-id list, strong scaling (BASELINE configs[3]); c2: classifier, 10M pairs per GPU")
    ap.add_argument("--pairs", type=int, default=0, help="c4: pairs of the whole job (default 100M); c2: pairs per GPU (10M)")
    ap.add_argument("--halo", type=int, default=1 << 20, help="c4: bytes of halo after a shard's own range")
    ap.add_argument("--setbuild", default="auto", choices=["auto", "sharded", "replicated"],
                    help="c4, N > 1: every rank partitions its own byte range of the id list and all ranks assemble the table "
                         "from everybody's lists (sharded), or the id list is replicated and every rank builds alone")
    ap.add_argument("--pull-lists", action="store_true", help="sharded set build: pull the other ranks' lists into local "
                                                              "buffers instead of reading them from peer memory")
    ap.add_argument("--gather", default="pull", choices=["pull", "nccl"],
                    help="c4, N > 1: how the id list's byte ranges reach every rank (peer pull over NVLink, or NCCL all-gather)")
    ap.add_argument("--cpu-pairs", type=int, default=1_000_000, help="bounded CPU-baseline sample")
    ap.add_argument("--cpu-seconds", type=float, default=10.0, help="CPU work timed for cpu_baseline")
    ap.add_argument("--cpu-step-seconds", type=float, default=3.0, help="--impl reference: CPU work per step")
    ap.add_argument("--e2e-steps", type=int, default=3)
    ap.add_argument("--split", action="store_true", help="also write the removed records (kept + removed)")
    ap.add_argument("--no-bind", action="store_true", help="do not bind the rank to its GPU's NUMA-local CPUs")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="one process only: write the outputs of the last timed step to DIR/*.npy (see dump_outputs)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl != "ours" or int(os.environ.get("WORLD_SIZE", "1")) > 1):
        ap.error("--dump-outputs needs --impl ours in a single process")
    if args.warmup < 3 and args.impl == "ours":
        args.warmup = 3
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
