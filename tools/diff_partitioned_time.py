"""Time and memory of the hash-partitioned diff (dist.diff_partitioned) beside the replicated one (dist.diff_sharded) on
ONE GPU (bench.py is not involved).

    python tools/diff_partitioned_time.py [--records 5000000] [--parts 8] [--reps 3]

Input: C5-shaped -- both mates of --records 2x150 records and their clean outputs (a third of the ids in the set).
1. diff_sharded vs diff_partitioned end to end at N = 1 (no process group), alternated, results compared with sgpu_diff;
2. the partitioned algebra per phase on --parts virtual ranks of this device (dist.plan_shards ranges; the exchange is
   the concatenation of each destination's parts): route, exchange, O_r build, probe, final merge -- per rank (the
   slowest rank's phase sum is what N GPUs would wait for) -- beside the replicated O build diff_sharded does on every
   rank; route GB/s (input bytes over the route call) and probe-lines M lines/s;
3. device memory per rank: torch.cuda.mem_get_info deltas (the library allocates outside torch's caching allocator)
   while the replicated O and then one O_r are built and held, and the sets' own table + arena bytes;
4. probe-lines on a set built from ONE partition's keys (P = --parts) against a set of the same size built from
   unpartitioned ids: equal times show that the owner bits do not skew the owner's page load.
Times are host clocks around synchronised calls; the card's name and power limit are read in the same run."""
import argparse
import heapq
import os
import statistics
import subprocess
import sys
import tempfile
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch

from scrubby_b200 import api, synth
from scrubby_b200.dist import GpuOps, diff_partitioned, diff_sharded, plan_shards

ap = argparse.ArgumentParser()
ap.add_argument("--records", type=int, default=5_000_000)
ap.add_argument("--parts", type=int, default=8)
ap.add_argument("--reps", type=int, default=3)
a = ap.parse_args()

smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                     capture_output=True, text=True).stdout.strip()
print(f"card: {smi}", flush=True)
dev = torch.device("cuda", 0)
ctx = api.Context(0)
ops = GpuOps(ctx)
n, P = a.records, a.parts


def now():
    torch.cuda.synchronize(dev)
    return time.perf_counter()


# ---- input
gs = api.IdSet.from_ids(ctx, [b"syn.%d" % i for i in range(0, n, 3)])
pairs = []
for m in (1, 2):
    fq = synth.gen_fastq(n, m).numpy().tobytes()
    pairs.append((fq, api.clean_fastq(ctx, gs, fq, want_other=False).written))
del gs
in_bytes = sum(len(f) for f, _ in pairs)
print(f"input: 2 mates x {n} records, {in_bytes / 1e9:.2f} GB in + {sum(len(o) for _, o in pairs) / 1e9:.2f} GB out",
      flush=True)
w = api.diff(ctx, pairs)
want = (w[0], w[1], w[2], w[3].sorted_ids())
del w

# ---- 1. end to end at N = 1
times = {"diff_sharded": [], "diff_partitioned": []}
for rep in range(a.reps + 1):
    for name, fn in (("diff_sharded", diff_sharded), ("diff_partitioned", diff_partitioned)):
        t0 = now()
        r = fn(ops, pairs)
        t = now() - t0
        assert (r.reads_in, r.reads_out, r.difference, r.diff_ids) == want, name
        if rep:
            times[name].append(t)
for name, ts in times.items():
    print(f"N=1 {name}: median {statistics.median(ts) * 1e3:.1f} ms of {['%.1f' % (x * 1e3) for x in ts]} "
          "(host bytes -> device, ids, sets, sorted dump; results equal sgpu_diff)", flush=True)

# ---- 2. phases on P virtual ranks


def shard_bufs(buf):
    out = []
    for sh in plan_shards(len(buf), P, 1 << 20):
        d = ops.upload(buf[sh.start: sh.start + sh.buf_len]) if sh.own_len else None
        out.append((sh, d, buf[: sh.start].count(b"\n")))
    return out


phase = {k: [0.0] * P for k in ("route", "exchange", "O_r build", "probe", "merge")}
route_bytes = route_t = probe_lines_n = probe_t = 0.0
d_sets = [api.IdSet.empty(ctx) for _ in range(P)]
repl_build = 0.0
for fin, fout in pairs:
    routed = {}
    for tag, buf in (("out", fout), ("in", fin)):
        parts = [[] for _ in range(P)]
        for q, (sh, d, nb) in enumerate(shard_bufs(buf)):
            if d is None:
                continue
            t0 = now()
            r = api.fastq_ids_route_shard_dev(ctx, d, sh.buf_len, sh.own_len, nb, sh.is_first, sh.is_last, P)
            t = now() - t0
            phase["route"][q] += t
            route_bytes += sh.own_len
            route_t += t
            pos = 0
            for dst in range(P):
                parts[dst].append(r.lines[pos: pos + r.part_bytes[dst]])
                pos += r.part_bytes[dst]
        recv = []
        for dst in range(P):
            t0 = now()
            recv.append(torch.cat(parts[dst]))
            phase["exchange"][dst] += now() - t0
        routed[tag] = recv
    o_sets = []
    for q in range(P):
        t0 = now()
        o_sets.append(ops.set_from_lines(routed["out"][q]))
        phase["O_r build"][q] += now() - t0
    # what diff_sharded builds on EVERY rank: the whole O from all ranks' lists
    everything = torch.cat(routed["out"])
    t0 = now()
    full = api.IdSet.from_txt(ctx, everything)
    repl_build += now() - t0
    full.free()
    for q in range(P):
        t0 = now()
        nl, _ = api.idset_probe_lines_dev(ctx, o_sets[q], routed["in"][q], routed["in"][q].numel(), d_sets[q])
        t = now() - t0
        phase["probe"][q] += t
        probe_lines_n += nl
        probe_t += t
        o_sets[q].free()
dumps = []
for q in range(P):
    t0 = now()
    dumps.append(d_sets[q].sorted_ids())
    phase["merge"][q] += now() - t0
t0 = time.perf_counter()
merged = list(heapq.merge(*dumps))
merge_host = time.perf_counter() - t0
assert merged == want[3]
print(f"virtual ranks P={P} (ms per rank: min / max over ranks):", flush=True)
for k, v in phase.items():
    print(f"  {k:10s} {min(v) * 1e3:8.2f} / {max(v) * 1e3:8.2f}", flush=True)
print(f"  merge of the {P} sorted host lists: {merge_host * 1e3:.1f} ms", flush=True)
print(f"  replicated O build (diff_sharded, every rank, all {P} ranks' ids): {repl_build * 1e3:.2f} ms vs O_r "
      f"max {max(phase['O_r build']) * 1e3:.2f} ms", flush=True)
print(f"route: {route_bytes / route_t / 1e9:.1f} GB/s of shard input (the ids pass + routing, per call); "
      f"probe-lines: {probe_lines_n / probe_t / 1e6:.1f} M lines/s", flush=True)

# ---- 3. memory per rank: set builds in a fresh process (this one's stream-ordered pool already holds the memory freed
# above, so its free-memory deltas would read zero)
lines_all = []
for sh, d, nb in shard_bufs(pairs[0][1]):
    if d is not None:
        r = api.fastq_ids_route_shard_dev(ctx, d, sh.buf_len, sh.own_len, nb, sh.is_first, sh.is_last, P)
        lines_all.append(r)
part0 = torch.cat([r.lines[: r.part_bytes[0]] for r in lines_all])
whole = torch.cat([r.lines for r in lines_all])
_MEM = """
import sys, numpy as np, torch
sys.path.insert(0, sys.argv[1])
from scrubby_b200 import api
ctx = api.Context(0)
dev = torch.device("cuda", 0)
bufs = [torch.from_numpy(np.fromfile(p, dtype=np.uint8)).to(dev) for p in sys.argv[2:4]]
torch.cuda.synchronize(dev)
held, out = [], []
for b in bufs:
    f0 = torch.cuda.mem_get_info(dev)[0]
    held.append(api.IdSet.from_txt(ctx, b))
    ctx.sync()
    img = held[-1].image()
    out.append((f0 - torch.cuda.mem_get_info(dev)[0], img.table_bytes + img.arena_bytes, len(held[-1])))
print(out)
"""
with tempfile.TemporaryDirectory() as tmp:
    paths = [os.path.join(tmp, "whole.txt"), os.path.join(tmp, "part0.txt")]
    for t, p in zip((whole, part0), paths):
        t.cpu().numpy().tofile(p)
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    out = subprocess.run([sys.executable, "-c", _MEM, root, *paths], capture_output=True, text=True)
    (d_full, b_full, n_full), (d_part, b_part, n_part) = eval(out.stdout.strip().splitlines()[-1])
print(f"memory per rank for O of mate 1: replicated ({n_full} ids) {d_full / 1e6:.1f} MB of device memory "
      f"(table + arena {b_full / 1e6:.1f} MB), partitioned O_0 of {P} ({n_part} ids) {d_part / 1e6:.1f} MB "
      f"(table + arena {b_part / 1e6:.1f} MB)", flush=True)
o_part = api.IdSet.from_txt(ctx, part0)

# ---- 4. page load of a partition's set
k = len(o_part)
plain_ids = torch.cat([r.lines for r in lines_all])  # unpartitioned: the first k ids of the file
cut = int((plain_ids == 10).nonzero()[k - 1]) + 1
o_plain = api.IdSet.from_txt(ctx, plain_ids[:cut].clone())
assert len(o_plain) == k
probe_buf = whole.clone()
res = {"partition set": [], "unpartitioned set": []}
for rep in range(a.reps + 1):
    for name, s in (("partition set", o_part), ("unpartitioned set", o_plain)):
        t0 = now()
        api.idset_probe_lines_dev(ctx, s, probe_buf, probe_buf.numel(), None)
        t = now() - t0
        if rep:
            res[name].append(t)
for name, ts in res.items():
    print(f"probe-lines of {probe_buf.numel() / 1e6:.0f} MB of lines against the {name} ({k} ids): "
          f"median {statistics.median(ts) * 1e3:.2f} ms {['%.2f' % (x * 1e3) for x in ts]}", flush=True)
ctx.close()
