"""Device and end-to-end time of the FASTA path (no FASTA workload is in bench.py, whose contract is FASTQ).

    python tools/fasta_time.py [--records 100000000] [--host-records 20000000] [--parent-lib PATH]

1. the device-resident whole-file call (sgpu_clean_fastq_dev on '>' input) of this tree, alternated with the same call
   of another build of the library (--parent-lib: e.g. the parent commit's libscrubby_gpu.so), outputs compared;
2. the chunked host path end to end (sgpu_clean_fastq on pinned host buffers);
3. the sharded device-resident step (dist.clean_fasta_files_sharded_dev) at N = 1 in this process.
Input: gen_fasta records (the 2x150 mate-1 records as FASTA, unwrapped and wrap=60); half the ids are in the set.
Reports reads/s, GB/s of input and algorithmic bytes (input + output) over the HBM copy peak measured in the same run
(a 4 GiB device-to-device copy: read + write bytes over time), with the card name and power limit read in the same run."""
import argparse
import ctypes as C
import os
import statistics
import subprocess
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch

from bench import taxids_for_config
from scrubby_b200 import _lib, api, dist as sdist, synth


ap = argparse.ArgumentParser()
ap.add_argument("--records", type=int, default=100_000_000)
ap.add_argument("--host-records", type=int, default=20_000_000)
ap.add_argument("--parent-lib", default=None)
ap.add_argument("--reps", type=int, default=5)
a = ap.parse_args()

smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                     capture_output=True, text=True).stdout.strip()
print(f"card: {smi}", flush=True)
dev = torch.device("cuda", 0)


def hbm_copy_peak():
    """bytes read + written per second by a 4 GiB device-to-device copy, best of 10 (outside L2)"""
    x = torch.empty(4 << 30, dtype=torch.uint8, device=dev)
    y = torch.empty_like(x)
    best = None
    for _ in range(10):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        y.copy_(x)
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1)
        best = ms if best is None else min(best, ms)
    del x, y
    torch.cuda.empty_cache()
    return 2 * (4 << 30) / (best / 1e3)


HBM_PEAK = hbm_copy_peak()
print(f"measured HBM copy peak: {HBM_PEAK / 1e12:.2f} TB/s (data sheet: 7.7 TB/s)", flush=True)
ctx = api.Context(0)
taxids = taxids_for_config()


def line(label, ms, n_rec, n_in, n_out):
    alg = n_in + n_out
    print(f"{label}: {ms:.2f} ms, {n_rec / ms / 1e3:.1f} M reads/s, {n_in / ms / 1e6:.1f} GB/s in, "
          f"algorithmic {alg / 1e9:.2f} GB -> {alg / (ms / 1e3) / HBM_PEAK * 100:.1f}% of the measured HBM copy peak", flush=True)


class Parent:
    """another build of the library, loaded beside this one (its own context on the same stream)"""

    def __init__(self, path):
        L = C.CDLL(path)
        vp, sz, i32 = C.c_void_p, C.c_size_t, C.c_int
        L.sgpu_ctx_create.argtypes = [i32, C.POINTER(vp)]
        L.sgpu_ctx_set_stream.argtypes = [vp, vp]
        L.sgpu_idset_from_reads_dev.argtypes = [vp, vp, sz, i32, C.POINTER(C.c_char_p), C.POINTER(sz), sz, C.POINTER(vp),
                                                C.POINTER(C.c_uint64)]
        L.sgpu_clean_fastq_dev.argtypes = [vp, vp, vp, sz, i32, vp, sz, C.POINTER(sz), vp, sz, C.POINTER(sz),
                                           C.POINTER(_lib.Counts)]
        self.L, self.h = L, vp()
        assert L.sgpu_ctx_create(0, C.byref(self.h)) == 0
        raw = torch.cuda.current_stream(0).cuda_stream
        assert L.sgpu_ctx_set_stream(self.h, vp(raw if raw else 1)) == 0

    def idset_from_reads(self, kr):
        bs = [t.encode() if isinstance(t, str) else bytes(t) for t in taxids]
        arr = (C.c_char_p * len(bs))(*bs)
        lens = (C.c_size_t * len(bs))(*[len(b) for b in bs])
        self.s, err = C.c_void_p(), C.c_uint64()
        assert self.L.sgpu_idset_from_reads_dev(self.h, C.c_void_p(kr.data_ptr()), kr.numel(), 0, arr, lens, len(bs),
                                                C.byref(self.s), C.byref(err)) == 0

    def clean(self, d_in, n_in, d_out):
        n1, n2, c = C.c_size_t(), C.c_size_t(), _lib.Counts()
        rc = self.L.sgpu_clean_fastq_dev(self.h, self.s, C.c_void_p(d_in.data_ptr()), n_in, 0, C.c_void_p(d_out.data_ptr()),
                                         d_out.numel(), C.byref(n1), None, 0, C.byref(n2), C.byref(c))
        assert rc == 0, rc
        return n1.value, c.reads_in, c.reads_out


def timed(fn):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    e0.record()
    r = fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1), r


kr = synth.gen_kraken_reads(a.records, device=dev)
ids = api.IdSet.from_reads(ctx, kr, 0, taxids)
parent = None
if a.parent_lib:
    parent = Parent(a.parent_lib)
    parent.idset_from_reads(kr)
del kr
torch.cuda.empty_cache()

for wrap in (None, 60):
    fa = synth.gen_fasta(a.records, 1, wrap=wrap, device=dev)
    n_in = fa.numel()
    d_in = torch.zeros(n_in + 16, dtype=torch.uint8, device=dev)
    d_in[:n_in] = fa
    del fa
    torch.cuda.empty_cache()
    d_out = torch.empty(n_in + n_in // 8 + 64, dtype=torch.uint8, device=dev)
    d_ref = torch.empty_like(d_out) if parent else None
    tag = f"{a.records} records, wrap={wrap}, {n_in / 1e9:.2f} GB"
    api.clean_fastq_dev(ctx, ids, d_in, n_in, d_out)  # warm-up of every shape
    if parent:
        parent.clean(d_in, n_in, d_ref)
    t_new, t_par = [], []
    for _ in range(a.reps):
        ms, r = timed(lambda: api.clean_fastq_dev(ctx, ids, d_in, n_in, d_out))
        t_new.append(ms)
        if parent:
            ms, rp = timed(lambda: parent.clean(d_in, n_in, d_ref))
            t_par.append(ms)
    assert r.reads_in == a.records and r.path == 3
    line(f"whole-file device call, this tree   [{tag}] median of {a.reps}", statistics.median(t_new), r.reads_in, n_in,
         r.n_written)
    print(f"  spread: min {min(t_new):.2f} max {max(t_new):.2f} ms", flush=True)
    if parent:
        line(f"whole-file device call, parent build [{tag}] median of {a.reps}", statistics.median(t_par), rp[1], n_in,
             rp[0])
        print(f"  spread: min {min(t_par):.2f} max {max(t_par):.2f} ms", flush=True)
        same = rp[0] == r.n_written and (rp[1], rp[2]) == (r.reads_in, r.reads_out) and \
            torch.equal(d_out[: r.n_written], d_ref[: r.n_written])
        print(f"  outputs equal to the parent build: {same}", flush=True)
        assert same
    # the sharded device-resident step at N = 1 (one rank: the whole file is the shard)
    sh = sdist.plan_shards(n_in, 1)[0]
    ms_s = []
    for _ in range(a.reps):
        ms, rs = timed(lambda: sdist.clean_fasta_files_sharded_dev(api, ctx, ids, [(d_in, sh, d_out, None)]))
        ms_s.append(ms)
    assert rs[0].reads_in == a.records and rs[0].total_written == r.n_written
    line(f"sharded device step, N = 1          [{tag}] median of {a.reps}", statistics.median(ms_s), a.records, n_in,
         r.n_written)
    del d_in, d_out, d_ref
    torch.cuda.empty_cache()

# chunked host path end to end (pinned buffers, 128 MiB chunks)
fa = synth.gen_fasta(a.host_records, 1, wrap=60, device=dev)
n_in = fa.numel()
h_in = torch.empty(n_in, dtype=torch.uint8, pin_memory=True)
h_in.copy_(fa)
want_bytes = None
del fa
h_out = torch.empty(n_in + 64, dtype=torch.uint8, pin_memory=True)
api.clean_fastq_host(ctx, ids, h_in, n_in, h_out)
t_h = []
for _ in range(a.reps):
    t0 = time.perf_counter()
    rh = api.clean_fastq_host(ctx, ids, h_in, n_in, h_out)
    t_h.append((time.perf_counter() - t0) * 1e3)
assert rh.reads_in == a.host_records
print(f"chunked host path, end to end [{a.host_records} records, wrap=60, {n_in / 1e9:.2f} GB]: median "
      f"{statistics.median(t_h):.1f} ms (min {min(t_h):.1f}), {a.host_records / statistics.median(t_h) / 1e3:.1f} M reads/s, "
      f"{n_in / statistics.median(t_h) / 1e6:.1f} GB/s in", flush=True)
print("sharded device step at N = 2, 4, 8: not measured here (needs a multi-GPU torchrun launch)", flush=True)
