"""Set-build time per evidence format and path, this tree beside another build of the library.

    python tools/paf_time.py [--parent-lib PATH] [--reps 7]

Inputs: C1-shaped PAF (gen_paf, 1 M pairs), the PAF of C3 (gen_ont_paf, 200 k ONT reads, about 8 lines per read),
C2's Kraken2 lines (gen_kraken_reads, 10 M reads), C4's id list (50 M ids of 100 M pairs) and a dense id list
(16 M lines of 7 bytes: about 2340 lines per 16 KiB tile, more than the tile kernel takes).
Paths: mode 0 (the tile kernel; for the dense list its fallback to the indexed kernel) and mode 1 (forced indexed).
Each rep runs this tree, then the other build (--parent-lib, e.g. the parent commit's libscrubby_gpu.so) on the same
device buffer; the medians and spreads are printed with the set sizes of both, with the card name and power limit read
in the same run."""
import argparse
import ctypes as C
import os
import statistics
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch

from bench import gen_txt_full, taxids_for_config
from scrubby_b200 import api, synth

ap = argparse.ArgumentParser()
ap.add_argument("--parent-lib", default=None)
ap.add_argument("--reps", type=int, default=7)
a = ap.parse_args()

smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                     capture_output=True, text=True).stdout.strip()
print(f"card: {smi}", flush=True)
dev = torch.device("cuda", 0)
taxids = [t.encode() if isinstance(t, str) else bytes(t) for t in taxids_for_config()]


class Parent:
    """another build of the library, loaded beside this one (its own context on the same stream)"""

    def __init__(self, path):
        L = C.CDLL(path)
        vp, sz, i32, u64 = C.c_void_p, C.c_size_t, C.c_int, C.c_uint64
        L.sgpu_ctx_create.argtypes = [i32, C.POINTER(vp)]
        L.sgpu_ctx_set_stream.argtypes = [vp, vp]
        L.sgpu_ctx_set_mode.argtypes = [vp, i32]
        L.sgpu_idset_from_paf_dev.argtypes = [vp, vp, sz, u64, C.c_double, C.c_uint8, C.POINTER(vp), C.POINTER(u64)]
        L.sgpu_idset_from_txt_dev.argtypes = [vp, vp, sz, C.POINTER(vp), C.POINTER(u64)]
        L.sgpu_idset_from_reads_dev.argtypes = [vp, vp, sz, i32, C.POINTER(C.c_char_p), C.POINTER(sz), sz, C.POINTER(vp),
                                                C.POINTER(u64)]
        L.sgpu_idset_len.argtypes = [vp]
        L.sgpu_idset_len.restype = u64
        L.sgpu_idset_free.argtypes = [vp]
        L.sgpu_idset_free.restype = None
        self.L, self.h = L, vp()
        assert L.sgpu_ctx_create(0, C.byref(self.h)) == 0
        raw = torch.cuda.current_stream(0).cuda_stream
        assert L.sgpu_ctx_set_stream(self.h, vp(raw if raw else 1)) == 0
        self.tax = ((C.c_char_p * len(taxids))(*taxids), (C.c_size_t * len(taxids))(*[len(t) for t in taxids]))

    def set_mode(self, mode):
        assert self.L.sgpu_ctx_set_mode(self.h, mode) == 0

    def build(self, kind, d):
        """the set's size"""
        s, err, p, n = C.c_void_p(), C.c_uint64(), C.c_void_p(d.data_ptr()), d.numel()
        if kind == "paf":
            rc = self.L.sgpu_idset_from_paf_dev(self.h, p, n, 50, 0.5, 50, C.byref(s), C.byref(err))
        elif kind == "txt":
            rc = self.L.sgpu_idset_from_txt_dev(self.h, p, n, C.byref(s), C.byref(err))
        else:
            rc = self.L.sgpu_idset_from_reads_dev(self.h, p, n, 0, *self.tax, len(taxids), C.byref(s), C.byref(err))
        assert rc == 0, rc
        k = self.L.sgpu_idset_len(s)
        self.L.sgpu_idset_free(s)
        return k


def build_here(ctx, kind, d):
    if kind == "paf":
        s = api.IdSet.from_paf(ctx, d, 50, 0.5, 50)
    elif kind == "txt":
        s = api.IdSet.from_txt(ctx, d)
    else:
        s = api.IdSet.from_reads(ctx, d, 0, taxids)
    k = len(s)
    s.free()
    return k


def timed(fn):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    e0.record()
    r = fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1), r


def dense_ids(n):
    """n lines of 6 hex digits and '\\n'"""
    i = torch.arange(n, dtype=torch.int64, device=dev)
    hexd = torch.tensor(list(b"0123456789abcdef"), dtype=torch.uint8, device=dev)
    cols = [hexd[(i >> (4 * k)) & 15] for k in range(5, -1, -1)] + [torch.full_like(i, 10, dtype=torch.uint8)]
    return torch.stack(cols, 1).reshape(-1)


def inputs():
    yield "C1 PAF (1 M pairs)", "paf", synth.gen_paf(1_000_000, device=dev)
    fq, lens, uu = synth.gen_ont_fastq(200_000, device=dev)
    del fq
    torch.cuda.empty_cache()
    yield "C3 PAF (200 k ONT reads)", "paf", synth.gen_ont_paf(lens, uu, device=dev)
    yield "C2 Kraken2 (10 M reads)", "reads", synth.gen_kraken_reads(10_000_000, device=dev)
    yield "C4 id list (50 M ids)", "txt", gen_txt_full(100_000_000, dev)
    yield "dense id list (16 M x 7 B)", "txt", dense_ids(1 << 24)


ctx = api.Context(0)
parent = Parent(a.parent_lib) if a.parent_lib else None
for label, kind, d in inputs():
    n_lines = int((d == 10).sum())
    for mode in (0, 1):
        ctx.set_mode(mode)
        if parent:
            parent.set_mode(mode)
        k_new = build_here(ctx, kind, d)  # warm-up of every shape
        k_par = parent.build(kind, d) if parent else None
        t_new, t_par = [], []
        for _ in range(a.reps):
            t_new.append(timed(lambda: build_here(ctx, kind, d))[0])
            if parent:
                t_par.append(timed(lambda: parent.build(kind, d))[0])
        med = statistics.median
        msg = (f"{label}, {d.numel() / 1e6:.0f} MB, {n_lines / 1e6:.2f} M lines, mode {mode}: this tree {med(t_new):.3f} ms "
               f"[{min(t_new):.3f} .. {max(t_new):.3f}]")
        if parent:
            msg += f", parent build {med(t_par):.3f} ms [{min(t_par):.3f} .. {max(t_par):.3f}]"
        print(msg + f"; {k_new} ids" + (f" (parent build {k_par})" if parent else ""), flush=True)
        if parent:
            assert k_new == k_par
    del d
    torch.cuda.empty_cache()
ctx.close()
