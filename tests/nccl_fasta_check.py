"""Real NCCL check of the FASTA multi-GPU driver (run under torchrun on >= 2 GPUs; tests/test_gpu_fasta_shards.py
launches it from pytest and self-skips below two devices):

    python -m torch.distributed.run --nnodes=1 --nproc-per-node 2 --master-addr 127.0.0.1 --master-port 29534 \
        tests/nccl_fasta_check.py

Every rank cleans its byte range of LF and CRLF FASTA files (dist.clean_fasta_files_sharded_{dev,host}, both modes, one
file whose CRLF decision lies in a later rank's range), runs the FASTA diff_sharded, and cleans a file with a parse
error in the last rank's range.  The rank-order concatenations and the counters must equal the single-GPU call.
"""
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
import torch.distributed as dist

from scrubby_b200 import api, synth
from scrubby_b200 import dist as sdist
from scrubby_b200.dist import GpuOps, ShardError, diff_sharded, plan_shards

rank, world, local = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ["LOCAL_RANK"])
torch.cuda.set_device(local)
dev = torch.device("cuda", local)
dist.init_process_group("nccl", device_id=dev)
ctx = api.Context(local)
ops = GpuOps(ctx)
n = 200_000
ids = api.IdSet.from_ids(ctx, [b"syn.%d" % i for i in range(0, n, 3)] + [b"h11"])
tail = synth.gen_fasta(n // 4, 2, crlf=True).numpy().tobytes()
files = {
    "lf_wrapped": synth.gen_fasta(n, 1, wrap=60).numpy().tobytes(),
    "crlf": synth.gen_fasta(n, 2, crlf=True).numpy().tobytes(),
    # header-only records (they decide nothing) fill rank 0's range: the CRLF decision is made in rank 1's
    "crlf_late": b"".join(b">h%d\n" % i for i in range(int(1.3 * len(tail) / max(1, world - 1) / 8))) + tail,
}
ok = True


def shard_of(fa, halo=1 << 16):
    sh = plan_shards(len(fa), world, halo)[rank]
    d = torch.zeros(sh.buf_len + 16, dtype=torch.uint8, device=dev)
    if sh.buf_len:
        d[: sh.buf_len] = torch.frombuffer(bytearray(fa[sh.start: sh.start + sh.buf_len]), dtype=torch.uint8).to(dev)
    return d, sh


def gather(b: bytes):
    parts = [None] * world
    dist.all_gather_object(parts, b)
    return b"".join(parts)


for name, fa in files.items():
    d, sh = shard_of(fa)
    for reverse in (False, True):
        cap = 2 * sh.buf_len + 64
        d_w = torch.empty(cap, dtype=torch.uint8, device=dev)
        d_o = torch.empty(cap, dtype=torch.uint8, device=dev)
        r = sdist.clean_fasta_files_sharded_dev(api, ctx, ids, [(d, sh, d_w, d_o)], dist, reverse)[0]
        cat_w, cat_o = gather(bytes(d_w[: r.n_written].cpu().numpy())), gather(bytes(d_o[: r.n_other].cpu().numpy()))
        h_in = torch.frombuffer(bytearray(fa[sh.start: sh.start + sh.buf_len] or b"\0"), dtype=torch.uint8)
        h_w, h_o = torch.empty(cap, dtype=torch.uint8), torch.empty(cap, dtype=torch.uint8)
        rh = sdist.clean_fasta_files_sharded_host(api, ctx, ids, [(h_in, sh, h_w, h_o)], dist, reverse)[0]
        hcat_w, hcat_o = gather(bytes(h_w[: rh.n_written].numpy())), gather(bytes(h_o[: rh.n_other].numpy()))
        if rank == 0:
            whole = api.clean_fastq(ctx, ids, fa, reverse)
            good = cat_w == whole.written == hcat_w and cat_o == whole.other == hcat_o and \
                (r.reads_in, r.reads_out) == (rh.reads_in, rh.reads_out) == (whole.reads_in, whole.reads_out) and \
                r.total_written == len(whole.written) and r.crlf == whole.crlf
            print(f"clean {name} reverse {reverse}: world {world} reads_in {r.reads_in} one_pass {r.one_pass} "
                  f"crlf {r.crlf} -> {'identical' if good else 'MISMATCH'}", flush=True)
            ok = ok and good

# FASTA diff (utils.rs:250-285) over two file pairs
pairs = []
for name in ("lf_wrapped", "crlf"):
    pairs.append((files[name], api.clean_fastq(ctx, ids, files[name]).written))
sd = diff_sharded(ops, pairs, dist, fasta=True)
if rank == 0:
    whole = api.diff(ctx, pairs)
    good = (sd.reads_in, sd.reads_out, sd.difference) == whole[:3] and sd.diff_ids == whole[3].sorted_ids()
    print(f"diff: world {world} reads_in {sd.reads_in} difference {sd.difference} -> {'identical' if good else 'MISMATCH'}",
          flush=True)
    ok = ok and good

# a parse error (an empty id) in the last rank's range: every rank raises, the failing one with the file's record index
recs = synth.gen_fasta(n, 1).numpy().tobytes()
at = recs.index(b">", len(recs) - len(recs) // (2 * world))
bad = recs[:at] + b">\nACGT\n" + recs[at:]
want_index = recs[:at].count(b">")
d, sh = shard_of(bad)
d_w = torch.empty(2 * sh.buf_len + 64, dtype=torch.uint8, device=dev)
try:
    sdist.clean_fasta_files_sharded_dev(api, ctx, ids, [(d, sh, d_w, None)], dist)
    got = ("none",)
except api.ScrubbyGpuError as e:
    got = ("own", e.status, e.index)
except ShardError as e:
    got = ("other", e.rank, e.status)
rows = [None] * world
dist.all_gather_object(rows, got)
if rank == 0:
    good = rows[-1] == ("own", 9, want_index) and all(r == ("other", world - 1, 9) for r in rows[:-1])
    print(f"parse error: {rows} (record {want_index}) -> {'identical' if good else 'MISMATCH'}", flush=True)
    ok = ok and good

dist.barrier()
if rank == 0:
    print("nccl_fasta_check ok" if ok else "nccl_fasta_check MISMATCH", flush=True)
dist.destroy_process_group()
sys.exit(0 if ok else 1)
