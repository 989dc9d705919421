"""Real NCCL check of the hash-partitioned diff (run under torchrun; tests/test_gpu_diff_partitioned.py launches it on
min(device count, 8) GPUs, world 1 included -- NCCL at world 1 still runs the real all_to_all_single):

    python -m torch.distributed.run --nnodes=1 --nproc-per-node 2 --master-addr 127.0.0.1 --master-port 29535 \
        tests/nccl_diff_partitioned_check.py

dist.diff_partitioned must equal the single-GPU sgpu_diff and dist.diff_sharded on FASTQ, FASTA and long-id (Illumina)
pairs on every rank, and a parse error in the input must end every rank exactly as it ends diff_sharded.
"""
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
import torch.distributed as dist

from scrubby_b200 import api, synth
from scrubby_b200.dist import GpuOps, ShardError, diff_partitioned, diff_sharded

rank, world, local = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ["LOCAL_RANK"])
torch.cuda.set_device(local)
dev = torch.device("cuda", local)
dist.init_process_group("nccl", device_id=dev)
ctx = api.Context(local)
ops = GpuOps(ctx)
n = 200_000
ok = True


def pairs_of(gen, ids):
    gs = api.IdSet.from_ids(ctx, ids)
    files = [gen(m).numpy().tobytes() for m in (1, 2)]
    return [(f, api.clean_fastq(ctx, gs, f).written) for f in files]


cases = {
    "fastq": (lambda m: synth.gen_fastq(n, m, read_len=80), [b"syn.%d" % i for i in range(0, n, 3)], False),
    "fasta": (lambda m: synth.gen_fasta(n, m, wrap=60, read_len=80), [b"syn.%d" % i for i in range(0, n, 3)], True),
}
ill = synth.gen_fastq_illumina(n, 1, read_len=80).numpy().tobytes()
ill_ids = [ln[1:].split(b" ")[0] for ln in ill.split(b"\n")[0::4][::3] if ln]
cases["long_ids"] = (lambda m: synth.gen_fastq_illumina(n, m, read_len=80), ill_ids, False)
for name, (gen, ids, fasta) in cases.items():
    pairs = pairs_of(gen, ids)
    w = api.diff(ctx, pairs)
    want = (w[0], w[1], w[2], w[3].sorted_ids())
    got = diff_partitioned(ops, pairs, dist, halo=1 << 16, fasta=fasta)
    ref = diff_sharded(ops, pairs, dist, halo=1 << 16, fasta=fasta)
    for tag, r in (("partitioned", got), ("sharded", ref)):
        if (r.reads_in, r.reads_out, r.difference, r.diff_ids) != want:
            ok = False
            print(f"MISMATCH rank {rank} {name} {tag}: {(r.reads_in, r.reads_out, r.difference, len(r.diff_ids))} vs "
                  f"{want[:3] + (len(want[3]),)}", flush=True)
    if rank == 0:
        print(f"{name}: world {world} reads_in={want[0]} reads_out={want[1]} difference={want[2]} "
              f"ids={len(want[3])}", flush=True)

# a parse error in the last rank's range of the second input file
pairs = pairs_of(cases["fastq"][0], cases["fastq"][1])
fin = bytearray(pairs[1][0])
pos = fin.rfind(b"\n@syn.", 0, len(fin) - 5000)
fin[pos + 1] = ord("X")
pairs[1] = (bytes(fin), pairs[1][1])
outcome = []
for fn in (diff_partitioned, diff_sharded):
    try:
        fn(ops, pairs, dist, halo=1 << 16)
        outcome.append(("ok",))
    except ShardError as e:
        outcome.append(("shard", e.rank, e.status))
    except api.ScrubbyGpuError as e:
        outcome.append(("own", e.status, e.index))
if outcome[0] != outcome[1] or outcome[0][0] == "ok":
    ok = False
    print(f"MISMATCH rank {rank} parse error: {outcome}", flush=True)
elif rank == 0:
    print(f"parse error: {outcome[0]}", flush=True)
flags = [None] * world
dist.all_gather_object(flags, ok)
if rank == 0 and all(flags):
    print("nccl_diff_partitioned_check ok", flush=True)
ctx.close()
dist.destroy_process_group()
sys.exit(0 if all(flags) else 1)
