"""FASTA shards on the B200: sgpu_clean_fasta_shard{,_dev} and sgpu_fasta_ids_shard_dev against the whole-file call and
the oracle, the chunked host path of sgpu_clean_fastq on FASTA, and its device memory.  The shards are chained the way
the drivers chain them (tests/test_fasta_shards_cpu.py: run_chain)."""
import os
import random
from concurrent.futures import ThreadPoolExecutor

import numpy as np
import pytest
import torch

from oracle import oracle as orc
from scrubby_b200 import api, synth
from test_fasta_shards_cpu import HAND, SGPU_ERR_HALO, ShardFailure, run_chain, standin, whole
from test_oracle_differential import FASTA_CASES, rand_fasta

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def ctx():
    c = api.Context(0)
    yield c
    c.close()


def _dev(b: bytes):
    d = torch.zeros(len(b) + 16, dtype=torch.uint8, device="cuda")
    if b:
        d[: len(b)] = torch.frombuffer(bytearray(b), dtype=torch.uint8).cuda()
    return d


def gpu_run(ctx, gs, buf: bytes, reverse: bool):
    """one shard through sgpu_clean_fasta_shard_dev, in run_chain's shape"""
    def run(a, own, blen, first, last, le):
        d = _dev(buf[a: a + blen])
        cap = 2 * blen + 64
        d_w = torch.empty(cap, dtype=torch.uint8, device="cuda")
        d_o = torch.empty(cap, dtype=torch.uint8, device="cuda")
        try:
            r = api.clean_fasta_shard_dev(ctx, gs, d, blen, own, first, last, le, d_w, d_o, reverse,
                                          raise_on_error=False)
        except api.ScrubbyGpuError as e:
            if e.status == SGPU_ERR_HALO:
                raise ShardFailure(SGPU_ERR_HALO)
            raise
        w = bytes(d_w[: r.n_written].cpu().numpy())
        o = bytes(d_o[: r.n_other].cpu().numpy())
        return r.error, r.error_record if r.error else 0, w, o, r.reads_in, r.reads_out, r.le_own if not r.error else -2
    return run


def _whole_gpu(ctx, gs, buf, reverse):
    g = api.clean_fastq(ctx, gs, buf, reverse, raise_on_error=False)
    return g.error, g.error_record if g.error else 0, g.written, g.other, g.reads_in, g.reads_out


def _check_sweeps(ctx, buf, ids, reverse, cut_sets, halos):
    oset, gs = orc.OSet.from_ids(ids), api.IdSet.from_ids(ctx, ids)
    want = whole(buf, oset, reverse)
    assert _whole_gpu(ctx, gs, buf, reverse) == want
    run, ref = gpu_run(ctx, gs, buf, reverse), standin(buf, oset, reverse)
    for cuts in cut_sets:
        for halo in halos:
            got = run_chain(run, len(buf), cuts, halo)
            assert got == want, (buf[:200], cuts, halo, reverse)
            assert run_chain(ref, len(buf), cuts, halo) == want


@pytest.mark.parametrize("reverse", [False, True])
def test_shard_dev_every_cut_matches_whole(ctx, reverse):
    for buf, ids, _, _, _ in FASTA_CASES:
        _check_sweeps(ctx, buf, ids, reverse, [[c] for c in range(1, len(buf))], (1, 8))
    for buf in HAND:
        _check_sweeps(ctx, buf, [b"b", b"c"], reverse, [[c] for c in range(1, len(buf))], (1, 8))


def test_shard_dev_random_files_many_shards(ctx):
    rng = random.Random(7700)
    ids = [b"b", b"q3", b"x" * 16]
    for _ in range(60):
        buf = rand_fasta(rng, rng.randrange(1, 12))
        if len(buf) < 5:
            continue
        cut_sets = [sorted(rng.sample(range(1, len(buf)), min(rng.randrange(1, 8), len(buf) - 1))) for _ in range(4)]
        _check_sweeps(ctx, buf, ids, rng.random() < 0.5, cut_sets, (rng.choice([1, 3, 17]),))


def test_shard_dev_decision_in_a_later_shard_and_errors(ctx):
    head = b"".join(b">h%d\n" % i for i in range(300))
    body = synth.gen_fasta(300, 1, wrap=40, crlf=True).numpy().tobytes()
    buf = head + body
    n = len(buf)
    cut_sets = [[n // 2], [n // 5, 2 * n // 5, 3 * n // 5], [len(head) - 3, len(head) + 2]]
    _check_sweeps(ctx, buf, [b"h5", b"syn.7"], False, cut_sets, (64, 4096))
    at = body.index(b">", 5000)
    bad = body[:at] + b">\nACGT\n" + body[at:]  # an empty id: get_id fails there
    _check_sweeps(ctx, bad, [b"syn.2"], True, [[2000], [1000, 4000, 6000, 9000]], (64,))


def test_shard_dev_argument_checks(ctx):
    gs = api.IdSet.empty(ctx)
    d = _dev(b"@a\nAC\n+\nII\n")
    out = torch.empty(64, dtype=torch.uint8, device="cuda")
    with pytest.raises(api.ScrubbyGpuError) as e:  # a first shard must start with '>'
        api.clean_fasta_shard_dev(ctx, gs, d, 12, 12, True, True, -1, out)
    assert e.value.status == 18
    d = _dev(b">a\nAC\n>b\nGG\n")
    with pytest.raises(api.ScrubbyGpuError) as e:  # a first shard decides the line ending itself
        api.clean_fasta_shard_dev(ctx, gs, d, 12, 6, True, False, 0, out)
    assert e.value.status == 18
    with pytest.raises(api.ScrubbyGpuError) as e:  # 16-byte alignment
        api.clean_fasta_shard_dev(ctx, gs, d[1:], 11, 11, False, True, 0, out)
    assert e.value.status == 18
    r = api.clean_fasta_shard_dev(ctx, gs, _dev(b">a\n"), 3, 3, True, True, -1, out)  # fewer than 5 bytes: empty input
    assert r.empty_input and r.n_written == 0
    r = api.clean_fasta_shard_dev(ctx, gs, _dev(b"\n>ab\nC"), 6, 6, False, True, 0, out)  # ... only for first-and-last
    assert not r.empty_input and r.reads_in == 1 and bytes(out[: r.n_written].cpu().numpy()) == b">ab\nC\n"


def test_shard_dev_unexpected_end_in_last_shard(ctx):
    gs = api.IdSet.empty(ctx)
    out = torch.empty(64, dtype=torch.uint8, device="cuda")
    r = api.clean_fasta_shard_dev(ctx, gs, _dev(b"A\n>a\n"), 5, 5, False, True, 0, out, raise_on_error=False)
    assert (r.error, r.error_record) == (6, 0)
    # the FASTQ ids shard entry point keeps refusing a shard of '>' input
    with pytest.raises(api.ScrubbyGpuError) as e:
        api.fastq_ids_shard_dev(ctx, None, _dev(b">a\nAC\n>b\nGG\n"), 12, 6, 0, True, False, None)
    assert e.value.status == 15


def test_ids_shards_united_equal_diff(ctx):
    rng = random.Random(31)
    fin = synth.gen_fasta(3000, 1, wrap=60).numpy().tobytes()
    ids = [b"syn.%d" % i for i in range(0, 3000, 3)]
    fout = orc.clean_fastq(fin, orc.OSet.from_ids(ids)).written
    want = api.diff(ctx, [(fin, fout)])
    for _ in range(4):
        halo = 512
        cuts_o = sorted(rng.sample(range(1, len(fout)), 3))
        cuts_i = sorted(rng.sample(range(1, len(fin)), 5))
        from test_fasta_shards_cpu import shards_from_cuts

        o_set = api.IdSet.empty(ctx)
        rout = 0
        for a, own, blen, first, last in shards_from_cuts(len(fout), cuts_o, halo):
            rec, _ = api.fasta_ids_shard_dev(ctx, None, _dev(fout[a: a + blen]), blen, own, first, last, o_set)
            rout += rec
        d_set = api.IdSet.empty(ctx)
        rin = diff = 0
        for a, own, blen, first, last in shards_from_cuts(len(fin), cuts_i, halo):
            rec, picked = api.fasta_ids_shard_dev(ctx, o_set, _dev(fin[a: a + blen]), blen, own, first, last, d_set)
            rin, diff = rin + rec, diff + picked
        assert (rin, rout, diff) == tuple(want[:3])
        assert d_set.sorted_ids() == want[3].sorted_ids()


def _host_cases():
    yield synth.gen_fasta(3000, 1, wrap=60).numpy().tobytes()
    yield synth.gen_fasta(3000, 2, crlf=True).numpy().tobytes()
    yield b"".join(b">h%d\n" % i for i in range(3000)) + synth.gen_fasta(2000, 1, wrap=33, crlf=True).numpy().tobytes()
    recs = synth.gen_fasta(3000, 1).numpy().tobytes()
    yield recs[:300_000] + b">\nAC\n" + recs[300_000 + recs[300_000:].index(b">"):]  # an empty id late in the file
    yield synth.gen_fasta(40, 1, read_len=30_000, wrap=80).numpy().tobytes()  # ONT-like: records longer than the halo


@pytest.mark.parametrize("chunk,halo", [(4096, 1024), (16384, 4096), (65536, 100_000)])
def test_host_chunked_equals_one_shot(ctx, monkeypatch, chunk, halo):
    ids = [b"syn.%d" % i for i in range(0, 3000, 4)] + [b"h9"]
    gs, oset = api.IdSet.from_ids(ctx, ids), orc.OSet.from_ids(ids)
    for buf in _host_cases():
        for rev in (False, True):
            want = whole(buf, oset, rev)
            monkeypatch.delenv("SGPU_PIPE_CHUNK", raising=False)
            assert _whole_gpu(ctx, gs, buf, rev) == want
            monkeypatch.setenv("SGPU_PIPE_CHUNK", str(chunk))
            monkeypatch.setenv("SGPU_PIPE_HALO", str(halo))
            assert _whole_gpu(ctx, gs, buf, rev) == want, (len(buf), chunk, halo, rev)
            # the host shard entry point, three shards chained
            n = len(buf)
            assert run_chain(host_run(ctx, gs, buf, rev), n, [n // 3, 2 * n // 3], 200_000) == want


def host_run(ctx, gs, buf: bytes, reverse: bool):
    h = torch.frombuffer(bytearray(buf), dtype=torch.uint8)

    def run(a, own, blen, first, last, le):
        h_w = torch.empty(2 * blen + 64, dtype=torch.uint8)
        h_o = torch.empty(2 * blen + 64, dtype=torch.uint8)
        try:
            r = api.clean_fasta_shard_host(ctx, gs, h[a: a + blen], blen, own, first, last, le, h_w, h_o, reverse,
                                           raise_on_error=False)
        except api.ScrubbyGpuError as e:
            if e.status == SGPU_ERR_HALO:
                raise ShardFailure(SGPU_ERR_HALO)
            raise
        return (r.error, r.error_record if r.error else 0, bytes(h_w[: r.n_written].numpy()),
                bytes(h_o[: r.n_other].numpy()), r.reads_in, r.reads_out, r.le_own if not r.error else -2)
    return run


@pytest.mark.parametrize("wrap", [None, 60])
def test_host_chunked_full_size_matches_oracle(ctx, wrap):
    """10 M records of 150 bases as FASTA through the chunked host path (128 MiB chunks); the oracle over record-aligned
    pieces of the same file"""
    n = 10_000_000
    fa = synth.gen_fasta(n, 1, wrap=wrap, device="cuda")
    h_in = torch.empty(fa.numel(), dtype=torch.uint8, pin_memory=True)
    h_in.copy_(fa)
    del fa
    ids = api.IdSet.from_reads(ctx, synth.gen_kraken_reads(n, device="cuda"), 0, _taxids())
    oset = orc.OSet.from_ids(ids.sorted_ids())
    h_w = torch.empty(h_in.numel() + 64, dtype=torch.uint8, pin_memory=True)
    h_o = torch.empty(h_in.numel() + 64, dtype=torch.uint8, pin_memory=True)
    r = api.clean_fastq_host(ctx, ids, h_in, h_in.numel(), h_w, h_o)
    assert r.reads_in == n and r.n_written + r.n_other == h_in.numel()
    # record-aligned pieces of 500 k records: every record of a digit class has the same length
    starts = _record_offsets(n, wrap, 500_000)
    a_np = h_in.numpy()

    def one(i):
        return orc.clean_fastq(a_np[starts[i]: starts[i + 1]], oset, False, want_bytes=False)

    ow = oo = rin = rout = 0
    with ThreadPoolExecutor(max(2, min(12, (os.cpu_count() or 4) - 2))) as ex:
        for rr in ex.map(one, range(len(starts) - 1)):
            assert np.array_equal(rr.written, h_w[ow: ow + rr.written.size].numpy())
            assert np.array_equal(rr.other, h_o[oo: oo + rr.other.size].numpy())
            ow, oo, rin, rout = ow + rr.written.size, oo + rr.other.size, rin + rr.reads_in, rout + rr.reads_out
    assert (ow, oo, rin, rout) == (r.n_written, r.n_other, r.reads_in, r.reads_out)


def _taxids():
    from bench import taxids_for_config

    return taxids_for_config()


def _record_offsets(n, wrap, per):
    def size(k):  # bytes of records 0 .. k-1 of gen_fasta(read_len=150)
        tot, lo = 0, 0
        lines = 1 if not wrap else -(-150 // wrap)
        while lo < k:
            d = len(str(lo))
            hi = min(k, 10 ** d)
            tot += (hi - lo) * (1 + 17 + d + 1 + 150 + lines)
            lo = hi
        return tot
    return [size(min(n, i)) for i in range(0, n + per, per)]


_MEM_PROBE = r"""
import sys, torch
sys.path.insert(0, sys.argv[1])
from scrubby_b200 import api, synth
fa = synth.gen_fasta(int(sys.argv[2]), 1, wrap=60).numpy().tobytes()
c = api.Context(0)
gs = api.IdSet.from_ids(c, [b"syn.%d" % i for i in range(0, int(sys.argv[2]), 2)])
torch.cuda.synchronize()
free0, _ = torch.cuda.mem_get_info()
l0 = c.launches
g = api.clean_fastq(c, gs, fa)
torch.cuda.synchronize()
free1, _ = torch.cuda.mem_get_info()
print(free0 - free1, c.launches - l0, len(fa), g.reads_in)
"""


def _mem_probe(records, env):
    """device memory taken by one sgpu_clean_fastq call on a FASTA file, in a fresh process (nothing retained in the
    stream-ordered pool from earlier work), and the kernel launches it issued"""
    import subprocess
    import sys

    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    r = subprocess.run([sys.executable, "-c", _MEM_PROBE, root, str(records)], capture_output=True, text=True,
                       timeout=600, env={**os.environ, **env})
    assert r.returncode == 0, r.stderr[-2000:]
    used, launches, n, reads = (int(x) for x in r.stdout.split()[-4:])
    assert reads == records
    return used, launches, n


def test_host_chunked_device_memory_is_bounded_by_the_chunks():
    """the chunked path takes the input staging plus chunk-sized output staging and per-chunk tables; the one-shot path
    takes the input, two file-sized outputs and an 8-byte-per-newline index.  The launch count tells the paths apart:
    the chunked path launches its kernels once per chunk."""
    chunk, halo = 1 << 20, 1 << 16
    env = {"SGPU_PIPE_CHUNK": str(chunk), "SGPU_PIPE_HALO": str(halo)}
    used_c, launches_c, n = _mem_probe(400_000, env)  # ~70 MB, ~1.2 M newlines
    used_1, launches_1, _ = _mem_probe(400_000, {"SGPU_PIPE_CHUNK": str(1 << 40)})  # one chunk: the one-shot path
    k = -(-n // chunk)
    assert launches_c >= 5 * k > launches_1, (launches_c, launches_1, k)
    # beyond the input staging: the four output staging buffers and the pool's per-chunk scratch, not file-sized
    obuf = 2 * (chunk + halo) + 64
    beyond_input = used_c - (n + 16) * 17 // 16
    assert beyond_input <= 4 * obuf * 17 // 16 + (64 << 20), (used_c, n)
    assert used_1 - used_c >= n, (used_1, used_c, n)
    # a file four times the size: what the chunked path takes beyond the input does not grow with it
    used_c4, _, n4 = _mem_probe(1_600_000, env)
    assert used_c4 - (n4 + 16) * 17 // 16 <= 4 * obuf * 17 // 16 + (64 << 20), (used_c4, n4)


@pytest.fixture(scope="module")
def cli():
    from scrubby_b200 import hostlib

    hostlib.build()
    return hostlib.CLI


@pytest.mark.parametrize("kind", ["gzip", "bgzf"])
def test_cli_fasta_gz_streams_through_the_shard_entry_point(cli, tmp_path, kind):
    """a gzip / BGZF FASTA goes inflate -> sgpu_clean_fasta_shard chunk by chunk -> deflate (clean_fasta_gz_stream); with
    small chunks it gives the bytes and report of SCRUBBY_NO_GZ_STREAM=1 (the whole-file path) and of the oracle"""
    import gzip
    import json
    import subprocess

    from bam_build import bgzf

    n = 6000
    head = b"".join(b">h%d\n" % i for i in range(400))  # the line ending is decided after a few chunks
    fa = head + synth.gen_fasta(n, 1, wrap=60, crlf=True).numpy().tobytes()
    ids = b"".join(b"syn.%d\n" % i for i in range(0, n, 4)) + b"h7\n"
    src = tmp_path / "reads.fa.gz"
    src.write_bytes(gzip.compress(fa, 1) if kind == "gzip" else bgzf(fa, 4000))
    ip = tmp_path / "ids.txt"
    ip.write_bytes(ids)
    for extract in (False, True):
        want = orc.clean_fastq(fa, orc.set_from_txt(ids), extract)
        outs = {}
        for mode, env in (("stream", {"SCRUBBY_STREAM_CHUNK": "20000", "SCRUBBY_STREAM_HALO": "300"}),
                          ("whole", {"SCRUBBY_NO_GZ_STREAM": "1"})):
            o, js = tmp_path / f"o_{extract}.fa.gz", tmp_path / f"r_{extract}.json"  # (the report names the paths)
            args = [cli, "alignment", "-i", src, "-o", o, "-a", ip, "-j", js] + (["-e"] if extract else [])
            r = subprocess.run([str(x) for x in args], capture_output=True, text=True, timeout=300,
                               env={**os.environ, **env})
            assert r.returncode == 0, r.stderr[-2000:]
            rep = json.load(open(js))
            rep.pop("date", None)
            outs[mode] = (gzip.decompress(o.read_bytes()), rep)
        assert outs["stream"][0] == outs["whole"][0] == want.written
        assert outs["stream"][1] == outs["whole"][1]
        assert (outs["stream"][1]["reads_in"], outs["stream"][1]["reads_out"]) == (want.reads_in, want.reads_out)


def test_nccl_fasta_sharded_run_is_identical_to_one_gpu():
    """FASTA clean (both modes, LF and CRLF files, a CRLF decision in a later rank), the FASTA diff and a parse error
    under NCCL on every GPU of the box (2..8): rank-order concatenations equal the single-GPU call (nccl_fasta_check.py)"""
    import socket
    import subprocess
    import sys

    n = torch.cuda.device_count()
    if n < 2:
        pytest.skip("needs at least two GPUs")
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    port = s.getsockname()[1]
    s.close()
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={min(n, 8)}",
                        "--master-addr", "127.0.0.1", "--master-port", str(port),
                        os.path.join(root, "tests", "nccl_fasta_check.py")], capture_output=True, text=True, timeout=900,
                       cwd=root)
    assert r.returncode == 0, (r.stdout[-3000:], r.stderr[-3000:])
    assert "nccl_fasta_check ok" in r.stdout and "MISMATCH" not in r.stdout
