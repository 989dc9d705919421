"""Parity of the CUDA path (through the C ABI) against the CPU oracle: bit-exact bytes, id sets and counts.

All tests here need a B200 (`-m gpu`).  Inputs are the hand-derived golden vectors, seeded synthetic
data of the BASELINE.json shapes at sizes the oracle finishes in seconds, and adversarial FASTQ.
"""
import random

import numpy as np
import pytest
import torch

from conftest import B
from oracle import oracle as orc
from scrubby_b200 import api, synth

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def ctx():
    c = api.Context(0)
    yield c
    c.close()


@pytest.fixture(scope="module", params=[0, 1], ids=["auto", "general"])
def ctx_mode(request):
    c = api.Context(0)
    c.set_mode(request.param)
    c.mode = request.param
    yield c
    c.close()


@pytest.fixture(scope="module")
def ctx_general():
    """a context forced onto the general paths (sgpu_ctx_set_mode(1)): evidence takes the indexed kernel"""
    c = api.Context(0)
    c.set_mode(1)
    c.mode = 1
    yield c
    c.close()


def _ids(lst):
    return sorted(B(x) for x in lst)


def _same_clean(ctx, buf: bytes, ids, reverse=False):
    """GPU vs oracle on one buffer, both outputs + counts (+ identical error class / index)"""
    o = orc.clean_fastq(buf, orc.OSet.from_ids(ids), reverse, raise_on_error=False)
    g = api.clean_fastq(ctx, api.IdSet.from_ids(ctx, ids), buf, reverse, raise_on_error=False)
    assert g.error == o.error, (g.error, o.error)
    if o.error:
        assert g.error_record == o.error_record
    assert g.written == o.written
    assert g.other == o.other
    assert (g.reads_in, g.reads_out) == (o.reads_in, o.reads_out)
    assert g.empty_input == o.empty_input
    if not o.error and not o.empty_input:
        assert g.crlf == o.crlf
    return g


# ---------------------------------------------------------------------------- golden vectors
def test_golden_fastq_cases(ctx_mode, golden):
    for c in golden["fastq_cases"]:
        ids = [B(i) for i in c["ids"]]
        g = api.clean_fastq(ctx_mode, api.IdSet.from_ids(ctx_mode, ids), B(c["buf"]), c["reverse"])
        assert g.written == B(c["written"]), c["name"]
        assert (g.reads_in, g.reads_out) == (c["reads_in"], c["reads_out"]), c["name"]
        assert g.empty_input == c.get("empty_input", False), c["name"]
        _same_clean(ctx_mode, B(c["buf"]), ids, c["reverse"])


def test_golden_fastq_errors(ctx_mode, golden):
    for c in golden["fastq_errors"]:
        g = api.clean_fastq(ctx_mode, api.IdSet.empty(ctx_mode), B(c["buf"]), raise_on_error=False)
        assert (g.error, g.error_record) == (c["error"], c["error_record"]), c["name"]
        _same_clean(ctx_mode, B(c["buf"]), [])


def test_golden_paf(ctx, ctx_general, golden):
    for cx in (ctx, ctx_general):  # the tile kernel, the indexed kernel
        for c in golden["paf_cases"]:
            s = api.IdSet.from_paf(cx, B(c["buf"]), c["min_len"], c["min_cov"], c["min_mapq"])
            assert s.sorted_ids() == _ids(c["expect"]), c["name"]
            assert len(s) == len(c["expect"])
        for c in golden["paf_errors"]:
            with pytest.raises(api.ScrubbyGpuError) as e:
                api.IdSet.from_paf(cx, B(c["buf"]))
            assert e.value.status == c["error"], c["name"]
            if "error_line" in c:
                assert e.value.index == c["error_line"]


def test_golden_sam(ctx, golden):
    for c in golden["sam_cases"]:
        s = api.IdSet.from_sam(ctx, B(c["buf"]), c["min_len"], c["min_cov"], c["min_mapq"])
        assert s.sorted_ids() == _ids(c["expect"]), c["name"]
    for c in golden["sam_errors"]:
        with pytest.raises(api.ScrubbyGpuError) as e:
            api.IdSet.from_sam(ctx, B(c["buf"]))
        assert e.value.status == c["error"], c["name"]
        if "error_line" in c:
            assert e.value.index == c["error_line"]


@pytest.mark.parametrize("seed", range(4))
def test_sam_random_matches_oracle(ctx, seed):
    from test_oracle_golden import _random_sam

    buf = _random_sam(seed, 5000)
    for args in ((0, 0.0, 0), (50, 0.5, 50), (100, 2.0, 30)):
        assert api.IdSet.from_sam(ctx, buf, *args).sorted_ids() == orc.set_from_sam(buf, *args).sorted_ids()
    # device-resident input
    d = torch.frombuffer(bytearray(buf), dtype=torch.uint8).cuda()
    assert api.IdSet.from_sam(ctx, d, 50, 0.5, 50).sorted_ids() == orc.set_from_sam(buf, 50, 0.5, 50).sorted_ids()


def test_golden_reads_and_txt(ctx, ctx_general, golden):
    for cx in (ctx, ctx_general):  # the tile kernel, the indexed kernel
        for c in golden["reads_cases"]:
            s = api.IdSet.from_reads(cx, B(c["buf"]), c["style"], [B(t) for t in c["taxids"]])
            assert s.sorted_ids() == _ids(c["expect"]), c["name"]
        for c in golden["reads_errors"]:
            with pytest.raises(api.ScrubbyGpuError) as e:
                api.IdSet.from_reads(cx, B(c["buf"]), c["style"], [])
            assert e.value.status == c["error"], c["name"]
        for c in golden["txt_cases"]:
            s = api.IdSet.from_txt(cx, B(c["buf"]))
            assert s.sorted_ids() == _ids(c["expect"])
            assert b"" in s and b"r2 " in s and b"r2" not in s


def test_golden_diff(ctx, golden):
    for c in golden["diff_cases"]:
        pairs = [(B(a), B(b)) for a, b in c["pairs"]]
        rin, rout, d, ids = api.diff(ctx, pairs)
        assert (rin, rout, d) == (c["reads_in"], c["reads_out"], c["difference"]), c["name"]
        assert ids.sorted_ids() == _ids(c["diff_ids"]), c["name"]


# ---------------------------------------------------------------------------- id set
def test_idset_inline_and_long_keys(ctx):
    rng = random.Random(7)
    keys = set()
    for n in list(range(1, 40)) + [100, 1000, 5000]:
        for _ in range(20):
            keys.add(bytes(rng.randrange(33, 127) for _ in range(n)))
    keys |= {b"a", b"a\x00", b"a\x00\x00", b"\x00", b"\xff" * 15, b"\xff" * 16, b"x" * 15, b"x" * 16, b"x" * 17}
    keys = sorted(keys)
    s = api.IdSet.from_ids(ctx, keys + keys[:50])  # duplicates offered
    assert len(s) == len(keys)
    assert s.sorted_ids() == keys
    for k in keys[::37]:
        assert k in s
    assert b"a\x00\x00\x00" not in s and b"x" * 18 not in s and b"" not in s
    # image round trip (what the NCCL broadcast carries)
    s2 = api.IdSet.from_image(ctx, s.image())
    assert s2.sorted_ids() == keys


def test_idset_many_keys_matches_oracle(ctx):
    txt = synth.gen_txt_ids(300_000).numpy().tobytes()
    s = api.IdSet.from_txt(ctx, txt)
    o = orc.set_from_txt(txt)
    assert len(s) == len(o)
    assert s.sorted_ids() == o.sorted_ids()


# ---------------------------------------------------------------------------- synthetic configs (small)
def test_c1_alignment_config_small(ctx_mode):
    """config 1 shape: 2x150 pairs + PAF, -l 50 -c 0.5 -q 50, deplete and extract"""
    n = 60_000
    paf = synth.gen_paf(n).numpy().tobytes()
    gs = api.IdSet.from_paf(ctx_mode, paf, 50, 0.5, 50)
    os_ = orc.set_from_paf(paf, 50, 0.5, 50)
    assert gs.sorted_ids() == os_.sorted_ids()
    for mate in (1, 2):
        fq = synth.gen_fastq(n, mate, start=7).numpy().tobytes()
        for reverse in (False, True):
            o = orc.clean_fastq(fq, os_, reverse)
            g = api.clean_fastq(ctx_mode, gs, fq, reverse)
            assert g.written == o.written and g.other == o.other
            assert (g.reads_in, g.reads_out) == (o.reads_in, o.reads_out)
            if ctx_mode is not None and reverse is False and mate == 1:
                assert g.path in (1, 2)


def test_c2_classifier_config_small(ctx, ctx_general):
    """config 2 shape: Kraken2 reads + report, -T Chordata -D 9606 (taxids from the oracle's host stage)"""
    n = 50_000
    rep = synth.gen_kraken_report(500)
    taxids = orc.taxids_from_report(rep, ["Chordata"], ["9606"]).sorted_ids()
    kr = synth.gen_kraken_reads(n).numpy().tobytes()
    os_ = orc.set_from_reads(kr, 0, orc.OSet.from_ids(taxids))
    assert api.IdSet.from_reads(ctx_general, kr, 0, taxids).sorted_ids() == os_.sorted_ids()  # the indexed kernel
    gs = api.IdSet.from_reads(ctx, kr, 0, taxids)
    assert gs.sorted_ids() == os_.sorted_ids()
    fq = synth.gen_fastq(n, 1).numpy().tobytes()
    for reverse in (False, True):
        o = orc.clean_fastq(fq, os_, reverse)
        g = api.clean_fastq(ctx, gs, fq, reverse)
        assert g.written == o.written and g.other == o.other


def test_c3_ont_config_small(ctx_mode):
    """config 3 shape: long reads, UUID ids (arena-resident keys), many PAF lines per read"""
    n = 300
    fq, lens, uu = synth.gen_ont_fastq(n, max_len=120_000)
    fqb = fq.numpy().tobytes()
    rng = random.Random(3)
    lines = []
    expect = set()
    for i in range(n):
        rid = bytes(uu[i].tolist()).decode()
        k = 1 + min(40, int(rng.expovariate(1 / 8)))
        passed = False
        for j in range(k):
            qlen = int(lens[i])
            alen = rng.randrange(20, qlen)
            mapq = rng.choice([0, 10, 49, 50, 60])
            lines.append(f"{rid}\t{qlen}\t0\t{alen}\t+\tchr1\t1000000\t5\t{5 + alen}\t{alen}\t{alen}\t{mapq}\ttp:A:P")
            if (alen >= 5000 or alen / qlen >= 0.5) and mapq >= 50:
                passed = True
        if passed:
            expect.add(rid.encode())
    paf = ("\n".join(lines) + "\n").encode()
    gs = api.IdSet.from_paf(ctx_mode, paf, 5000, 0.5, 50)
    os_ = orc.set_from_paf(paf, 5000, 0.5, 50)
    assert gs.sorted_ids() == os_.sorted_ids() == sorted(expect)
    for reverse in (False, True):
        o = orc.clean_fastq(fqb, os_, reverse)
        g = api.clean_fastq(ctx_mode, gs, fqb, reverse)
        assert g.written == o.written and g.other == o.other
        assert (g.reads_in, g.reads_out) == (o.reads_in, o.reads_out)


def test_diff_fused_ids_pass_matches_general_and_oracle(ctx_mode):
    """ReadDifference (utils.rs:250-285): the one-pass ids mode of the fused kernel (canonical files) and the
    indexed general path give the oracle's counts and id set -- short inline ids, 36-byte ONT ids, device and
    host buffers, an empty output file, and a non-canonical (CRLF) input that must fall back"""
    n = 150_000
    fq = synth.gen_fastq(n, 1).numpy().tobytes()
    keep = orc.OSet.from_ids([f"syn.{i}".encode() for i in range(0, n, 3)])
    out = orc.clean_fastq(fq, keep, True).written  # extract: the output holds every third read
    ont, lens, uu = synth.gen_ont_fastq(3000, max_len=60_000)
    ontb = ont.numpy().tobytes()
    oset = orc.OSet.from_ids([bytes(uu[i].tolist()) for i in range(0, 3000, 2)])
    ont_out = orc.clean_fastq(ontb, oset, False).written
    lines = fq.split(b"\n")
    crlf = b"\r\n".join(lines[:200]) + b"\r\n"      # 50 records, CRLF line endings
    crlf_out = b"\r\n".join(lines[:80]) + b"\r\n"   # the first 20 of them
    cases = [[(fq, out)], [(ontb, ont_out)], [(fq, out), (ontb, ont_out)], [(fq, b"")], [(crlf, crlf_out)]]
    for pairs in cases:
        o = orc.diff(pairs)
        g = api.diff(ctx_mode, pairs)
        assert g[:3] == o[:3]
        assert g[3].sorted_ids() == o[3].sorted_ids()
    d_pairs = [(torch.frombuffer(bytearray(fq), dtype=torch.uint8).cuda(), torch.frombuffer(bytearray(out), dtype=torch.uint8).cuda())]
    o = orc.diff([(fq, out)])
    g = api.diff(ctx_mode, d_pairs)
    assert g[:3] == o[:3] and g[3].sorted_ids() == o[3].sorted_ids()


@pytest.mark.parametrize("k", [1, 2, 5])
def test_fastq_ids_shards_unite_to_the_whole_file(ctx_mode, k):
    """sgpu_fastq_ids_shard_dev: the shards' records and picked ids add up to ReadDifference's loops over the
    whole file (utils.rs:259-283), for 2x150 reads and long ONT reads, with and without a probe set"""
    from scrubby_b200.dist import GpuOps, plan_shards

    ops = GpuOps(ctx_mode)
    fq = synth.gen_fastq(30_000, 1).numpy().tobytes()
    ont, lens, uu = synth.gen_ont_fastq(1500, max_len=80_000)
    for buf, probe_ids, halo in ((fq, [f"syn.{i}".encode() for i in range(0, 30_000, 3)], 4096),
                                 (ont.numpy().tobytes(), [bytes(uu[i].tolist()) for i in range(0, 1500, 2)], 1 << 20)):
        oprobe = orc.OSet.from_ids(probe_ids)
        kept = orc.clean_fastq(buf, oprobe, True).written          # a file holding exactly the probe's records
        want_all = orc.diff([(buf, b"")])                           # every id of the file
        want_abs = orc.diff([(buf, kept)])                          # ids absent from the probe
        gprobe = api.IdSet.from_ids(ctx_mode, probe_ids)
        for probe, want in ((None, want_all), (gprobe, want_abs)):
            into = api.IdSet.empty(ctx_mode)
            rec = picked = 0
            nlb = 0
            for sh in plan_shards(len(buf), k, halo):
                if sh.own_len == 0:
                    continue
                d = ops.upload(buf[sh.start : sh.start + sh.buf_len])
                r, p_ = ops.ids_shard(probe, d, sh, nlb, into)
                rec, picked = rec + r, picked + p_
                nlb += buf[sh.start : sh.start + sh.own_len].count(b"\n")
            assert (rec, picked) == (want[0], want[2])
            assert into.sorted_ids() == want[3].sorted_ids()


def test_c5_diff_small(ctx):
    n = 40_000
    ids = orc.set_from_txt(synth.gen_txt_ids(n).numpy().tobytes())
    gids = api.IdSet.from_txt(ctx, synth.gen_txt_ids(n).numpy().tobytes())
    pairs = []
    for mate in (1, 2):
        fq = synth.gen_fastq(n, mate).numpy().tobytes()
        out = api.clean_fastq(ctx, gids, fq).written
        assert out == orc.clean_fastq(fq, ids).written
        pairs.append((fq, out))
    o = orc.diff(pairs)
    g = api.diff(ctx, pairs)
    assert g[:3] == o[:3]
    assert g[3].sorted_ids() == o[3].sorted_ids()
    assert g[2] == 2 * len(ids) and len(g[3]) == len(ids)


# ---------------------------------------------------------------------------- adversarial framing
def _rand_fastq(rng, n_rec, crlf_first=False, ids_pool=None):
    out = bytearray()
    for i in range(n_rec):
        style = rng.randrange(8)
        rid = rng.choice(ids_pool) if ids_pool else f"r{i}".encode()
        desc = rng.choice([b"", b" d", b"\t1:N:0", b" a b c", b"\x0bvt", " ü".encode(), b" \r x"])
        L = rng.choice([0, 1, 2, 15, 16, 17, 31, 64, 150, 151, 1000])
        seq = bytes(rng.choice(b"ACGTN") for _ in range(L))
        qual = bytes(rng.randrange(33, 74) for _ in range(L))
        if L and style == 1:
            qual = b"@" + qual[1:]
        if L and style == 2:
            qual = b"+" + qual[1:]
        e = b"\r\n" if (crlf_first and i == 0) or style == 3 else b"\n"
        sep = b"+" + (rid + desc if style == 4 else b"")
        out += b"@" + rid + desc + e + seq + e + sep + e + qual + e
    return bytes(out)


@pytest.mark.parametrize("seed", range(6))
def test_adversarial_fastq(ctx_mode, seed):
    rng = random.Random(seed)
    pool = [f"id{k}".encode() for k in range(50)] + [b"x" * 15, b"x" * 16, b"y" * 40, "é1".encode()]
    buf = _rand_fastq(rng, 400, crlf_first=bool(seed & 1), ids_pool=pool)
    ids = rng.sample(pool, 20)
    tails = [b"", b"\n", b"\n\n", b"\r\n", b"\r\n\n"]
    for reverse in (False, True):
        _same_clean(ctx_mode, buf + rng.choice(tails), ids, reverse)
    # missing final newline
    _same_clean(ctx_mode, buf[:-1] if buf.endswith(b"\n") else buf, ids)
    # truncations and corruptions: same error class and index as the oracle
    for _ in range(12):
        cut = rng.randrange(1, len(buf))
        _same_clean(ctx_mode, buf[:cut], ids)
    for _ in range(12):
        b2 = bytearray(buf)
        pos = rng.randrange(len(b2))
        b2[pos] = rng.choice(b"\n@+\rA\xff")
        _same_clean(ctx_mode, bytes(b2), ids)


def test_canonical_input_is_byte_copy(ctx_mode):
    """for canonical input (LF, bare '+', final newline) output bytes == kept records' input bytes"""
    fq = synth.gen_fastq(5000, 1).numpy().tobytes()
    g = api.clean_fastq(ctx_mode, api.IdSet.empty(ctx_mode), fq)
    assert g.written == fq and g.other == b"" and g.reads_out == 5000
    g = api.clean_fastq(ctx_mode, api.IdSet.empty(ctx_mode), fq, reverse=True)
    assert g.written == b"" and g.other == fq


# ---------------------------------------------------------------------------- shards (multi-GPU unit of work)
def _record_starts(fq: bytes):
    pos, out = 0, []
    while pos < len(fq):
        out.append(pos)
        for _ in range(4):
            pos = fq.index(b"\n", pos) + 1
    return out


@pytest.mark.parametrize("k,cut_mode", [(2, "random"), (3, "random"), (8, "random"), (4, "at_start"), (4, "after_start"),
                                        (4, "before_start")])
def test_sharded_concat_is_identical(ctx_mode, k, cut_mode):
    """cut the file at arbitrary byte offsets into k shards (also exactly at / next to record starts);
    concatenated outputs == unsharded output"""
    ctx = ctx_mode
    n = 20_000
    fq_t = synth.gen_fastq(n, 1, start=3)
    fq = fq_t.numpy().tobytes()
    ids_txt = synth.gen_txt_ids(n + 10).numpy().tobytes()
    gs = api.IdSet.from_txt(ctx, ids_txt)
    whole = api.clean_fastq(ctx, gs, fq)
    rng = random.Random(k)
    if cut_mode == "random":
        cuts = sorted(rng.randrange(1, len(fq)) for _ in range(k - 1))
    else:
        starts = _record_starts(fq)
        d = {"at_start": 0, "after_start": 1, "before_start": -1}[cut_mode]
        cuts = sorted(starts[rng.randrange(1, len(starts))] + d for _ in range(k - 1))
    bounds = [0] + cuts + [len(fq)]
    halo = 4096
    outs, others, rin, rout = [], [], 0, 0
    nl_before = 0
    for s in range(k):
        a, b = bounds[s], bounds[s + 1]
        end = len(fq) if s == k - 1 else min(len(fq), b + halo)
        d_in = torch.zeros(end - a + 16, dtype=torch.uint8, device="cuda")
        d_in[: end - a] = torch.frombuffer(bytearray(fq[a:end]), dtype=torch.uint8).cuda()
        d_out = torch.empty(2 * (end - a) + 64, dtype=torch.uint8, device="cuda")
        d_oth = torch.empty(2 * (end - a) + 64, dtype=torch.uint8, device="cuda")
        r = api.clean_fastq_shard_dev(ctx, gs, d_in, end - a, b - a, nl_before, s == 0, s == k - 1, False, d_out,
                                      d_oth)
        assert nl_before == fq[:a].count(b"\n")
        if ctx.mode == 0 and b - a > 400:
            assert r.path == 1, "canonical shards must run through the fused kernel"
        nl_before += api.count_newlines_dev(ctx, d_in, b - a)
        outs.append(d_out[: r.n_written].cpu().numpy().tobytes())
        others.append(d_oth[: r.n_other].cpu().numpy().tobytes())
        rin += r.reads_in
        rout += r.reads_out
    assert b"".join(outs) == whole.written
    assert b"".join(others) == whole.other
    assert (rin, rout) == (whole.reads_in, whole.reads_out)


def test_device_buffers_and_stream(ctx):
    """the _dev entry point on torch tensors, enqueued on torch's current stream"""
    n = 30_000
    fq = synth.gen_fastq(n, 2, device="cuda")
    ids = synth.gen_txt_ids(n, device="cuda")
    s = torch.cuda.Stream()
    with torch.cuda.stream(s):
        ctx.set_stream(s)
        gs = api.IdSet.from_txt(ctx, ids)
        out = torch.empty(fq.numel() + 64, dtype=torch.uint8, device="cuda")
        oth = torch.empty(fq.numel() + 64, dtype=torch.uint8, device="cuda")
        r = api.clean_fastq_dev(ctx, gs, fq, fq.numel(), out, oth)
    s.synchronize()
    ctx.set_stream(torch.cuda.current_stream())
    fqb = fq.cpu().numpy().tobytes()
    o = orc.clean_fastq(fqb, orc.set_from_txt(ids.cpu().numpy().tobytes()))
    assert out[: r.n_written].cpu().numpy().tobytes() == o.written
    assert oth[: r.n_other].cpu().numpy().tobytes() == o.other
    assert r.n_written + r.n_other == len(fqb)  # canonical input: a pure partition of the bytes


# ---------------------------------------------------------------------------- fused single-pass kernel
def test_fused_path_is_taken_and_matches_general(ctx):
    """canonical input must run through the fused kernel (path 1) and equal the general path bit for bit"""
    n = 200_000
    ids = synth.gen_txt_ids(n).numpy().tobytes()
    gs = api.IdSet.from_txt(ctx, ids)
    os_ = orc.set_from_txt(ids)
    for mate in (1, 2):
        fq = synth.gen_fastq(n, mate, start=99_000).numpy().tobytes()
        for reverse in (False, True):
            ctx.set_mode(0)
            f = api.clean_fastq(ctx, gs, fq, reverse)
            ctx.set_mode(1)
            g = api.clean_fastq(ctx, gs, fq, reverse)
            ctx.set_mode(0)
            assert f.path == 1 and g.path == 2
            assert f.written == g.written and f.other == g.other
            assert (f.reads_in, f.reads_out) == (g.reads_in, g.reads_out)
            o = orc.clean_fastq(fq, os_, reverse)
            assert f.written == o.written and f.other == o.other
            assert (f.reads_in, f.reads_out) == (o.reads_in, o.reads_out)


def test_fused_long_reads_straddle_many_tiles(ctx):
    fq, lens, uu = synth.gen_ont_fastq(400, max_len=300_000)
    fqb = fq.numpy().tobytes()
    ids = [bytes(uu[i].tolist()) for i in range(0, 400, 3)]
    gs = api.IdSet.from_ids(ctx, ids)
    os_ = orc.OSet.from_ids(ids)
    for reverse in (False, True):
        f = api.clean_fastq(ctx, gs, fqb, reverse)
        o = orc.clean_fastq(fqb, os_, reverse)
        assert f.path == 1
        assert f.written == o.written and f.other == o.other
        assert (f.reads_in, f.reads_out) == (o.reads_in, o.reads_out)


@pytest.mark.parametrize("n", [1, 2, 49, 50, 51, 3000])
def test_fused_small_and_tile_edge_sizes(ctx, n):
    """tiny inputs and inputs whose size lands around a 16 KiB boundary"""
    ids = [f"syn.{i}".encode() for i in range(0, n + 5, 2)]
    gs = api.IdSet.from_ids(ctx, ids)
    os_ = orc.OSet.from_ids(ids)
    for rl in (150, 141, 142, 143):
        fq = synth.gen_fastq(n, 1, read_len=rl).numpy().tobytes()
        f = api.clean_fastq(ctx, gs, fq)
        o = orc.clean_fastq(fq, os_)
        assert f.path == 1
        assert f.written == o.written and f.other == o.other


def _fastq_with_record_end_at(target: int, n_after: int = 300) -> bytes:
    """canonical FASTQ whose k-th record ends exactly at byte offset `target` (exclusive)"""
    out = bytearray()
    i = 0
    while True:
        rec = f"@syn.{i} 1:N:0:ATCACG\n{'ACGT' * 37}AC\n+\n{'I' * 150}\n".encode()
        if len(out) + len(rec) + 60 > target:
            break
        out += rec
        i += 1
    rest = target - len(out)  # bytes of the record that must end at `target`
    hdr = f"@syn.{i} x".encode()
    body = rest - len(hdr) - 5  # "\n" seq "\n+\n" qual "\n"
    if body % 2:
        hdr += b"y"
        body -= 1
    L = body // 2
    assert L >= 1
    out += hdr + b"\n" + b"G" * L + b"\n+\n" + b"#" * L + b"\n"
    assert len(out) == target
    for j in range(i + 1, i + 1 + n_after):
        out += f"@syn.{j} 1:N:0:ATCACG\n{'ACGT' * 37}AC\n+\n{'I' * 150}\n".encode()
    return bytes(out)


@pytest.mark.parametrize("edge", [16384, 32768, 36864, 2 * 36864])
@pytest.mark.parametrize("delta", [-2, -1, 0, 1, 2])
def test_fused_record_boundary_on_tile_edge(ctx, edge, delta):
    """a record ends exactly on / next to a tile edge (tiles are 36 KiB; 16 / 32 KiB kept for other builds)"""
    fq = _fastq_with_record_end_at(edge + delta)
    ids = [f"syn.{i}".encode() for i in range(0, 800, 3)]
    gs = api.IdSet.from_ids(ctx, ids)
    os_ = orc.OSet.from_ids(ids)
    for reverse in (False, True):
        f = api.clean_fastq(ctx, gs, fq, reverse)
        o = orc.clean_fastq(fq, os_, reverse)
        assert f.path == 1
        assert f.written == o.written and f.other == o.other
        assert (f.reads_in, f.reads_out) == (o.reads_in, o.reads_out)


@pytest.mark.parametrize("read_len", [1, 5, 20, 30, 36, 41, 45, 50, 75, 100, 251, 1000])
def test_record_density_sweep(ctx, read_len):
    """short reads put hundreds of records into one 36 KiB tile (the fused kernel handles <= 360 per tile and
    two newlines per 16-byte chunk, denser input must fall back to the general path): same bytes either way"""
    n = 6000
    fq = synth.gen_fastq(n, 1, read_len=read_len).numpy().tobytes()
    ids = [f"syn.{i}".encode() for i in range(0, n, 2)] + [f"syn.{i}".encode() for i in range(1, n, 7)]
    gs = api.IdSet.from_ids(ctx, ids)
    os_ = orc.OSet.from_ids(ids)
    for reverse in (False, True):
        f = api.clean_fastq(ctx, gs, fq, reverse)
        o = orc.clean_fastq(fq, os_, reverse)
        assert f.written == o.written and f.other == o.other, (read_len, f.path)
        assert (f.reads_in, f.reads_out) == (o.reads_in, o.reads_out)
    d = api.diff(ctx, [(fq, orc.clean_fastq(fq, os_, False).written)])
    od = orc.diff([(fq, orc.clean_fastq(fq, os_, False).written)])
    assert d[:3] == od[:3] and d[3].sorted_ids() == od[3].sorted_ids()


def test_fused_falls_back_on_noncanonical(ctx):
    fq = synth.gen_fastq(3000, 1).numpy().tobytes()
    gs = api.IdSet.from_ids(ctx, [b"syn.5", b"syn.77"])
    os_ = orc.OSet.from_ids([b"syn.5", b"syn.77"])
    variants = {
        "crlf_one_line": fq.replace(b"\n", b"\r\n", 1),
        "crlf_late": fq[:500_000] + fq[500_000:].replace(b"\n", b"\r\n", 1),
        "plus_id": fq.replace(b"\n+\n", b"\n+syn\n", 1),
        "no_final_newline": fq[:-1],
        "blank_tail": fq + b"\n",
        "high_byte_header": fq.replace(b"ATCACG\n", "ATCACGé\n".encode(), 1),
        "bad_len": fq[:700_000] + fq[700_000:].replace(b"A", b"", 1),
    }
    for name, buf in variants.items():
        o = orc.clean_fastq(buf, os_, raise_on_error=False)
        f = api.clean_fastq(ctx, gs, buf, raise_on_error=False)
        assert f.path == 2, name
        assert (f.error, f.error_record) == (o.error, o.error_record), name
        assert f.written == o.written and f.other == o.other, name


def test_fused_one_million_records(ctx):
    """~331 MB per file: larger than L2, tens of thousands of tiles"""
    n = 1_000_000
    ids = synth.gen_txt_ids(n, device="cuda")
    gs = api.IdSet.from_txt(ctx, ids)
    os_ = orc.set_from_txt(ids.cpu().numpy().tobytes())
    fq = synth.gen_fastq(n, 1, device="cuda", start=9_500_000)
    out = torch.empty(fq.numel() + 64, dtype=torch.uint8, device="cuda")
    oth = torch.empty(fq.numel() + 64, dtype=torch.uint8, device="cuda")
    r = api.clean_fastq_dev(ctx, gs, fq, fq.numel(), out, oth)
    assert r.path == 1
    o = orc.clean_fastq(fq.cpu().numpy(), os_, want_bytes=False)
    assert (r.reads_in, r.reads_out) == (o.reads_in, o.reads_out)
    assert r.n_written == o.written.size and r.n_other == o.other.size
    assert np.array_equal(out[: r.n_written].cpu().numpy(), o.written)
    assert np.array_equal(oth[: r.n_other].cpu().numpy(), o.other)


# ---------------------------------------------------------------------------- multi-GPU driver pieces on one GPU
def test_dist_driver_world1_and_set_image(ctx):
    """scrubby_b200.dist with the GPU ops (world 1) + the export/import pair used to replicate the set"""
    from scrubby_b200 import dist as sdist

    n = 5000
    fq = synth.gen_fastq(n, 2, start=11).numpy().tobytes()
    ids_txt = synth.gen_txt_ids(n + 3).numpy().tobytes()
    gs = api.IdSet.from_txt(ctx, ids_txt)
    clone = api.IdSet.from_image(ctx, gs.image())  # what a non-source rank does after the NCCL broadcast
    assert clone.sorted_ids() == gs.sorted_ids()
    o = orc.clean_fastq(fq, orc.set_from_txt(ids_txt))
    r = sdist.clean_fastq_sharded(sdist.GpuOps(ctx), clone, fq, None, want_other=True)
    assert r.written == o.written and r.other == o.other
    assert (r.reads_in, r.reads_out, r.offset_written, r.total_written) == (o.reads_in, o.reads_out, 0, len(o.written))
    t = sdist._as_tensor(torch, gs.image().d_table, 64, torch.device("cuda", 0))  # raw device pointer as a tensor
    assert t.is_cuda and t.numel() == 64


def test_idset_keys_dev_and_device_union(ctx):
    """sgpu_idset_keys_dev (the exchange format of the multi-GPU diff): the keys as "id\\n" lines on the device, and
    GpuOps.unite_sets (all-gather of those lists + one set build) at world 1; diff_sharded through the device path
    equals sgpu_diff and the oracle"""
    from scrubby_b200 import dist as sdist

    rng = random.Random(11)
    keys = {bytes(rng.randrange(33, 127) for _ in range(n)) for n in list(range(1, 40)) * 8 + [100, 700]}
    keys |= {b"x" * 15, b"x" * 16, "éè".encode(), "rあd".encode() * 6}
    a, b = sorted(keys)[::2], sorted(keys)[1::2] + sorted(keys)[:7]
    sa, sb = api.IdSet.from_ids(ctx, a), api.IdSet.from_ids(ctx, b)
    flat = bytes(sa.keys_dev().cpu().numpy())
    assert flat.endswith(b"\n") and sorted(flat.split(b"\n")[:-1]) == sorted(a)
    ops = sdist.GpuOps(ctx)
    assert ops.unite_sets([sa, sb], None).sorted_ids() == sorted(keys)
    assert ops.unite_sets([], None).sorted_ids() == [] and len(api.IdSet.empty(ctx).keys_dev()) == 0
    # a set with the empty id (a blank TXT line, alignment.rs:72-75) keeps it through the exchange
    se = api.IdSet.from_txt(ctx, b"r1\n\nr2\n")
    assert ops.unite_sets([se], None).sorted_ids() == [b"", b"r1", b"r2"]
    # config 5 through the sharded driver's device path
    n = 3000
    pairs = []
    ids = api.IdSet.from_txt(ctx, synth.gen_txt_ids(n).numpy().tobytes())
    for mate in (1, 2):
        fq = synth.gen_fastq(n, mate).numpy().tobytes()
        pairs.append((fq, api.clean_fastq(ctx, ids, fq).written))
    sd = sdist.diff_sharded(ops, pairs, None)
    whole, o = api.diff(ctx, pairs), orc.diff(pairs)
    assert (sd.reads_in, sd.reads_out, sd.difference) == whole[:3] == o[:3]
    assert sd.diff_ids == whole[3].sorted_ids() == o[3].sorted_ids()


def test_sharded_long_reads_fused(ctx):
    """ONT-like records that straddle many tiles, cut into shards at arbitrary offsets"""
    n = 300
    fq_t, lens, uu = synth.gen_ont_fastq(n, seed=9)
    fq = fq_t.numpy().tobytes()
    ids = [bytes(uu[i].tolist()) for i in range(0, n, 3)]
    o = orc.clean_fastq(fq, orc.OSet.from_ids(ids))
    gs = api.IdSet.from_ids(ctx, ids)
    rng = random.Random(5)
    k = 5
    bounds = [0] + sorted(rng.randrange(1, len(fq)) for _ in range(k - 1)) + [len(fq)]
    halo = 600_000
    outs, others, rin, rout, nl_before = [], [], 0, 0, 0
    for s in range(k):
        a, b = bounds[s], bounds[s + 1]
        end = len(fq) if s == k - 1 else min(len(fq), b + halo)
        d_in = torch.zeros(end - a + 16, dtype=torch.uint8, device="cuda")
        d_in[: end - a] = torch.frombuffer(bytearray(fq[a:end]), dtype=torch.uint8).cuda()
        d_out = torch.empty(end - a + 64, dtype=torch.uint8, device="cuda")
        d_oth = torch.empty(end - a + 64, dtype=torch.uint8, device="cuda")
        r = api.clean_fastq_shard_dev(ctx, gs, d_in, end - a, b - a, nl_before, s == 0, s == k - 1, False, d_out, d_oth)
        nl_before += api.count_newlines_dev(ctx, d_in, b - a)
        outs.append(d_out[: r.n_written].cpu().numpy().tobytes())
        others.append(d_oth[: r.n_other].cpu().numpy().tobytes())
        rin += r.reads_in
        rout += r.reads_out
    assert b"".join(outs) == o.written
    assert b"".join(others) == o.other
    assert (rin, rout) == (o.reads_in, o.reads_out)


# ---------------------------------------------------------------------------- evidence tile kernel
def _reads_vs_oracle(ctx, buf: bytes, style: int, taxids):
    ot = orc.OSet.from_ids([t if isinstance(t, bytes) else t.encode() for t in taxids])
    try:
        o = orc.set_from_reads(buf, style, ot)
        oerr = None
    except orc.OracleError as e:
        o, oerr = None, (e.code, e.index)
    try:
        g = api.IdSet.from_reads(ctx, buf, style, taxids)
        gerr = None
    except api.ScrubbyGpuError as e:
        g, gerr = None, (e.status, e.index)
    assert gerr == oerr, (gerr, oerr)
    if o is not None:
        assert g.sorted_ids() == o.sorted_ids()


def _txt_vs_oracle(ctx, buf: bytes):
    try:
        o = orc.set_from_txt(buf)
        oerr = None
    except orc.OracleError as e:
        o, oerr = None, (e.code, e.index)
    try:
        g = api.IdSet.from_txt(ctx, buf)
        gerr = None
    except api.ScrubbyGpuError as e:
        g, gerr = None, (e.status, e.index)
    assert gerr == oerr, (gerr, oerr)
    if o is not None:
        assert g.sorted_ids() == o.sorted_ids()
        assert len(g) == len(o)


@pytest.mark.parametrize("seed", range(4))
def test_reads_tile_kernel_edge_cases(ctx, ctx_general, seed):
    """Kraken2 / Metabuli lines across tile (16 KiB) and halo (1 KiB) edges, CRLF, whitespace to trim, non-ASCII
    lines, very long lines, a missing final newline -- all against the oracle, on the tile and the indexed kernel."""
    rng = random.Random(1000 + seed)
    taxids = ["9606", "7711", "0", "123456", "x9"]
    style = seed & 1
    lines = []
    for i in range(3000):
        tid = rng.choice(["9606", "562", "7711", " 9606", "9606 ", "09606", "+9606", "0", "123456", "x9", ""])
        rid = rng.choice([f"r{i}", f" r{i} ", f"r{i}/1", f"read.{i}.{'x' * rng.randint(0, 40)}", f"ré{i}", f"r{i} "])
        kmer = " ".join(f"{rng.randint(0, 9999)}:{rng.randint(1, 30)}" for _ in range(rng.choice([0, 1, 3, 8, 40, 400])))
        if style == 0:
            f = ["C", rid, tid, "150|150", kmer]
        else:
            f = ["1", rid, tid, "100", "80.5", "genus", kmer]
        if rng.random() < 0.05:
            f += ["extra", "fields"]
        eol = "\r\n" if rng.random() < 0.1 else "\n"
        lines.append("\t".join(f) + eol)
    body = "".join(lines)
    long_line = ("C\tlong\t9606\t1\t" if style == 0 else "1\tlong\t9606\t1\t2\tg\t") + "k" * 50000 + "\n"
    for cx in (ctx, ctx_general):
        for tail in ("", "C\tlast\t9606\t1\tx" if style == 0 else "1\tlast\t9606\t1\t2\tg\tx"):
            _reads_vs_oracle(cx, (body + tail).encode(), style, taxids)
        # a line longer than tile + halo, and tiles without any newline
        _reads_vs_oracle(cx, (body + long_line + body).encode(), style, taxids)


def test_reads_tile_kernel_errors(ctx, ctx_general):
    """too few fields (the reference panics) and invalid UTF-8 report the reference's error class and line, on the
    tile and the indexed kernel"""
    good = "".join(f"C\tr{i}\t9606\t150\tk\n" for i in range(2000))
    for cx in (ctx, ctx_general):
        for bad, at in (("C\tr\t9606\t150\n", 700), ("\n", 1500), ("C\tr\n", 0), ("only one field", 2000)):
            ls = good.splitlines(keepends=True)
            ls.insert(at, bad)
            _reads_vs_oracle(cx, "".join(ls).encode(), 0, ["9606"])
        raw = bytearray(good.encode())
        raw[30000] = 0xFF  # invalid UTF-8 in some line
        _reads_vs_oracle(cx, bytes(raw), 0, ["9606"])
        two = good.splitlines(keepends=True)
        two.insert(100, "C\tr\n")
        two.insert(1900, "x\n")
        _reads_vs_oracle(cx, "".join(two).encode(), 0, ["9606"])  # the first error wins


def test_fasta_input_matches_oracle(ctx_mode):
    """'>' input: needletail's FASTA reader (multi-line sequences kept verbatim, line-ending rules, UnexpectedEnd);
    clean in both modes, both outputs, error class and record index; diff on FASTA files"""
    from test_oracle_differential import FASTA_CASES, rand_fasta

    for buf, ids, rev, w, o in FASTA_CASES:
        g = _same_clean(ctx_mode, buf, ids, rev)
        assert (g.written, g.other) == (w, o)
    for buf in (b">abcd", b">a\nAC\n>b\n", b">a\nAC\n>\nTT\n", b">a\nAC\n>\xff\nTT\n", b">a\n>b\n>c\n", b">a\nA"):
        _same_clean(ctx_mode, buf, [b"a"])
    rng = random.Random(9100)
    ids = [b"b", b"q3", b"x" * 16]
    for _ in range(120):
        _same_clean(ctx_mode, rand_fasta(rng, rng.randrange(1, 9)), ids, rng.random() < 0.5)
    # a larger file: 20 k records of 1-3 sequence lines, every third id in the set
    recs = []
    for i in range(20_000):
        lines = [bytes(rng.choice(b"ACGT") for _ in range(60)) for _ in range(1 + i % 3)]
        recs.append(b">ctg%d len=%d\n" % (i, 60 * len(lines)) + b"\n".join(lines) + b"\n")
    big = b"".join(recs)
    big_ids = [b"ctg%d" % i for i in range(0, 20_000, 3)]
    g = _same_clean(ctx_mode, big, big_ids)
    assert g.reads_in == 20_000 and g.reads_out == 20_000 - len(big_ids) and g.written + g.other != b""
    _same_clean(ctx_mode, big[:-1], big_ids, True)
    # diff (utils.rs:250-285) over FASTA files
    pairs = [(big, g.written), (rand_fasta(random.Random(5), 40), b"")]
    try:
        o, oerr = orc.diff(pairs), None
    except orc.OracleError as e:
        o, oerr = None, (e.code, e.index)
    try:
        d, gerr = api.diff(ctx_mode, pairs), None
    except api.ScrubbyGpuError as e:
        d, gerr = None, (e.status, e.index)
    assert gerr == oerr
    if o is not None:
        assert d[:3] == o[:3] and d[3].sorted_ids() == o[3].sorted_ids()
    d1, o1 = api.diff(ctx_mode, pairs[:1]), orc.diff(pairs[:1])
    assert d1[:3] == o1[:3] == (20_000, 20_000 - len(big_ids), len(big_ids)) and d1[3].sorted_ids() == o1[3].sorted_ids()


def _bam_vs_oracle(ctx, buf: bytes, ml=0, mc=0.0, mq=0):
    try:
        o, oerr = orc.set_from_bam(buf, ml, mc, mq), None
    except orc.OracleError as e:
        o, oerr = None, (e.code, e.index)
    try:
        g, gerr = api.IdSet.from_bam(ctx, buf, ml, mc, mq), None
    except api.ScrubbyGpuError as e:
        g, gerr = None, (e.status, e.index)
    assert gerr == oerr, (gerr, oerr)
    if o is not None:
        assert g.sorted_ids() == o.sorted_ids()
    return g


def test_bam_hand_derived_and_edge_cases(ctx):
    """sgpu_idset_from_bam (alignment.rs:117-146 for binary BAM) on the vectors of tests/test_oracle_bam.py"""
    import struct

    import bam_build as bb

    recs = [bb.record(b"r1", cigar="150M"), bb.record(b"r2", cigar="40M110S"), bb.record(b"r3", cigar="10S35M15S"),
            bb.record(b"r4", cigar="150M", mapq=49), bb.record(b"r5", flag=4), bb.record(b"r6", cigar="30M10I10D40M70S"),
            bb.record(b"r7", cigar="40=40X70S"), bb.record(b"r8", cigar="40M40S", mapq=50), bb.record(b"r9", cigar="", l_seq=0),
            bb.record(b"r5", flag=0x904, cigar="150M"), bb.record(b"ra", flag=0x110, cigar="100M50H")]
    s = bb.stream(recs)
    g = _bam_vs_oracle(ctx, s, 50, 0.5, 50)
    assert g.sorted_ids() == [b"r1", b"r3", b"r6", b"r8", b"ra"]
    for thr in [(0, 0.0, 0), (0, 2.0, 0), (1, 2.0, 0)]:
        _bam_vs_oracle(ctx, s, *thr)
    _bam_vs_oracle(ctx, bb.stream([]))
    # qname rules
    for rs in ([bb.record(b"ok", cigar="10M"), bb.record(b"r\xff", cigar="10M")], [bb.record(b"r\xff", flag=4), bb.record(b"ok", cigar="10M")],
               [bb.record(b"nonul", cigar="10M", nul=False)], [bb.record(b"a\x00b", cigar="10M")], [bb.record(b"", cigar="10M")],
               [bb.record(b"", cigar="10M", nul=False)], [bb.record(b"x" * 15, cigar="9M"), bb.record(b"x" * 16, cigar="9M"), bb.record(b"y" * 200, cigar="9M")]):
        _bam_vs_oracle(ctx, bb.stream(rs))
    # long CIGAR in the CG tag
    real = bb.cigar_ops("100M20I30M50S")
    cg = b"CGBI" + struct.pack("<I", len(real)) + b"".join(struct.pack("<I", v) for v in real)
    other = b"NMi" + struct.pack("<i", 3) + b"MDZ" + b"10A5\x00" + b"XSBc" + struct.pack("<I", 3) + b"\x01\x02\x03"
    fake = [(200 << 4) | 4, (1000 << 4) | 3]
    for aux, kw in ((other + cg, {}), (other, {}), (other + cg, dict(ref_id=-1)), (other + cg, dict(pos=-1)),
                    (b"CGZ100M\x00" + cg, {}), (b"XXq\x00" + cg, {}),
                    (b"CGBI" + struct.pack("<I", 1) + struct.pack("<I", 200 << 4), {})):
        for thr in [(150, 2.0, 0), (1, 2.0, 0)]:
            _bam_vs_oracle(ctx, bb.stream([bb.record(b"long", ops=fake, l_seq=200, aux=aux, **kw)]), *thr)
    wrap = [(0xFFFFFFF << 4) | 0] * 17
    for ml in ((17 * 0xFFFFFFF) & 0xFFFFFFFF, ((17 * 0xFFFFFFF) & 0xFFFFFFFF) + 1):
        _bam_vs_oracle(ctx, bb.stream([bb.record(b"w", ops=wrap, l_seq=10)]), ml, 1e30, 0)
    # structural errors: the first failing record wins
    r = [bb.record(b"r%d" % i, cigar="100M") for i in range(5)]
    s = bb.stream(r)
    neg = bytearray(bb.record(b"x", cigar="10M"))
    neg[20:24] = struct.pack("<i", -1)
    for buf in (s[:-1], s[: len(s) - len(r[4]) + 2], s[: len(s) - len(r[4])], b"BAM\x02" + s[4:], b"", s[:10],
                bb.stream(r[:2] + [struct.pack("<I", 8) + b"\x00" * 8] + r[2:]),
                bb.stream(r[:3] + [bb.record(b"x", cigar="100M", block_size_delta=-60)]), bb.stream(r[:1] + [bytes(neg)]),
                bb.stream([bb.record(b"\xff", cigar="10M")] + r)[:-3]):
        _bam_vs_oracle(ctx, buf)


@pytest.mark.parametrize("seed", range(8))
def test_bam_random_streams_match_oracle(ctx, seed):
    from test_oracle_bam import rand_stream

    rng = random.Random(8000 + seed)
    s = rand_stream(rng, rng.choice([1, 20, 200, 5000]))
    for thr in [(0, 0.0, 0), (50, 0.5, 50), (100, 2.0, 0), (1 << 40, 0.75, 10)]:
        _bam_vs_oracle(ctx, s, *thr)
    for _ in range(6):
        _bam_vs_oracle(ctx, s[: rng.randrange(0, len(s))], 50, 0.5, 50)
    for _ in range(12):
        b = bytearray(s)
        for _ in range(rng.choice([1, 1, 3])):
            b[rng.randrange(len(b))] = rng.choice([0, 1, 4, 0x44, 0x7F, 0x80, 0xFF])
        _bam_vs_oracle(ctx, bytes(b), 50, 0.5, 50)


def _paf_vs_oracle(ctx, buf: bytes, ml=0, mc=0.0, mq=0):
    try:
        o, oerr = orc.set_from_paf(buf, ml, mc, mq), None
    except orc.OracleError as e:
        o, oerr = None, (e.code, e.index)
    try:
        g, gerr = api.IdSet.from_paf(ctx, buf, ml, mc, mq), None
    except api.ScrubbyGpuError as e:
        g, gerr = None, (e.status, e.index)
    assert gerr == oerr, (gerr, oerr)
    if o is not None:
        assert g.sorted_ids() == o.sorted_ids()


@pytest.mark.parametrize("seed", range(12))
def test_paf_adversarial_fields(ctx_mode, seed):
    """random PAF with Rust-parse edge cases ('+150', '', ' 15', '-1', 2^64, mapq 256, short rows, CRLF, missing final
    newline, invalid UTF-8), alone and buried in thousands of valid lines (tile edges): same set, or the same error
    class at the same line, on the tile path and on the indexed path"""
    from test_oracle_differential import _rand_paf

    rng = random.Random(7000 + seed)
    small = _rand_paf(rng, rng.choice([3, 10, 40]))
    good = "".join(f"r{i % 997}\t150\t{i % 50}\t{100 + i % 50}\t+\tt\t1000\t0\t100\t90\t100\t{(i * 7) % 61}\ttp:A:P\n"
                   for i in range(4000)).encode()
    cut = good.rfind(b"\n", 0, rng.randrange(1, len(good))) + 1
    big = good[:cut] + small + (b"" if small.endswith(b"\n") else b"\n") + good[cut:]
    for buf in (small, big):
        for ml, mc, mq in [(0, 0.0, 0), (50, 0.5, 50), (1 << 63, 2.0, 0)]:
            _paf_vs_oracle(ctx_mode, buf, ml, mc, mq)
    bad = bytearray(big)
    bad[rng.randrange(len(bad))] = 0xFF
    _paf_vs_oracle(ctx_mode, bytes(bad), 50, 0.5, 50)


@pytest.mark.parametrize("seed", range(3))
def test_txt_tile_kernel_edge_cases(ctx, ctx_general, seed):
    rng = random.Random(2000 + seed)
    lines = []
    for i in range(5000):
        lines.append(rng.choice([f"id{i}", f"id{i} ", "", f"id{i % 50}", "x" * rng.randint(1, 60), f"é{i}",
                                 "y" * rng.choice([15, 16, 17, 300, 5000])]) + rng.choice(["\n", "\n", "\r\n"]))
    body = "".join(lines)
    for cx in (ctx, ctx_general):  # the tile kernel, the indexed kernel
        _txt_vs_oracle(cx, body.encode())
        _txt_vs_oracle(cx, (body + "last-without-newline").encode())
        _txt_vs_oracle(cx, (body + "z" * 40000 + "\n" + body).encode())
        _txt_vs_oracle(cx, b"\n")
        _txt_vs_oracle(cx, b"a")


def _around_dense(sparse, dense, bads):
    """sparse lines, a dense region, sparse lines: as they are, without the final newline, and with each bad line
    planted before the dense region, inside it, after it, and both before and after (the first error wins)"""
    pre, post = sparse[: len(sparse) // 2], sparse[len(sparse) // 2:]
    half = len(dense) // 2

    def join(*parts):
        return b"".join(x for p in parts for x in p)

    yield join(pre, dense, post)
    yield join(pre, dense, post).rstrip(b"\n")
    for bad in bads:
        yield join(pre, [bad], dense, post)
        yield join(pre, dense[:half], [bad], dense[half:], post)
        yield join(pre, dense, [bad], post)
        yield join(pre, [bad], dense, [bad], post)


def test_txt_dense_fallback(ctx):
    """id lines of at most 7 bytes: 2341 or more lines per 16 KiB tile, more than the tile kernel's 2048, so the whole
    list takes the indexed kernel on the default path; CRLF lines, invalid UTF-8 before / inside / after the dense
    region, no final newline -- against the oracle"""
    rng = random.Random(3100)
    sparse = [b"sparse-id-%06d\n" % i for i in range(2000)]
    dense = [b"t%d%s" % (rng.randrange(10_000), rng.choice([b"\n", b"\n", b"\r\n"])) for _ in range(20_000)]
    assert max(map(len, dense)) <= 7
    for buf in _around_dense(sparse, dense, [b"t\xff1\n", b"\xc3\n"]):
        _txt_vs_oracle(ctx, buf)


def test_reads_dense_fallback(ctx):
    """Kraken2 lines of about 12 bytes: 5 separators each, about 6600 per 16 KiB tile, more than the tile kernel's
    5120, so the whole file takes the indexed kernel on the default path; CRLF lines, whitespace to trim, invalid
    UTF-8 and too few fields before / inside / after the dense region, no final newline -- against the oracle"""
    rng = random.Random(3200)
    sparse = [b"C\tsp%d\t1\t150\t%s\n" % (i, b" ".join(b"%d:1" % k for k in range(8))) for i in range(1000)]
    dense = [b"C\t%s\t%s\t1\t%s" % (rng.choice([b"r%d"] * 7 + [b" r%d"]) % rng.randrange(1000),
                                     rng.choice([b"1", b"2"] * 4 + [b"1 "]), rng.choice([b"\n"] * 3 + [b"\r\n"]))
             for _ in range(20_000)]
    assert sum(map(len, dense)) / len(dense) < 13
    for buf in _around_dense(sparse, dense, [b"C\tr\xff\t1\t1\tk\n", b"C\tr1\t1\n", b"\n"]):
        _reads_vs_oracle(ctx, buf, 0, ["1"])


def test_paf_dense_fallback(ctx):
    """bare 12-column PAF lines of at most 30 bytes: 12 separators each, more than 6500 per 16 KiB tile, more than the
    tile kernel's 5120, so the whole file takes the indexed kernel on the default path; several lines per qname, CRLF
    lines, invalid UTF-8, too few fields and a bad integer before / inside / after the dense region, no final newline
    -- against the oracle"""
    rng = random.Random(3300)
    sparse = [b"s%d\t150\t%d\t%d\t+\tt\t1000\t0\t100\t90\t100\t%d\ttp:A:P\tcg:Z:150M\n" % (i, i % 50, 100 + i % 50,
                                                                                               (i * 7) % 61)
              for i in range(1200)]
    dense = [b"r%d\t%d\t%d\t%d\t+\tt\t9\t0\t9\t9\t9\t%d%s" % (i // 3, rng.randrange(10), rng.randrange(5),
                                                               rng.randrange(10), rng.randrange(100),
                                                               rng.choice([b"\n", b"\n", b"\r\n"]))
             for i in range(20_000)]
    assert max(map(len, dense)) <= 30
    bads = [b"r\xff\t9\t0\t9\t+\tt\t9\t0\t9\t9\t9\t60\n", b"r1\t9\t0\n", b"r1\t9\t0\tx\t+\tt\t9\t0\t9\t9\t9\t60\n"]
    for buf in _around_dense(sparse, dense, bads):
        for ml, mc, mq in [(0, 0.0, 0), (5, 0.5, 50)]:
            _paf_vs_oracle(ctx, buf, ml, mc, mq)


def test_misaligned_device_evidence_is_refused(ctx, ctx_general):
    """a device view that does not start on a 16-byte boundary is SGPU_ERR_INVALID_ARG for every line format, on the
    default and the general path"""
    paf = b"r1\t150\t0\t150\t+\tt\t1000\t0\t150\t150\t150\t60\n" * 4
    sam = b"@SQ\tSN:t\tLN:1000\n" + b"r1\t0\tt\t1\t60\t4M\t*\t0\t0\tACGT\tIIII\n" * 4
    calls = [(paf, lambda cx, d: api.IdSet.from_paf(cx, d)), (b"r1\nr2\n" * 8, lambda cx, d: api.IdSet.from_txt(cx, d)),
             (b"C\tr1\t1\t1\tk\n" * 8, lambda cx, d: api.IdSet.from_reads(cx, d, 0, ["1"])),
             (sam, lambda cx, d: api.IdSet.from_sam(cx, d))]
    for cx in (ctx, ctx_general):
        for buf, call in calls:
            d = torch.frombuffer(bytearray(b"\n" + buf), dtype=torch.uint8).cuda()
            assert len(call(cx, d[1:].clone())) >= 1  # the same bytes, aligned, are accepted
            with pytest.raises(api.ScrubbyGpuError) as e:
                call(cx, d[1:])
            assert e.value.status == 18  # SGPU_ERR_INVALID_ARG


# ---------------------------------------------------------------------------- pipelined host-buffer path
@pytest.fixture()
def small_pipeline_chunks(monkeypatch):
    monkeypatch.setenv("SGPU_PIPE_CHUNK", str(256 * 1024))
    monkeypatch.setenv("SGPU_PIPE_HALO", str(8 * 1024))


def test_host_pipeline_matches_oracle(ctx, small_pipeline_chunks):
    """sgpu_clean_fastq on host buffers cut into chunks (H2D / kernels / D2H overlapped): same bytes and counts
    as the oracle, deplete, extract and split"""
    n = 12000
    fq = synth.gen_fastq(n, 1).numpy().tobytes()  # ~4 MB -> 16 chunks
    ids = [b"syn.%d" % i for i in range(0, n, 3)]
    for reverse in (False, True):
        g = _same_clean(ctx, fq, ids, reverse)
        assert g.path == 1
    # no final newline, and a cut that falls right after a newline
    _same_clean(ctx, fq[:-1], ids)
    # a cut that falls exactly on a record boundary: a filler record pads the first chunk to 256 KiB
    b = fq.rindex(b"\n@syn.", 0, 256 * 1024 - 100) + 1
    room = 256 * 1024 - b
    name = b"@pad" if (room - 9) % 2 == 0 else b"@padd"
    L = (room - len(name) - 5) // 2
    filler = name + b"\n" + b"A" * L + b"\n+\n" + b"I" * L + b"\n"
    assert len(filler) == room
    _same_clean(ctx, fq[:b] + filler + fq[b:], ids)
    # a malformed join in a late chunk: same error, same records before it
    cut = fq.index(b"\n", 3 * 256 * 1024 + 77) + 1
    _same_clean(ctx, fq[:cut - 40] + fq[cut:], ids)


def test_host_pipeline_crlf_errors_and_long_records(ctx, small_pipeline_chunks):
    n = 6000
    fq = synth.gen_fastq(n, 2).numpy().tobytes()
    ids = [b"syn.%d" % i for i in range(1, n, 2)]
    _same_clean(ctx, fq.replace(b"\n", b"\r\n"), ids)  # CRLF: every chunk on the general path
    bad = bytearray(fq)
    p = fq.index(b"\n@syn.4000 ") + 1
    bad[p] = ord("X")  # invalid record start in a late chunk: same error class and record index
    _same_clean(ctx, bytes(bad), ids)
    # a record longer than the halo: the pipelined path steps aside for the one-shot path
    long_rec = b"@long\n" + b"A" * 20000 + b"\n+\n" + b"I" * 20000 + b"\n"
    k = fq.index(b"\n@syn.900 ") + 1
    _same_clean(ctx, fq[:k] + long_rec + fq[k:], ids + [b"long"])


@pytest.mark.parametrize("n,mates", [(10_000_000, (1, 2)), (14_000_000, (2,))])
def test_c2_full_size_properties(ctx, n, mates):
    """BASELINE configs[1] at its full size (10 M reads per mate file, 3.3 GB each; the oracle would need minutes)
    and one file beyond 4 GiB (14 M reads, 4.6 GB: every offset past 2^32, as in configs[3]'s 33 GB files):
    size-independent properties of the fused path -- byte partition, checksum linearity, line counts,
    removed == |set|, extract mode == the complementary stream, idempotence."""
    from bench import taxids_for_config

    dev = torch.device("cuda", 0)
    d_k = synth.gen_kraken_reads(n, device=dev)
    ids = api.IdSet.from_reads(ctx, d_k, 0, taxids_for_config())
    del d_k
    assert 0 < len(ids) < n
    for mate in mates:
        d_r = synth.gen_fastq(n, mate, device=dev)
        n_in = d_r.numel()
        d_w = torch.empty(n_in + 64, dtype=torch.uint8, device=dev)
        d_o = torch.empty(n_in + 64, dtype=torch.uint8, device=dev)
        r = api.clean_fastq_dev(ctx, ids, d_r, n_in, d_w, d_o)
        assert r.path == 1, "the fused kernel must take canonical input"
        assert r.reads_in == n and r.reads_out == n - len(ids)          # every set id is one read of the file
        assert r.n_written + r.n_other == n_in                          # byte partition of the input
        w, o = d_w[: r.n_written], d_o[: r.n_other]
        assert int(w.sum(dtype=torch.int64)) + int(o.sum(dtype=torch.int64)) == int(d_r.sum(dtype=torch.int64))
        assert int((w == 10).sum()) == 4 * r.reads_out and int((o == 10).sum()) == 4 * (n - r.reads_out)
        assert int(w[0]) == ord("@") and int(w[-1]) == 10
        # extract mode writes exactly the complementary stream
        d_w2 = torch.empty(n_in + 64, dtype=torch.uint8, device=dev)
        r2 = api.clean_fastq_dev(ctx, ids, d_r, n_in, d_w2, None, True)
        assert r2.n_written == r.n_other and torch.equal(d_w2[: r2.n_written], o)
        # idempotence: the depleted file holds no id of the set
        r3 = api.clean_fastq_dev(ctx, ids, w.clone(), r.n_written, d_w2, None)
        assert (r3.reads_in, r3.reads_out, r3.n_written) == (r.reads_out, r.reads_out, r.n_written)
        assert torch.equal(d_w2[: r3.n_written], w)
        del d_r, d_w, d_o, d_w2, w, o
        torch.cuda.empty_cache()
    ids.free()
