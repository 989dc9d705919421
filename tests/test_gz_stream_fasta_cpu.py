"""FastqCleaner::clean_reads on a gzip / BGZF FASTA runs as the same pipeline as FASTQ (scrubby_host.cpp:
clean_fasta_gz_stream: inflate thread -> sgpu_clean_fasta_shard chunk by chunk -> deflate / write behind it).  Here the
shard call is the CPU stand-in of the FASTA shard contract (tests/test_fasta_shards_cpu.py), so the chunking, the
line-ending chaining, the halo growth, the error indices and the writers are checked against the oracle's whole-file
bytes without a GPU."""
import ctypes as C
import gzip
import os
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from oracle import oracle as orc  # noqa: E402
from scrubby_b200 import _lib, hostlib, synth  # noqa: E402
from test_fasta_shards_cpu import SGPU_ERR_HALO, ShardFailure, shard_clean  # noqa: E402

CB = C.CFUNCTYPE(C.c_int, C.c_void_p, C.c_size_t, C.c_size_t, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_size_t,
                 C.POINTER(C.c_size_t), C.POINTER(_lib.Counts), C.POINTER(C.c_int))


def _stand_in(ids, reverse, log):
    def cb(p_in, n_in, own_len, is_first, is_last, le_before, p_out, cap, p_nout, p_counts, p_le):
        buf = C.string_at(p_in, n_in)
        log.append(dict(n_in=n_in, own_len=own_len, is_first=is_first, is_last=is_last, le=le_before, rc=0))
        p_nout[0] = 0
        try:
            st, err, w, _, rin, rout, le_own = shard_clean(buf, own_len, is_first, is_last, le_before, ids, reverse)
        except ShardFailure as e:
            log[-1]["rc"] = e.status
            return e.status
        if len(w) > cap:
            log[-1]["rc"] = _lib.SGPU_ERR_CAPACITY
            return _lib.SGPU_ERR_CAPACITY
        C.memmove(p_out, w, len(w))
        p_nout[0] = len(w)
        c = p_counts[0]
        c.reads_in, c.reads_out, c.error_record = rin, rout, err
        p_le[0] = le_own if le_own >= 0 else -1
        log[-1]["rc"] = st
        return st

    return CB(cb)


def _stream(src, dst, ids, chunk, halo, reverse=False):
    H = hostlib.load()
    H.scrubby_host_stream_clean_fasta.argtypes = [C.c_char_p, C.c_char_p, C.c_size_t, C.c_size_t, CB,
                                                  C.POINTER(C.c_int), C.POINTER(C.c_uint64)]
    log = []
    cb = _stand_in(ids, reverse, log)
    handled, err = C.c_int(-1), C.c_uint64(0)
    rc = H.scrubby_host_stream_clean_fasta(str(src).encode(), str(dst).encode(), chunk, halo, cb, C.byref(handled),
                                           C.byref(err))
    return rc, handled.value, err.value, log


def _read_out(path):
    raw = open(path, "rb").read()
    return gzip.decompress(raw) if str(path).endswith(".gz") else raw


IDS = [b"syn.%d" % i for i in range(0, 3000, 3)] + [b"h4"]


def _files():
    yield "wrapped", synth.gen_fasta(400, 1, wrap=60).numpy().tobytes()
    yield "crlf", synth.gen_fasta(400, 2, wrap=70, crlf=True).numpy().tobytes()
    yield "late_decision", b"".join(b">h%d\n" % i for i in range(500)) + synth.gen_fasta(200, 1, crlf=True).numpy().tobytes()
    yield "no_final_newline", synth.gen_fasta(300, 1).numpy().tobytes()[:-1]
    yield "blank_tail", synth.gen_fasta(300, 1).numpy().tobytes() + b"\n\n\n"


@pytest.mark.parametrize("chunk,halo", [(1000, 300), (4096, 512), (50_000, 1 << 16), (1 << 22, 1 << 20)])
@pytest.mark.parametrize("reverse", [False, True])
def test_fasta_gz_stream_matches_the_whole_file(tmp_path, chunk, halo, reverse):
    ids = orc.OSet.from_ids(IDS)
    for name, fa in _files():
        want = orc.clean_fastq(fa, ids, reverse)
        src = tmp_path / f"{name}.fa.gz"
        src.write_bytes(gzip.compress(fa, 1))
        dst = tmp_path / f"{name}_out.fa.gz"
        rc, handled, _, log = _stream(src, dst, ids, chunk, halo, reverse)
        assert (rc, handled) == (0, 1), name
        assert _read_out(dst) == want.written, (name, chunk, halo)
        good = [c for c in log if c["rc"] == 0]
        assert good[0]["is_first"] == 1 and good[0]["le"] == -1 and good[-1]["is_last"] == 1
        assert good[-1]["own_len"] == good[-1]["n_in"]
        assert sum(c["own_len"] for c in good) == len(fa)
        if name == "crlf" and len(good) > 1:
            assert all(c["le"] == 1 for c in good[1:])


def test_fasta_gz_stream_long_records_grow_the_halo(tmp_path):
    fa = synth.gen_fasta(12, 1, read_len=6000, wrap=80).numpy().tobytes()
    ids = orc.OSet.from_ids([b"syn.3", b"syn.7"])
    want = orc.clean_fastq(fa, ids)
    src = tmp_path / "ont.fa.gz"
    src.write_bytes(gzip.compress(fa))
    for chunk, halo in ((2000, 100), (700, 64)):
        dst = tmp_path / f"o_{chunk}.fa"
        rc, handled, _, log = _stream(src, dst, ids, chunk, halo)
        assert (rc, handled) == (0, 1)
        assert _read_out(dst) == want.written
        assert any(c["rc"] == SGPU_ERR_HALO for c in log)


def test_fasta_gz_stream_multi_member_and_bgzf(tmp_path):
    from bam_build import bgzf

    fa = synth.gen_fasta(1500, 1, wrap=50, crlf=True).numpy().tobytes()
    ids = orc.OSet.from_ids(IDS)
    want = orc.clean_fastq(fa, ids)
    cut = len(fa) // 2 + 33
    raws = {"multi": gzip.compress(fa[:7001]) + gzip.compress(fa[7001:cut]) + gzip.compress(fa[cut:]),
            "bgzf": bgzf(fa), "bgzf_small": bgzf(fa, 700), "gzip_then_bgzf": gzip.compress(fa[:cut]) + bgzf(fa[cut:])}
    for name, raw in raws.items():
        src = tmp_path / f"{name}.fa.gz"
        src.write_bytes(raw)
        assert hostlib.read_file(str(src)) == fa
        for chunk, halo in ((3000, 500), (40_000, 4000)):
            dst = tmp_path / f"{name}_{chunk}.fa"
            rc, handled, _, log = _stream(src, dst, ids, chunk, halo)
            assert (rc, handled) == (0, 1), name
            assert _read_out(dst) == want.written, name
            assert len([c for c in log if c["rc"] == 0]) > 1


def test_fasta_gz_stream_truncated_and_corrupt(tmp_path):
    from bam_build import bgzf

    fa = synth.gen_fasta(1500, 1, wrap=60).numpy().tobytes()
    ids = orc.OSet.from_ids(IDS)
    gz = bytearray(gzip.compress(fa))
    gz[len(gz) // 2] ^= 0xFF
    gz[len(gz) // 2 + 1] ^= 0xFF
    for name, raw in (("corrupt", bytes(gz)), ("garbage", gzip.compress(fa) + b"garbage-after-the-member")):
        src = tmp_path / f"{name}.fa.gz"
        src.write_bytes(raw)
        rc, handled, _, _ = _stream(src, tmp_path / f"{name}.out.fa", ids, 3000, 500)
        assert rc >= 100, name
    # a BGZF file cut short: the stream gives what the whole-file reader gives (the members before the cut), filtered
    b = bgzf(fa, 700)
    src = tmp_path / "bgzf_truncated.fa.gz"
    src.write_bytes(b[: len(b) * 2 // 3])
    whole = hostlib.read_file(str(src))
    want = orc.clean_fastq(whole, ids, raise_on_error=False)
    dst = tmp_path / "bgzf_truncated.out.fa"
    rc, handled, err, _ = _stream(src, dst, ids, 3000, 500)
    assert handled == 1 or rc
    assert (rc >= 100 and err == want.error_record) if want.error else rc == 0
    assert _read_out(dst) == want.written


def test_fasta_gz_stream_parse_error_carries_the_file_index(tmp_path):
    recs = [b">r%d\nACGT\nAC\n" % i for i in range(400)]
    recs[311] = b">\nACGT\n"
    fa = b"".join(recs)
    ids = orc.OSet.from_ids([b"r5"])
    want = orc.clean_fastq(fa, ids, raise_on_error=False)
    assert want.error and want.error_record == 311
    src = tmp_path / "bad.fa.gz"
    src.write_bytes(gzip.compress(fa))
    for chunk in (1000, 1 << 20):
        dst = tmp_path / f"bad_{chunk}.fa.gz"
        rc, handled, err, _ = _stream(src, dst, ids, chunk, 200)
        assert rc >= 100 and err == 311
        assert _read_out(dst) == want.written


def test_fasta_gz_stream_leaves_other_inputs_to_the_whole_file_path(tmp_path):
    ids = orc.OSet.from_ids([])
    cases = {
        "plain.fa": b">a\nACGT\n>b\nAC\n",                          # not gzip
        "fastq.fq.gz": gzip.compress(synth.gen_fastq(20, 1).numpy().tobytes()),  # FASTQ: its own stream
        "empty.fa.gz": gzip.compress(b""),
        "tiny.fa.gz": gzip.compress(b">a\n"),                       # fewer than 5 bytes: the empty-input rule
        "junk.fa.gz": gzip.compress(b"hello\n"),
    }
    for name, raw in cases.items():
        src = tmp_path / name
        src.write_bytes(raw)
        dst = tmp_path / (name + ".out")
        rc, handled, _, log = _stream(src, dst, ids, 1000, 100)
        assert (rc, handled) == (0, 0), name
        assert not log and not dst.exists(), name
