"""Deterministic synthetic inputs of the shapes BASELINE.json names (SURVEY.md section 8d).

Written with torch ops so that the same code fills HBM directly for bench.py (device="cuda")
and small CPU tensors for the tests.  This is data plumbing, not part of the hot path.

  2x150 pairs : R1 `@syn.{i} 1:N:0:ATCACG`, R2 `@syn.{i} 2:N:0:ATCACG`, unpadded decimal i (mates
                share the id token), uniform ACGT, qualities '!'..'I' with the first quality
                forced to '@' for i%64==0 and '+' for i%64==1 (adversarial framing), LF, bare '+',
                final newline => 323 + digits(i) bytes per record (331 at 8 digits).
  membership  : read i is "host" iff splitmix64(i ^ seed) & 1.
"""
from __future__ import annotations

import torch

SEED = 0x5C2BB1E5
_M64 = (1 << 64) - 1


def _i64(v: int) -> int:
    v &= _M64
    return v - (1 << 64) if v >= (1 << 63) else v


def _lsr(x: torch.Tensor, k: int) -> torch.Tensor:
    return (x >> k) & ((1 << (64 - k)) - 1)


def splitmix64(x: torch.Tensor) -> torch.Tensor:
    """splitmix64 finaliser on int64 tensors (two's complement wrap == mod 2^64)"""
    z = x + _i64(0x9E3779B97F4A7C15)
    z = (z ^ _lsr(z, 30)) * _i64(0xBF58476D1CE4E5B9)
    z = (z ^ _lsr(z, 27)) * _i64(0x94D049BB133111EB)
    return z ^ _lsr(z, 31)


def is_host(idx: torch.Tensor, seed: int = SEED) -> torch.Tensor:
    return (splitmix64(idx ^ _i64(seed)) & 1).bool()


def _bytes(s: str, device) -> torch.Tensor:
    return torch.tensor(list(s.encode()), dtype=torch.uint8, device=device)


def _digits(n: int) -> int:
    return len(str(n))


def fastq_size(n: int, start: int = 0, read_len: int = 150) -> int:
    total, lo = 0, start
    while lo < start + n:
        d = _digits(lo)
        hi = min(start + n, 10 ** d)
        total += (hi - lo) * (23 + 2 * read_len + d)
        lo = hi
    return total


def gen_fastq(n: int, mate: int = 1, seed: int = SEED, device="cpu", start: int = 0, out: torch.Tensor | None = None,
              read_len: int = 150) -> torch.Tensor:
    """n records syn.{start} .. syn.{start+n-1} of one mate file as a flat uint8 tensor"""
    g = torch.Generator(device=device)
    g.manual_seed((seed * 2 + mate) & 0x7FFFFFFF)
    lo = start
    classes = []
    while lo < start + n:
        d = _digits(lo)
        hi = min(start + n, 10 ** d)
        classes.append((lo, hi, d))
        lo = hi
    total = fastq_size(n, start, read_len)
    if out is None:
        out = torch.empty(total, dtype=torch.uint8, device=device)
    assert out.numel() >= total
    tail = _bytes(f" {mate}:N:0:ATCACG\n", device)
    acgt = _bytes("ACGT", device)
    pos = 0
    CH = 1 << 20  # records per chunk (bounds temporaries)
    for lo, hi, d in classes:
        L = 23 + 2 * read_len + d
        for a in range(lo, hi, CH):
            b = min(hi, a + CH)
            m = b - a
            buf = out[pos: pos + m * L].view(m, L)
            pos += m * L
            idx = torch.arange(a, b, dtype=torch.int64, device=device)
            buf[:, 0:5] = _bytes("@syn.", device)
            for k in range(d):
                buf[:, 5 + k] = ((idx // (10 ** (d - 1 - k))) % 10 + 48).to(torch.uint8)
            buf[:, 5 + d: 19 + d] = tail
            s0 = 19 + d
            bases = torch.randint(0, 4, (m, read_len), dtype=torch.uint8, device=device, generator=g)
            buf[:, s0: s0 + read_len] = acgt[bases.long()]
            buf[:, s0 + read_len] = 10
            buf[:, s0 + read_len + 1] = 43  # '+'
            buf[:, s0 + read_len + 2] = 10
            q0 = s0 + read_len + 3
            buf[:, q0: q0 + read_len] = torch.randint(33, 74, (m, read_len), dtype=torch.uint8, device=device,
                                                      generator=g)
            first = buf[:, q0]
            first[(idx % 64) == 0] = 64  # '@'
            first[(idx % 64) == 1] = 43  # '+'
            buf[:, q0 + read_len] = 10
    return out[:total]


def gen_fasta(n: int, mate: int = 1, wrap: int | None = None, crlf: bool = False, seed: int = SEED, device="cpu",
              start: int = 0, read_len: int = 150) -> torch.Tensor:
    """the gen_fastq records as FASTA (same ids and sequences, so the id lists and PAF generators apply):
    '>' header E sequence E, the sequence in lines of `wrap` bases (None: one line), E = CRLF when `crlf`.
    read_len=30_000 gives ONT-like long records (shard halo tests)."""
    fq = gen_fastq(n, mate, seed, device, start, read_len=read_len)
    e = _bytes("\r\n" if crlf else "\n", device)
    E = e.numel()
    w = read_len if not wrap else wrap
    n_lines = -(-read_len // w)
    parts, pos, lo = [], 0, start
    while lo < start + n:
        d = _digits(lo)
        hi = min(start + n, 10 ** d)
        m, L = hi - lo, 23 + 2 * read_len + d
        rows = fq[pos: pos + m * L].view(m, L)
        pos += m * L
        H = 17 + d  # header without '@' and '\n'
        out = torch.empty((m, 1 + H + E + read_len + n_lines * E), dtype=torch.uint8, device=device)
        out[:, 0] = 62  # '>'
        out[:, 1: 1 + H] = rows[:, 1: 1 + H]
        out[:, 1 + H: 1 + H + E] = e
        o, s0 = 1 + H + E, 19 + d
        for k in range(n_lines):
            a, b = k * w, min(read_len, (k + 1) * w)
            out[:, o: o + b - a] = rows[:, s0 + a: s0 + b]
            out[:, o + b - a: o + b - a + E] = e
            o += b - a + E
        parts.append(out.view(-1))
        lo = hi
    return torch.cat(parts) if parts else torch.empty(0, dtype=torch.uint8, device=device)


def _num_field(v: torch.Tensor, width: int):
    """left-aligned decimal rendering of non-negative int64 values: (chars [n,width], mask [n,width])"""
    dev = v.device
    nd = torch.ones_like(v)
    for k in range(1, width):
        nd = nd + (v >= 10 ** k).long()
    col = torch.arange(width, device=dev).unsqueeze(0)
    exp = (nd.unsqueeze(1) - 1 - col).clamp(min=0)
    p10 = torch.tensor([10 ** k for k in range(width)], dtype=torch.int64, device=dev)
    chars = ((v.unsqueeze(1) // p10[exp]) % 10 + 48).to(torch.uint8)
    return chars, col < nd.unsqueeze(1)


def _const_field(s: str, n: int, device):
    b = _bytes(s, device)
    return b.unsqueeze(0).expand(n, b.numel()), torch.ones((n, b.numel()), dtype=torch.bool, device=device)


def _choice_field(options: list[str], which: torch.Tensor):
    """per-row choice among strings of different lengths"""
    dev = which.device
    w = max(len(o) for o in options)
    tab = torch.zeros((len(options), w), dtype=torch.uint8, device=dev)
    lens = torch.tensor([len(o) for o in options], device=dev)
    for k, o in enumerate(options):
        tab[k, : len(o)] = _bytes(o, dev)
    col = torch.arange(w, device=dev).unsqueeze(0)
    return tab[which], col < lens[which].unsqueeze(1)


def _render(fields) -> torch.Tensor:
    chars = torch.cat([f[0] for f in fields], dim=1)
    mask = torch.cat([f[1] for f in fields], dim=1)
    return chars[mask]


# taxids used by the classifier config (all present in the extended report below)
KRAKEN_TAXA = ["9606", "40674", "562", "0"]  # human 40%, other Chordata 10%, bacterial 30%, unclassified 20%


def gen_kraken_reads(n: int, seed: int = SEED, device="cpu", start: int = 0, chunk: int = 1 << 21) -> torch.Tensor:
    """one line per pair: C|U \\t syn.{i} \\t taxid \\t 150|150 \\t kmer-LCA string"""
    parts = []
    for a in range(start, start + n, chunk):
        b = min(start + n, a + chunk)
        idx = torch.arange(a, b, dtype=torch.int64, device=device)
        r = _lsr(splitmix64(idx ^ _i64(seed ^ 0xC1A55)), 11).double() / float(1 << 53)
        host = is_host(idx, seed)
        # host reads are human (80%) or another chordate (20%); the rest bacterial (60%) / unclassified (40%)
        which = torch.where(host, torch.where(r < 0.8, 0, 1), torch.where(r < 0.6, 2, 3))
        m = b - a
        fields = [
            _choice_field(["C", "C", "C", "U"], which), _const_field("\tsyn.", m, device), _num_field(idx, 10),
            _const_field("\t", m, device), _choice_field(KRAKEN_TAXA, which),
            _const_field("\t150|150\t", m, device),
            _choice_field(["9606:45 0:20 9606:51 |:| 9606:116", "40674:30 1:86 |:| 0:116", "562:116 |:| 562:80 2:36",
                           "0:116 |:| 0:116"], which),
            _const_field("\n", m, device),
        ]
        parts.append(_render(fields))
    return torch.cat(parts) if len(parts) != 1 else parts[0]


def gen_kraken_report(n_filler: int = 5000) -> bytes:
    """the SURVEY 8c report extended to ~5k taxa (bacterial species after 'D Bacteria')"""
    rows = [
        ("U", 0, "unclassified", 200), ("R", 1, "root", 5), ("R1", 131567, "cellular organisms", 3),
        ("D", 2759, "Eukaryota", 2), ("D1", 33154, "Opisthokonta", 1), ("K", 33208, "Metazoa", 4),
        ("K1", 6072, "Eumetazoa", 0), ("K2", 33213, "Bilateria", 6), ("K3", 33511, "Deuterostomia", 7),
        ("P", 7711, "Chordata", 8), ("P1", 89593, "Craniata", 9), ("C", 40674, "Mammalia", 10),
        ("O", 9443, "Primates", 0), ("F", 9604, "Hominidae", 11), ("G", 9605, "Homo", 12),
        ("S", 9606, "Homo sapiens", 430), ("C", 8782, "Aves", 10), ("K3", 33317, "Protostomia", 13),
        ("P", 6656, "Arthropoda", 14), ("C", 50557, "Insecta", 30), ("D", 2, "Bacteria", 15),
        ("S", 562, "Escherichia coli", 180),
    ]
    out = []
    for code, tid, name, direct in rows:
        out.append(f"  1.50\t{direct + 7}\t{direct}\t{code}\t{tid}\t  {name}")
    for k in range(n_filler):
        out.append(f"  0.01\t{k % 9 + 1}\t{k % 9 + 1}\tS\t{1000000 + k}\t      Bacterium sp. {k}")
    return ("\n".join(out) + "\n").encode()


def gen_paf(n: int, seed: int = SEED, device="cpu", start: int = 0, mates: int = 2, chunk: int = 1 << 20
            ) -> torch.Tensor:
    """minimap2 sr-like PAF (12 columns + tags) for reads syn.{start..start+n-1}.

    Host reads get 1-2 lines per mate (alen ~ U{20..150}, mapq 60 w.p. 0.7 else U{0..59}) and, so that the
    set is exactly the host reads, one guaranteed passing line (alen 150, mapq 60) on mate 1; 5% of the
    non-host reads get one low-quality line (alen 30, mapq 10) that must fail -l 50 -c 0.5 -q 50.
    """
    parts = []
    for a in range(start, start + n, chunk):
        b = min(start + n, a + chunk)
        idx = torch.arange(a, b, dtype=torch.int64, device=device)
        host = is_host(idx, seed)
        m = b - a
        # up to 5 candidate lines per read: [sure, m1 extra, m2 first, m2 extra, nonhost low]
        lines = []
        for slot in range(5):
            h = splitmix64(idx * 8 + slot + _i64(seed))
            u1 = _lsr(h, 40) % 1000
            if slot == 0:
                on, alen, mapq = host, torch.full_like(idx, 150), torch.full_like(idx, 60)
            elif slot == 4:
                on, alen, mapq = (~host) & (u1 < 50), torch.full_like(idx, 30), torch.full_like(idx, 10)
            else:
                on = host & ((u1 < 500) if slot in (1, 3) else torch.ones_like(host))
                alen = 20 + _lsr(h, 8) % 131
                mapq = torch.where(_lsr(h, 20) % 10 < 7, torch.full_like(idx, 60), _lsr(h, 28) % 60)
            lines.append((on, alen, mapq))
        on = torch.stack([l[0] for l in lines], 1).reshape(-1)
        alen = torch.stack([l[1] for l in lines], 1).reshape(-1)[on]
        mapq = torch.stack([l[2] for l in lines], 1).reshape(-1)[on]
        rid = idx.repeat_interleave(5)[on]
        k = int(on.sum())
        qs = (150 - alen) // 2
        ts = 1000 + (rid * 7919) % 1000000
        fields = [
            _const_field("syn.", k, device), _num_field(rid, 10), _const_field("\t150\t", k, device),
            _num_field(qs, 3), _const_field("\t", k, device), _num_field(qs + alen, 3),
            _const_field("\t+\tchr7\t159345973\t", k, device), _num_field(ts, 8), _const_field("\t", k, device),
            _num_field(ts + alen, 8), _const_field("\t", k, device), _num_field(alen - alen // 20, 3),
            _const_field("\t", k, device), _num_field(alen, 3), _const_field("\t", k, device), _num_field(mapq, 2),
            _const_field("\ttp:A:P\tcm:i:12\ts1:i:140\ts2:i:0\tdv:f:0.0100\trl:i:0\n", k, device),
        ]
        parts.append(_render(fields))
    return torch.cat(parts) if len(parts) != 1 else parts[0]


def gen_txt_ids(n: int, seed: int = SEED, device="cpu", start: int = 0) -> torch.Tensor:
    """the depletion set of config 4 as a one-column TXT list (host reads only)"""
    idx = torch.arange(start, start + n, dtype=torch.int64, device=device)
    idx = idx[is_host(idx, seed)]
    k = idx.numel()
    return _render([_const_field("syn.", k, device), _num_field(idx, 10), _const_field("\n", k, device)])


def gen_ont_fastq(n: int, seed: int = SEED, device="cpu", mean_log: float = 8.6, sigma: float = 0.8,
                  min_len: int = 200, max_len: int = 500_000, group_bytes: int = 1 << 28):
    """ONT-like long reads: lognormal lengths, 36-char UUID-style ids.  Returns (fastq bytes, lengths, ids hex).
    Records are rendered in groups of about `group_bytes` so that the temporaries stay bounded (2 M reads = 30 GB)."""
    g = torch.Generator(device="cpu")
    g.manual_seed(seed & 0x7FFFFFFF)
    lens = torch.empty(n).log_normal_(mean_log, sigma, generator=g).clamp(min_len, max_len).long()
    rec = 1 + 36 + 1 + lens + 1 + 2 + lens + 1
    off = torch.zeros(n + 1, dtype=torch.int64)
    off[1:] = torch.cumsum(rec, 0)
    total = int(off[-1])
    out = torch.empty(total, dtype=torch.uint8, device=device)
    hexd = _bytes("0123456789abcdef", device)
    idx = torch.arange(n, dtype=torch.int64, device=device)
    uu = torch.empty((n, 36), dtype=torch.uint8, device=device)
    col = 0
    for k in range(36):
        if k in (8, 13, 18, 23):
            uu[:, k] = 45
        else:
            uu[:, k] = hexd[(_lsr(splitmix64(idx * 2 + (col // 16) + _i64(seed)), 4 * (col % 16)) & 15)]
            col += 1
    del idx
    # group boundaries: consecutive records of about group_bytes
    g0 = 0
    grp = 0
    while g0 < n:
        g1 = int(torch.searchsorted(off, off[g0] + group_bytes, right=True))
        g1 = max(g0 + 1, min(n, g1 - 1 if g1 > g0 + 1 else g1))
        base = int(off[g0])
        size = int(off[g1]) - base
        gd = torch.Generator(device=device)
        gd.manual_seed((seed + 17 + 7919 * grp) & 0x7FFFFFFF)
        r = torch.randint(0, 4, (size,), dtype=torch.uint8, device=device, generator=gd)
        # 'A','C','G','T' = 65, 67, 71, 84 from r = 0..3 without an index tensor
        o = 65 + r * 2 + (r == 2).to(torch.uint8) * 2 + (r == 3).to(torch.uint8) * 13
        del r
        start = (off[g0:g1] - base).to(device)
        lensd = lens[g0:g1].to(device)
        o[start] = 64
        for k in range(36):
            o[start + 1 + k] = uu[g0:g1, k]
        o[start + 37] = 10
        o[start + 38 + lensd] = 10
        o[start + 39 + lensd] = 43
        o[start + 40 + lensd] = 10
        o[start + 41 + 2 * lensd] = 10
        # qualities: any printable; make them distinct from bases so that framing bugs show up
        qmask = torch.zeros(size + 1, dtype=torch.int32, device=device)
        qmask[start + 41 + lensd] += 1
        qmask[start + 41 + 2 * lensd] -= 1
        inq = torch.cumsum(qmask[:size], 0, dtype=torch.int32).bool()
        del qmask
        o[inq] = o[inq] // 2 + 20  # 'A','C','G','T' -> 52,53,55,62 ('4','5','7','>')
        out[base: base + size] = o
        del o, inq
        g0 = g1
        grp += 1
    return out, lens, uu


def gen_ont_paf(lens: torch.Tensor, uu: torch.Tensor, seed: int = SEED, device="cpu", chunk: int = 1 << 18,
                max_lines: int = 15) -> torch.Tensor:
    """map-ont-style PAF for the reads of gen_ont_fastq: 1..max_lines alignments per read (mean 8), grouped by qname in
    read order -- the "many alignments per read" shape of BASELINE configs[2].  A read is host iff splitmix64(i ^ seed)
    & 1: its first line passes -l 50 -c 0.5 -q 50 (80 % of the read aligned, mapq 60), its other lines are random
    sub-alignments; every line of a non-host read has mapq < 50 and therefore fails whatever its length."""
    n = lens.numel()
    parts = []
    for a in range(0, n, chunk):
        b = min(n, a + chunk)
        idx = torch.arange(a, b, dtype=torch.int64, device=device)
        L = lens[a:b].to(device)
        host = is_host(idx, seed)
        k = 1 + _lsr(splitmix64(idx * 3 + _i64(seed ^ 0x0A7)), 17) % max_lines
        rid = torch.repeat_interleave(torch.arange(b - a, device=device), k)  # local read index per line
        first = torch.ones_like(rid, dtype=torch.bool)
        first[1:] = rid[1:] != rid[:-1]
        ln = torch.arange(rid.numel(), dtype=torch.int64, device=device)
        h = splitmix64((idx[rid] << 5) + ln + _i64(seed ^ 0xBEEF))
        Lr = L[rid]
        sure = first & host[rid]
        qs = torch.where(sure, Lr // 10, _lsr(h, 8) % (Lr - 60))
        span = torch.where(sure, Lr * 8 // 10, 30 + _lsr(h, 30) % (Lr - qs - 29))
        qe = qs + span
        mapq = torch.where(sure, torch.full_like(h, 60),
                           torch.where(host[rid], _lsr(h, 50) % 61, _lsr(h, 50) % 50))
        ts = 10_000 + _lsr(h, 20) % 100_000_000
        m = rid.numel()
        fields = [
            (uu[a:b].to(device)[rid], torch.ones((m, 36), dtype=torch.bool, device=device)),
            _const_field("\t", m, device), _num_field(Lr, 7), _const_field("\t", m, device), _num_field(qs, 7),
            _const_field("\t", m, device), _num_field(qe, 7),
            _choice_field(["\t+\tchr1\t248956422\t", "\t-\tchr7\t159345973\t"], (_lsr(h, 3) & 1)),
            _num_field(ts, 9), _const_field("\t", m, device), _num_field(ts + span, 9), _const_field("\t", m, device),
            _num_field(span - span // 12, 7), _const_field("\t", m, device), _num_field(span, 7),
            _const_field("\t", m, device), _num_field(mapq, 2),
            _const_field("\ttp:A:P\tcm:i:412\ts1:i:3301\ts2:i:0\tdv:f:0.0712\trl:i:57\n", m, device),
        ]
        parts.append(_render(fields))
    return torch.cat(parts) if len(parts) != 1 else parts[0]


def gen_fastq_illumina(n: int, mate: int = 1, seed: int = SEED, device="cpu", start: int = 0, read_len: int = 150
                       ) -> torch.Tensor:
    """2x150 records with Illumina-style 40-byte names `A00123:0456:H7ABCDEFG:1:TTTT:XXXXX:YYYYY` (instrument : run :
    flowcell : lane : tile : x : y, fixed width, unique per index) -- ids longer than the 15 bytes a slot holds inline,
    i.e. the fingerprint + key-arena path of the id set.  Record = 40 + 24 + 2 * read_len bytes."""
    g = torch.Generator(device=device)
    g.manual_seed((seed * 2 + mate + 77) & 0x7FFFFFFF)
    head = _bytes("@A00123:0456:H7ABCDEFG:1:", device)
    tail = _bytes(f" {mate}:N:0:ATCACG\n", device)
    L = head.numel() + 16 + tail.numel() + 2 * read_len + 4
    out = torch.empty(n * L, dtype=torch.uint8, device=device)
    CH = 1 << 20
    for a in range(0, n, CH):
        b = min(n, a + CH)
        m = b - a
        buf = out[a * L: b * L].view(m, L)
        idx = torch.arange(start + a, start + b, dtype=torch.int64, device=device)
        p = 0
        buf[:, p: p + head.numel()] = head
        p += head.numel()
        for val, width in ((1101 + idx // 10_000_000_000, 4), ((idx // 100_000) % 100_000, 5), (idx % 100_000, 5)):
            for k in range(width):
                buf[:, p + k] = ((val // (10 ** (width - 1 - k))) % 10 + 48).to(torch.uint8)
            p += width
            if width == 4 or p == head.numel() + 10:
                buf[:, p] = 58  # ':'
                p += 1
        buf[:, p: p + tail.numel()] = tail
        p += tail.numel()
        r = torch.randint(0, 4, (m, read_len), dtype=torch.uint8, device=device, generator=g)
        buf[:, p: p + read_len] = 65 + r * 2 + (r == 2).to(torch.uint8) * 2 + (r == 3).to(torch.uint8) * 13
        p += read_len
        buf[:, p] = 10
        buf[:, p + 1] = 43
        buf[:, p + 2] = 10
        p += 3
        buf[:, p: p + read_len] = torch.randint(33, 74, (m, read_len), dtype=torch.uint8, device=device, generator=g)
        buf[:, p + read_len] = 10
    return out


def gen_txt_ids_illumina(n: int, seed: int = SEED, device="cpu", start: int = 0) -> torch.Tensor:
    """the id list of the host reads (is_host) of gen_fastq_illumina"""
    idx = torch.arange(start, start + n, dtype=torch.int64, device=device)
    idx = idx[is_host(idx, seed)]
    k = idx.numel()
    w = lambda v, width: (torch.stack([(v // (10 ** (width - 1 - j))) % 10 + 48 for j in range(width)], 1).to(torch.uint8),
                          torch.ones((k, width), dtype=torch.bool, device=device))
    return _render([_const_field("A00123:0456:H7ABCDEFG:1:", k, device), w(1101 + idx // 10_000_000_000, 4),
                    _const_field(":", k, device), w((idx // 100_000) % 100_000, 5), _const_field(":", k, device),
                    w(idx % 100_000, 5), _const_field("\n", k, device)])
