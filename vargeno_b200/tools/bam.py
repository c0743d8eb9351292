"""BAM (SAM/BAM specification section 4.2) writer and plain-Python FASTQ conversion: test and bench tooling for the device-side BAM
input (vgb_submit_bam).  A BAM file is BGZF (tools/bgzf) holding a header -- magic, SAM header text, reference names and lengths --
and then records, each prefixed with its length.

to_fastq() is the contract vgb_submit_bam implements, what `samtools fastq` writes with its default settings, with empty names:
secondary and supplementary records (flag 0x900) and records without bases are skipped, flag 0x10 is turned back to the sequenced
orientation (reverse complement, quality reversed), bases are =ACMGRSVTWYHKDBN, quality is qual + 33, or 1 ('"') for a record stored
without quality; more than 1022 bases, a bad magic, a truncated file and a record that fails the record check are errors."""
from __future__ import annotations

import struct
import zlib
from typing import Iterable, List, Optional, Sequence, Tuple

from . import bgzf

CODES = b"=ACMGRSVTWYHKDBN"
COMPLEMENT = b"=TGKCYSBAWRDMHVN"          # samtools' seq_comp_table, indexed by the 4-bit code
REC_MAX = 1 << 20                         # largest block_size the device accepts
SEQ_MAX = 1022


def header(refs: Sequence[Tuple[str, int]] = (), text: Optional[bytes] = None) -> bytes:
    """magic, l_text, text (default: @HD and one @SQ line per reference), n_ref, references"""
    if text is None:
        text = b"@HD\tVN:1.6\tSO:unsorted\n" + b"".join(b"@SQ\tSN:%s\tLN:%d\n" % (n.encode(), ln) for n, ln in refs)
    out = [b"BAM\x01", struct.pack("<i", len(text)), text, struct.pack("<i", len(refs))]
    for name, ln in refs:
        out.append(struct.pack("<i", len(name) + 1) + name.encode() + b"\0" + struct.pack("<i", ln))
    return b"".join(out)


def record(name: bytes, seq: bytes, qual: Optional[bytes], flag: int = 4, ref_id: int = -1, pos: int = -1, mapq: int = 0,
           cigar: Sequence[Tuple[int, int]] = (), next_ref_id: int = -1, next_pos: int = -1, tlen: int = 0, aux: bytes = b"") -> bytes:
    """One record.  seq: bases as text (lower case is stored upper case, as in BAM); qual: FASTQ quality characters (phred + 33),
    None for a record without quality; cigar: (length, op code) pairs; aux: raw tag bytes."""
    seq = seq.upper()
    codes = [CODES.index(bytes([b])) for b in seq]
    if len(codes) % 2:
        codes.append(0)
    packed = bytes((codes[i] << 4) | codes[i + 1] for i in range(0, len(codes), 2))
    q = b"\xff" * len(seq) if qual is None else bytes(c - 33 for c in qual)
    assert len(q) == len(seq)
    cig = b"".join(struct.pack("<I", (ln << 4) | op) for ln, op in cigar)
    core = struct.pack("<iiBBHHHIiii", ref_id, pos, len(name) + 1, mapq, 4680, len(cigar), flag, len(seq), next_ref_id, next_pos, tlen)
    body = core + name + b"\0" + cig + packed + q + aux
    return struct.pack("<i", len(body)) + body


def revcomp(seq: bytes) -> bytes:
    return bytes(COMPLEMENT[CODES.index(bytes([b]))] for b in reversed(seq.upper()))


def write(raw: bytes, **bgzf_args) -> bytes:
    """uncompressed BAM bytes (header + records) -> BGZF file (tools/bgzf.compress arguments: block, level, sizes)"""
    return bgzf.compress(raw, **bgzf_args)


def fastq_reads(text: bytes) -> List[Tuple[bytes, bytes, bytes]]:
    """(name, sequence, quality) of every record of FASTQ text"""
    lines = text.split(b"\n")
    return [(lines[i][1:], lines[i + 1], lines[i + 3]) for i in range(0, len(lines) - 3, 4)]


def inflate(buf: bytes) -> Tuple[bytes, List[int]]:
    """BGZF file -> its uncompressed bytes and the offset at which each member's bytes end"""
    out, ends, at = [], [], 0
    for off, size, poff, isize in bgzf.scan(buf):
        data = zlib.decompress(buf[off + poff:off + size - 8], -15)
        assert len(data) == isize
        if isize:
            out.append(data)
            at += isize
            ends.append(at)
    return b"".join(out), ends


def parse_header(raw: bytes) -> Tuple[int, int]:
    """(offset of the first record, n_ref); ValueError for a bad magic or a truncated header"""
    if raw[:4] != b"BAM\x01":
        raise ValueError("bad magic")
    if len(raw) < 12:
        raise ValueError("truncated header")
    l_text = struct.unpack_from("<i", raw, 4)[0]
    at = 8 + l_text
    if len(raw) < at + 4:
        raise ValueError("truncated header")
    n_ref = struct.unpack_from("<i", raw, at)[0]
    at += 4
    for _ in range(n_ref):
        if len(raw) < at + 4:
            raise ValueError("truncated header")
        at += 8 + struct.unpack_from("<i", raw, at)[0]
        if at > len(raw):
            raise ValueError("truncated header")
    return at, n_ref


def check(raw: bytes, o: int, n_ref: int) -> bool:
    """the record check of vgb_bam.cuh (bam_check): can a record start at raw[o]?"""
    if o + 36 > len(raw):
        return False
    bs, ref, _, l_name, _, _, n_cigar, _, l_seq, next_ref = struct.unpack_from("<iiiBBHHHIi", raw, o)
    if bs < 33 or bs > REC_MAX or not (-1 <= ref < n_ref) or not (-1 <= next_ref < n_ref) or l_name < 1:
        return False
    if 32 + l_name + 4 * n_cigar + (l_seq + 1) // 2 + l_seq > bs or o + 36 + l_name > len(raw):
        return False
    name = raw[o + 36:o + 36 + l_name]
    return name[-1] == 0 and all(0x21 <= c <= 0x7E for c in name[:-1])


def record_starts(raw: bytes) -> Tuple[List[int], int]:
    """offsets of every record, and n_ref"""
    at, n_ref = parse_header(raw)
    starts = []
    while at + 4 <= len(raw):
        starts.append(at)
        at += 4 + struct.unpack_from("<i", raw, at)[0]
    return starts, n_ref


def repair_share(raw: bytes, tile: int = 65536) -> Tuple[int, int]:
    """(tiles, tiles the chain walks again) of the device framing over the whole file at once: a tile is walked again when the
    first offset in it that passes the record check is not the first true record start at or behind the tile's start"""
    import bisect
    starts, n_ref = record_starts(raw)
    first = starts[0] if starts else len(raw)
    nt = (len(raw) - first + tile - 1) // tile
    repaired = 0
    for k in range(1, nt):
        a = first + k * tile
        i = bisect.bisect_left(starts, a)
        true = starts[i] if i < len(starts) else len(raw)
        if true >= min(a + tile, len(raw)) or any(check(raw, o, n_ref) for o in range(a, true)):
            repaired += 1
    return nt, repaired


def to_fastq(buf: bytes) -> bytes:
    """FASTQ text of a BAM file (BGZF bytes, or its uncompressed bytes): the contract of vgb_submit_bam"""
    raw = inflate(buf)[0] if buf[:2] == b"\x1f\x8b" else buf
    at, n_ref = parse_header(raw)
    out = []
    while at < len(raw):
        if at + 4 > len(raw):
            raise ValueError("truncated record")
        bs = struct.unpack_from("<i", raw, at)[0]
        if bs > REC_MAX:
            raise ValueError("record larger than 1 MiB")
        if not check(raw, at, n_ref):
            raise ValueError("truncated record" if at + 36 > len(raw) else "record fails the record check")
        if at + 4 + bs > len(raw):
            raise ValueError("truncated record")
        l_name, n_cigar, flag, l_seq = struct.unpack_from("<B", raw, at + 12)[0], *struct.unpack_from("<HHI", raw, at + 16)
        if not (flag & 0x900) and l_seq:
            if l_seq > SEQ_MAX:
                raise ValueError("record with more than 1022 bases")
            s = at + 36 + l_name + 4 * n_cigar
            packed = raw[s:s + (l_seq + 1) // 2]
            codes = [(packed[i // 2] >> (0 if i & 1 else 4)) & 15 for i in range(l_seq)]
            q = raw[s + (l_seq + 1) // 2:s + (l_seq + 1) // 2 + l_seq]
            qual = b'"' * l_seq if q[0] == 0xFF else bytes(c + 33 for c in q)
            if flag & 0x10:
                seq, qual = bytes(COMPLEMENT[c] for c in reversed(codes)), qual[::-1]
            else:
                seq = bytes(CODES[c] for c in codes)
            out.append(b"@\n" + seq + b"\n+\n" + qual + b"\n")
        at += 4 + bs
    return b"".join(out)


def ubam_fixed(text: bytes) -> bytes:
    """uncompressed unaligned BAM of FASTQ text whose records all have the same layout (name and read length: the bench's reads),
    built with numpy; the same bytes record() writes for them"""
    import numpy as np
    a = np.frombuffer(text, dtype=np.uint8)
    nl = np.flatnonzero(a == 10)
    rb = int(nl[3]) + 1
    n = a.size // rb
    assert n * rb == a.size and nl.size == 4 * n and (nl.reshape(n, 4) - rb * np.arange(n)[:, None] == nl[:4]).all(), "records differ in layout"
    r = a.reshape(n, rb)
    ln_name, L = int(nl[0]) - 1, int(nl[1] - nl[0]) - 1
    lut = np.zeros(256, np.uint8)
    for i, ch in enumerate(CODES):
        lut[ch] = i
        lut[bytes([ch]).lower()[0]] = i
    codes = lut[r[:, nl[0] + 1:nl[0] + 1 + L]]
    if L % 2:
        codes = np.concatenate([codes, np.zeros((n, 1), np.uint8)], axis=1)
    half = (L + 1) // 2
    bs = 32 + ln_name + 1 + half + L
    out = np.zeros((n, 4 + bs), np.uint8)
    out[:, :36] = np.frombuffer(struct.pack("<iiiBBHHHIiii", bs, -1, -1, ln_name + 1, 0, 4680, 0, 4, L, -1, -1, 0), np.uint8)
    out[:, 36:36 + ln_name] = r[:, 1:1 + ln_name]
    out[:, 37 + ln_name:37 + ln_name + half] = (codes[:, 0::2] << 4) | codes[:, 1::2]
    out[:, 37 + ln_name + half:] = r[:, nl[2] + 1:nl[2] + 1 + L] - 33
    return header() + out.tobytes()


def from_reads(reads: Iterable[Tuple[bytes, bytes, bytes]], refs: Sequence[Tuple[str, int]] = (), aligned: bool = False,
               extra_every: int = 0, seed: int = 1) -> bytes:
    """uncompressed BAM of FASTQ reads (name, seq, qual): unaligned (flag 4), or aligned-style -- every second read stored reverse
    complemented with flag 0x10, mapped to a reference with a CIGAR and aux tags, and, every `extra_every` reads, a secondary and a
    supplementary copy with a different sequence inserted (to_fastq skips them)"""
    import random
    rng = random.Random(seed)
    refs = list(refs) or [("chr1", 1000000)]
    out = [header(refs if aligned else [])]
    for i, (name, seq, qual) in enumerate(reads):
        if not aligned:
            out.append(record(name, seq, qual, aux=b"RGZfoo\0"))
            continue
        rev = i % 2 == 1
        s, q = (revcomp(seq), qual[::-1]) if rev else (seq, qual)
        ref = rng.randrange(len(refs))
        cig = [(len(seq), 0)] if seq else []
        aux = b"NMC" + bytes([rng.randrange(3)]) + b"MDZ" + str(len(seq)).encode() + b"\0"
        out.append(record(name, s, q, flag=0x10 if rev else 0, ref_id=ref, pos=rng.randrange(1000), mapq=60, cigar=cig, aux=aux))
        if extra_every and i % extra_every == 0 and seq:
            other = bytes(rng.choice(b"ACGT") for _ in range(len(seq)))
            out.append(record(name, other, qual, flag=0x100, ref_id=ref, pos=0, cigar=cig))
            out.append(record(name, other[: max(1, len(seq) // 2)], qual[: max(1, len(seq) // 2)], flag=0x800 | (0x10 if rev else 0),
                              ref_id=ref, pos=5, cigar=[(max(1, len(seq) // 2), 0)]))
    return b"".join(out)
