"""The bulk (memory-mapped, multi-threaded) FASTA reader of skch::Map gives exactly what the line reader gives
(reference seqiter.hpp:20-111 semantics), and declines what it cannot map (gzip, FASTQ). CPU only."""
import gzip
import os

import numpy as np
import pytest

from mashmap_b200 import hostlib


def write(path, data):
    with open(path, "wb") as f:
        f.write(data)
    return path


def random_bases(rng, n):
    return bytes(np.frombuffer(b"ACGTacgtNn", dtype=np.uint8)[rng.integers(0, 10, n)])


@pytest.mark.parametrize("threads", [1, 3, 16])
def test_bulk_reader_equals_line_reader(tmp_path, threads):
    rng = np.random.default_rng(3)
    recs = []
    for i in range(400):
        n = int(rng.choice([0, 1, 17, 59, 60, 61, 1000, 5000, 20011]))
        recs.append((f"read{i} some description\twith tab", random_bases(rng, n)))
    # single-line records, trailing newline
    a = b"".join(b">" + n.encode() + b"\n" + s + b"\n" for n, s in recs)
    # 60-column lines, an empty line here and there, '>' in the middle of a header, no newline at the end of the file
    b = b""
    for n, s in recs:
        b += b">" + n.encode() + b" >not a record\n"
        for o in range(0, len(s), 60):
            b += s[o : o + 60] + b"\n"
        if len(s) % 7 == 0:
            b += b"\n"
    b = b.rstrip(b"\n")
    # CRLF line ends (the reference keeps the '\r': so do both readers)
    c = a.replace(b"\n", b"\r\n")
    # headers without any space, one record only, record without sequence lines at the very end
    d = b">x\nACGT\n>y"
    for name, data in (("a.fa", a), ("b.fa", b), ("c.fa", c), ("d.fa", d)):
        p = write(str(tmp_path / name), data)
        diff, n_rec, n_bases = hostlib.fasta_readers_diff(p, threads)
        assert diff == 0, (name, diff)
        assert n_rec > 0
    assert hostlib.fasta_readers_diff(write(str(tmp_path / "a2.fa"), a), threads)[1] == len(recs)


def test_bulk_reader_declines_gzip_and_fastq(tmp_path):
    fa = b">r1\nACGTACGT\n>r2\nTTTT\n"
    gz = str(tmp_path / "x.fa.gz")
    with gzip.open(gz, "wb") as f:
        f.write(fa)
    fq = write(str(tmp_path / "x.fq"), b"@r1\nACGT\n+\nIIII\n@r2\nGG\n+\nII\n")
    assert hostlib.fasta_readers_diff(gz)[0] == -1 and hostlib.fasta_readers_diff(gz)[1] == 2
    assert hostlib.fasta_readers_diff(fq)[0] == -1 and hostlib.fasta_readers_diff(fq)[1] == 2


def test_host_packer_matches_the_format_statement():
    """seqio::pack_bases (AVX2 + scalar tail) == the numpy statement of the nibble format (capi.pack_bases): every byte
    value, lower case, IUPAC codes, odd lengths, lengths around the 32-byte vector width"""
    import numpy as np

    from mashmap_b200 import capi

    rng = np.random.default_rng(3)
    allbytes = np.arange(256, dtype=np.uint8)
    dna = np.frombuffer(b"ACGTacgtNnRYKM", dtype=np.uint8)[rng.integers(0, 14, size=5000)]
    for seq in (allbytes, dna, dna[:31], dna[:32], dna[:33], dna[:63], dna[:64], dna[:65], dna[:1], dna[:4999]):
        want = capi.pack_bases(seq)
        got = hostlib.pack_bases(seq)
        if len(seq) & 1:  # the unused high nibble of the last byte is an N in both
            assert want[-1] >> 4 == 8 and got[-1] >> 4 == 8
        assert np.array_equal(want, got), len(seq)


def _digest(lib_fn, *args):
    import ctypes as C

    n, b, d = C.c_uint64(), C.c_uint64(), C.c_uint64()
    rc = lib_fn(*args, C.byref(n), C.byref(b), C.byref(d))
    return rc, n.value, b.value, d.value


READER_GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "reference_reader.json")


def reader_files():
    """awkward FASTA files (and one FASTQ) of the reader comparison, as {file name: bytes}"""
    rng = np.random.default_rng(11)
    files = {}
    for v in range(12):
        recs = []
        for i in range(int(rng.integers(1, 60))):
            n = int(rng.choice([0, 1, 17, 59, 60, 61, 1000, 7001]))
            name = f"s{v}_{i}" + (" desc with\ttab" if rng.random() < 0.5 else "") + (" >inner" if rng.random() < 0.2 else "")
            recs.append((name, random_bases(rng, n)))
        width = int(rng.choice([0, 60, 80, 7]))
        data = b""
        for name, s in recs:
            data += b">" + name.encode() + b"\n"
            if width == 0:
                data += s + b"\n"
            else:
                for o in range(0, len(s), width):
                    data += s[o : o + width] + b"\n"
                if rng.random() < 0.2:
                    data += b"\n"
        if rng.random() < 0.3:
            data = data.rstrip(b"\n")
        if rng.random() < 0.25:
            data = data.replace(b"\n", b"\r\n")
        files[f"v{v}.fa"] = data
    files["fq.fq"] = b"".join(b"@r%d extra\n" % i + random_bases(rng, int(rng.integers(1, 300))) + b"\n+\n" + b"I" * 3 + b"\n" for i in range(40))
    return files


def test_both_readers_equal_the_reference_reader(tmp_path):
    """the reference's own reader (common/seqiter.hpp:20-111) against the product's line reader and its memory-mapped bulk
    reader on the same files: same records, same names, same bases (an FNV-1a digest over every name and sequence in
    order). Multi-line FASTA with blank lines, descriptions, '>' inside a header, CRLF ends (the '\\r' stays in the
    sequence in the reference, and in both readers), no newline at the end, a record without sequence, lower case and
    IUPAC letters; gzip and FASTQ for the line reader (the bulk reader declines them). The reference reader's digests of
    the plain and the gzip'ed file are stored in tests/golden/reference_reader.json (written through oracle/_ref by
    tests/golden/make_reference_reader.py)."""
    import ctypes as C
    import json

    H = hostlib.lib()
    H.skch_read_file_digest.argtypes = [C.c_char_p, C.c_int, C.c_int, C.POINTER(C.c_uint64), C.POINTER(C.c_uint64), C.POINTER(C.c_uint64)]
    with open(READER_GOLDEN) as f:
        reference = json.load(f)
    for name, data in reader_files().items():
        p = write(str(tmp_path / name), data)
        want, want_gz = (tuple(x) for x in reference[name])
        assert want_gz == want, name  # the reference reads the gzip'ed file as the plain one
        assert _digest(H.skch_read_file_digest, p.encode(), 0, 1) == want, name
        bulk = _digest(H.skch_read_file_digest, p.encode(), 1, 3)
        assert bulk == want or (bulk[0] == -1 and name.endswith(".fq")), name
        gz = str(tmp_path / (name + ".gz"))
        with gzip.open(gz, "wb") as f:
            f.write(data)
        assert _digest(H.skch_read_file_digest, gz.encode(), 0, 1) == want, name
