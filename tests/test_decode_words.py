"""The word-wide FASTA reader (phenotypeseeker_b200/csrc/ps_decode_bits.h): the write pass's word step and the count
pass's chunk summary against a byte-at-a-time reader on the host (every line width 1..200, CRLF, TAB, lower case,
IUPAC, NUL, bytes >= 128, '>' at every byte of a word, headers over two and three chunks, chunks that start in a
header, every [jlo, jhi) edge and output alignment); on the GPU, both FASTA write passes against the oracle on text of
mixed line widths: the word-wide one (an all-FASTA launch) and the byte transducer's FASTA branch (the same files in
one launch with a FASTQ sample)."""
import os
import subprocess

import numpy as np
import pytest

from conftest import ROOT


def test_word_reader_equals_byte_transducer(tmp_path):
    exe = str(tmp_path / "decode_words_check")
    subprocess.check_call(["g++", "-O2", "-std=c++17", "-o", exe, os.path.join(ROOT, "tests", "native", "decode_words_check.cpp")])
    r = subprocess.run([exe], capture_output=True, text=True)
    assert r.returncode == 0 and r.stdout.startswith("OK"), r.stdout + r.stderr


def _mixed_width_fasta(rng, n_bases):
    """Contigs whose line width changes from contig to contig and inside a contig, with the odd bytes the reader
    has rules for. No NUL: the reference ends its input there and this reader breaks a window (DESIGN.md "Reader
    semantics"); the host check covers NUL."""
    parts = []
    done = 0
    ci = 0
    while done < n_bases:
        hdr = ">c%d " % ci + "x" * int(rng.choice([0, 5, 70, 150]))      # some headers span two or three chunks
        eol = "\r\n" if ci % 3 == 2 else "\n"
        body = rng.choice(list("ACGT"), size=int(rng.integers(200, 9000)))
        if ci % 2:
            low = rng.random(body.size) < 0.3
            body[low] = np.char.lower(body[low])
        odd = rng.random(body.size) < 0.004
        body[odd] = rng.choice(list("NnRYu-*\t"), size=int(odd.sum()))
        text = "".join(body)
        lines, i = [], 0
        while i < len(text):
            w = int(rng.choice([1, 7, 59, 60, 61, 70, 80, 200]))
            lines.append(text[i:i + w])
            i += w
        parts.append((hdr + eol + eol.join(lines) + eol).encode())
        if ci % 4 == 3:
            parts.append(b"ACGT\x80GGCA\xc1TT\xffAC\n")                        # bytes >= 128 break windows
        done += body.size
        ci += 1
    return b"".join(parts)


def _small_fastq(rng):
    """Two reads: a launch that holds it decodes with k_decode_write<0>, format per file."""
    reads = ["".join(rng.choice(list("ACGT"), size=n)) for n in (150, 97)]
    return "".join("@r%d\n%s\n+\n%s\n" % (i, r, "I" * len(r)) for i, r in enumerate(reads)).encode()


@pytest.mark.gpu
@pytest.mark.parametrize("decode", ["default", "mixed"])
def test_fasta_write_passes_on_mixed_line_widths(decode):
    from oracle import kmers as ok
    from phenotypeseeker_b200._native import Context
    from phenotypeseeker_b200.pipeline import unpack_rows
    rng = np.random.default_rng(31)
    files = [_mixed_width_fasta(rng, int(n)) for n in (50, 16_000, 40_000, 120_000, 300_000)]
    files.append(b"junk before the first record\n" + files[1])
    if decode == "mixed":
        files.append(_small_fastq(rng))
    lists = [ok.count_kmers(f, 16) for f in files]
    u = ok.union([l[0] for l in lists])
    c = Context(0)
    try:
        c.begin(16, len(files))
        c.add_samples(0, files)
        for s, l in enumerate(lists):
            km, ct = c.sample_kmers(s)
            assert np.array_equal(km, l[0]) and np.array_equal(ct, l[1]), s
        assert c.build_union() == len(u)
        assert np.array_equal(c.get_union(), u)
        assert np.array_equal(unpack_rows(c.get_rows(), len(files)), ok.presence_matrix(u, lists))
    finally:
        c.close()
