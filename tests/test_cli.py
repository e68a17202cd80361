"""The `abpoa` command line over libabpoa_b200 (abpoa_b200/bin/abpoa; reference src/abpoa.c) and its FASTA/FASTQ reader.

CPU part: the reader (poa_read_fastx, grammar of the reference's kseq-based abpoa_read_seq) on the reference's own
test inputs, plain and gzip-compressed.  GPU part: the real binary reproduces the md5 vectors recorded from the
reference CLI (SURVEY 8c / tests/golden/golden.json) and, in list mode (-l: all files as ONE GPU batch), prints
byte for byte what the reference binary prints for the same list (md5 stored, tests/golden_reference.py)."""
import ctypes as C
import gzip
import hashlib
import subprocess
from pathlib import Path

import numpy as np
import pytest

from abpoa_b200 import capi, synth
from abpoa_b200.aligner import decode
from helpers import INPUTS

ROOT = Path(__file__).resolve().parent.parent
BIN = ROOT / "abpoa_b200" / "bin" / "abpoa"
REF_BIN = ROOT / "oracle" / "_ref" / "abpoa_ref"      # the reference CLI (oracle/Makefile), only to record the stored md5


def read_with_library(lib, path):
    d = lib.dll
    d.poa_read_fastx.restype = C.c_int
    d.poa_read_fastx.argtypes = [C.c_char_p, C.c_void_p]
    ab = lib.abpoa_init()
    try:
        n = d.poa_read_fastx(str(path).encode(), ab.contents.abs)
        abs_ = ab.contents.abs.contents
        assert n == abs_.n_seq
        out = []
        for i in range(n):
            get = lambda f: (f[i].s[: f[i].l].decode() if f[i].l > 0 else "")
            out.append((get(abs_.name), get(abs_.comment), get(abs_.seq), get(abs_.qual)))
        return out
    finally:
        lib.abpoa_free(ab)


def simple_parse(path):
    lines = Path(path).read_text().splitlines()
    recs = []
    if lines and lines[0].startswith("@"):
        for i in range(0, len(lines) - 3, 4):
            name, _, comment = lines[i][1:].partition(" ")
            recs.append((name, comment, lines[i + 1], lines[i + 3]))
        return recs
    name = comment = None
    seq = []
    for ln in lines:
        if ln.startswith(">"):
            if name is not None:
                recs.append((name, comment, "".join(seq), ""))
            name, _, comment = ln[1:].partition(" ")
            seq = []
        else:
            seq.append(ln.strip())
    if name is not None:
        recs.append((name, comment, "".join(seq), ""))
    return recs


@pytest.mark.parametrize("fname", ["seq.fa", "test.fa", "heter.fa", "heter.fq", "3alleles.fa"])
def test_fastx_reader(product_lib, tmp_path, fname):
    want = simple_parse(INPUTS / fname)
    assert read_with_library(product_lib, INPUTS / fname) == want
    gz = tmp_path / (fname + ".gz")
    gz.write_bytes(gzip.compress((INPUTS / fname).read_bytes()))
    assert read_with_library(product_lib, gz) == want


def test_fastx_reader_multiline_and_crlf(product_lib, tmp_path):
    p = tmp_path / "m.fa"
    p.write_bytes(b">r1 first read\r\nACGT\r\nAC\r\n\r\n>r2\nGG\nTT\nA\n>r3\tx y\nC")
    assert read_with_library(product_lib, p) == [("r1", "first read", "ACGTAC", ""), ("r2", "", "GGTTA", ""), ("r3", "x y", "C", "")]


def md5_of(args):
    out = subprocess.run([str(BIN), *args], capture_output=True, check=True).stdout
    return hashlib.md5(out).hexdigest()


@pytest.mark.gpu
@pytest.mark.parametrize("args,md5", [
    (["-O", "4", "-E", "2"], "f1f63c16e4d9b905ef3a535861b285ba"),
    (["-O", "4", "-E", "2", "-r1"], "44ddefbbffa0cf93765d198ddd6595e6"),
    (["-O", "4", "-E", "2", "-r2"], "0820511c857d38df92cd4bac3a1eab40"),
    ([], "f1f63c16e4d9b905ef3a535861b285ba"),
])
def test_cli_md5_vectors_seq_fa(args, md5):
    """SURVEY 8c: md5 of the reference CLI's stdout on test_data/seq.fa."""
    assert md5_of([*args, str(INPUTS / "seq.fa")]) == md5


@pytest.mark.gpu
def test_cli_md5_vector_test_fa():
    assert md5_of([str(INPUTS / "test.fa")]) == "b3575081cd951243d4f3e6abec605212"


@pytest.mark.gpu
@pytest.mark.parametrize("opts", [[], ["-r1"], ["-r2"], ["-r5"], ["-m", "1", "-r2"], ["-Q", "-r2"]])
def test_cli_list_mode_matches_reference_binary(reference_lib, tmp_path, opts):
    """-l: every file is one read group; ours runs them as one GPU batch (device chain for consensus output, launch
    engine otherwise) and must print what the reference prints file by file.  The files are named relative to the
    working directory, so the list and the output are the same wherever the test runs."""
    files = []
    for g in range(7):
        reads = synth.make_group(7000 + g, 4 + g % 4, 150 + 60 * g, 0.06)
        p = tmp_path / f"g{g}.fa"
        p.write_text("".join(f">read{g}_{i} len={len(r)}\n{decode(r)}\n" for i, r in enumerate(reads)))
        files.append(p.name)
    for f in ("seq.fa", "heter.fq"):
        (tmp_path / f).write_bytes((INPUTS / f).read_bytes())
        files.append(f)
    lst = tmp_path / "list.txt"
    lst.write_text("".join(f"{p}\n" for p in files))
    run = lambda exe: subprocess.run([str(exe), *opts, "-l", lst.name], cwd=tmp_path, capture_output=True, check=True).stdout
    ours = run(BIN)
    question = (opts, [(tmp_path / f).read_bytes().decode() for f in files])
    ref = reference_lib.value("cli_list_md5", question, lambda lib: hashlib.md5(run(REF_BIN)).hexdigest())
    assert hashlib.md5(ours).hexdigest() == ref
