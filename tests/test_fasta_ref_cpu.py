"""FASTA tokeniser (csrc/fasta_host.cpp) against the reference's OWN compiled reader: klib kseq as vendored in
src/kseq2.h:167-207, built unmodified into oracle/_ref/libldw_ref.so (oracle/Makefile, target `ref`).

CPU only (the reader is host code behind the C ABI; no device call is made)."""
import ctypes as C
import gzip
import os
import subprocess
import sys

import numpy as np
import pytest
from hypothesis import HealthCheck, given, settings
from hypothesis import strategies as st

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "oracle"))
sys.path.insert(0, os.path.join(ROOT, "tests", "golden"))
import make_golden_ref_cases as GC  # noqa: E402
import ref_lib  # noqa: E402

HAVE_REF = ref_lib.available()
needs_ref = pytest.mark.skipif(not HAVE_REF, reason="oracle/_ref not built and the reference sources absent")


def reference_view(path):
    """What the reference's callers see of each record: strlen() of the sequence and the C string of the name
    (src/getACGTNsites.cpp:36,51-52), for the records `while ((l = kseq_read(seq)) >= 0)` yields."""
    names, seqs, rc = ref_lib.kseq_read_all(path)
    seqs = [s.split(b"\0", 1)[0] for s in seqs]
    names = [n for n in names]  # c_char_p already stops at NUL
    return names, seqs, rc


def product_view(path, chunk=None):
    """ldw_read_fasta_alloc through ctypes, in a child process when a hand-over buffer size is forced (the library
    reads LDW_FASTA_CHUNK once per call, so an env change in-process works too; kept in-process for speed)."""
    from ldweaver_b200 import _lib
    L = _lib.lib()
    old = os.environ.pop("LDW_FASTA_CHUNK", None)
    if chunk is not None:
        os.environ["LDW_FASTA_CHUNK"] = str(chunk)
    try:
        nseq, slen, nlen = C.c_int64(), C.c_int64(), C.c_int64()
        aln_p, names_p = C.c_void_p(), C.c_void_p()
        _lib.check(L.ldw_read_fasta_alloc(os.fsencode(path), C.byref(nseq), C.byref(slen), C.byref(aln_p),
                                          C.byref(names_p), C.byref(nlen)))
        raw = C.string_at(names_p, nlen.value) if names_p else b""
        L.ldw_buffer_free(names_p)
        aln = None
        if aln_p:
            aln = C.string_at(aln_p, nseq.value * slen.value)
            L.ldw_buffer_free(aln_p)
        return nseq.value, slen.value, raw.split(b"\0")[:nseq.value], aln
    finally:
        os.environ.pop("LDW_FASTA_CHUNK", None)
        if old is not None:
            os.environ["LDW_FASTA_CHUNK"] = old


GOLD = GC.load()


def stored_views(group):
    """The reference reader's (names, sequences) for each stored input of `group` (tests/golden/ref_cases.npz)."""
    return list(zip(GC.get_lists(GOLD, group + "_names"), GC.get_lists(GOLD, group + "_seqs")))


def expected_view(want, path):
    """`want` (stored), checked against the compiled reader where it is built."""
    if HAVE_REF:
        names, seqs, _ = reference_view(path)
        assert (names, seqs) == tuple(want), "tests/golden/ref_cases.npz differs from the compiled reader"
    return want


def check_same(path, want, chunk=None):
    rnames, rseqs = want
    nseq, slen, names, aln = product_view(path, chunk)
    assert nseq == len(rseqs), (nseq, len(rseqs))
    assert names == rnames
    if nseq == 0:
        return
    lens = {len(s) for s in rseqs}
    if len(lens) > 1:
        assert slen == -1 and aln is None  # "Error! sequences are of different lengths!" src/getACGTNsites.cpp:54-56
        return
    assert slen == len(rseqs[0])
    if slen == 0:
        assert aln is None
    else:
        assert aln == b"".join(rseqs)


CASES = {
    "plain": b">a desc\nACGT\nAC\n>b\nTTTTGG\n",
    "crlf": b">a desc\r\nACGT\r\nAC\r\n>b\r\nTTTT\r\nGG\r\n",           # CR kept: 8 bytes per record, not 6
    "crlf_name_only": b">a\r\nACGT\r\n>b\r\nACGT\r\n",
    "inner_blanks": b">s1\tx y\nAC GT\n a c\t-n\n>s2 \nTTTT GGGG xxxxx\n",
    "empty_line_glues_next_line": b">a\nACGT\n\n>b\nAC\n",                 # one record: ACGT\n>bAC
    "empty_line_mid_record": b">a\nAC\n\nGT\n>b\nAC\nGTxx\n",
    "gt_inside_line_is_sequence": b">x\nAC>y\nGT\n",
    "at_line_starts_a_record": b">x\nACGT\n@y\nTTTT\n",
    "at_first": b"@x\nACGT\n>y\nTTTT\n",
    "junk_before_then_gt_mid_line": b"junk before >s1 c\nACGT\n>s2\nTTTT\n",
    "fastq": b"@r1\nACGT\n+\nIIII\n@r2\nTTTT\n+r2\nJJJJ\n",
    "fastq_multi_line_qual": b"@r1\nACGT\nAC\n+\nIII\nIII\n@r2\nTTTTTT\n+\nJJJJJJ\n",
    "fastq_then_fasta_skips_to_header": b"@r1\nACGT\n+\nIIII\njunk\n>r2\nTTTT\n",
    "fastq_qual_too_long_stops_reading": b">a\nACGT\n>b\nACGT\n+\nIIIII\n>c\nACGT\n",
    "fastq_qual_missing_stops_reading": b">a\nACGT\n>b\nACGT\n+",
    "fastq_qual_short_at_eof": b">a\nACGT\n>b\nACGT\n+\nII",
    "plus_with_empty_seq": b">a\n+\n\n>b\n+\n\n",
    "no_trailing_newline": b">x\nACGT\n>y\nTTTT",
    "header_only_at_eof": b">x\nACGT\n>y",
    "bare_header_char_at_eof": b">x\nACGT\n>",
    "empty_records": b">x\n>y\n",
    "empty": b"",
    "no_header": b"ACGT\nACGT\n",
    "embedded_nul": b">a\nAC\0T\n>b\nAC\n",
    "nul_in_name": b">a\0b c\nACGT\n>c\nACGT\n",
    "vertical_tab_ends_name": b">a\x0bb\nACGT\n>c\x0cd\nACGT\n",
    "lowercase_and_gaps": b">a\nacgtn-\n>b\nACGTN-\n",
    "one_long_line": b">only\n" + b"ACGTN-acgtn" * 5000 + b"\n",
}


@pytest.mark.parametrize("name", sorted(CASES))
def test_reader_matches_kseq_on_handwritten_files(tmp_path, name):
    i = sorted(CASES).index(name)
    assert GC.get_lists(GOLD, "hand_in")[i] == [CASES[name]]
    want = stored_views("hand")[i]
    p = tmp_path / (name + ".fa")
    p.write_bytes(CASES[name])
    expected_view(want, str(p))
    check_same(str(p), want)
    for chunk in (1, 2, 3, 7):
        check_same(str(p), want, chunk)
    q = tmp_path / (name + ".fa.gz")
    with gzip.open(q, "wb") as fh:
        fh.write(CASES[name])
    expected_view(want, str(q))
    check_same(str(q), want)


def test_documented_semantics_are_the_references(tmp_path):
    """The cases VERDICT/ADVICE name: the expected values come from the compiled kseq2.h, spelled out once here.  The
    reader is held to them everywhere; the compiled kseq2.h is checked against them too where it is built."""
    p = tmp_path / "crlf.fa"
    p.write_bytes(b">a\r\nACGT\r\nAC\r\n")
    if HAVE_REF:
        names, seqs, rc = reference_view(str(p))
        assert (names, seqs, rc) == ([b"a"], [b"ACGT\rAC\r"], -1)     # seq.length 8, where a whitespace stripper gives 6
    assert product_view(str(p))[:2] == (1, 8)
    assert product_view(str(p))[3] == b"ACGT\rAC\r"
    p.write_bytes(b">a\nACGT\n\n>b\nAC\n")
    if HAVE_REF:
        assert reference_view(str(p))[1] == [b"ACGT\n>bAC"]
    assert product_view(str(p))[3] == b"ACGT\n>bAC"


EDGE16K_TOTALS = (16384, 16383, 32768, 16385)


def edge16k_stream(total):
    body = b">a\n" + b"A" * (total - 3 - 2) + b"\n>"
    assert len(body) == total
    return body


def test_header_char_as_last_byte_of_a_16384_multiple_stream(tmp_path):
    """ks_getuntil only knows EOF after a short read (src/kseq2.h:87-98): a lone '>' closing a stream whose length is a
    multiple of the 16384-byte buffer yields one more, empty, record; any other length yields none."""
    for total, want in zip(EDGE16K_TOTALS, stored_views("edge16k")):
        p = tmp_path / f"t{total}.fa"
        p.write_bytes(edge16k_stream(total))
        expected_view(want, str(p))
        check_same(str(p), want)
        check_same(str(p), want, 5)


ALPHABET = [b">", b"@", b"+", b"\n", b"\n", b"\r", b" ", b"\t", b"A", b"c", b"N", b"-", b"\0", b"x"]


@needs_ref
@settings(max_examples=400, deadline=None, suppress_health_check=[HealthCheck.function_scoped_fixture])
@given(data=st.lists(st.sampled_from(ALPHABET), min_size=0, max_size=60).map(b"".join), chunk=st.sampled_from([None, 1, 2, 5]))
def test_reader_matches_kseq_on_random_byte_streams(tmp_path, data, chunk):
    p = tmp_path / "fuzz.fa"
    p.write_bytes(data)
    names, seqs, _ = reference_view(str(p))
    check_same(str(p), (names, seqs), chunk)


@needs_ref
@settings(max_examples=150, deadline=None, suppress_health_check=[HealthCheck.function_scoped_fixture])
@given(recs=st.lists(st.tuples(st.sampled_from([b">", b"@"]),
                               st.lists(st.sampled_from([b"ACGT", b"acgtn-", b"", b"AC GT", b"\r", b"+", b"II"]),
                                        min_size=0, max_size=5),
                               st.sampled_from([b"\n", b"\r\n"])), min_size=1, max_size=6),
       chunk=st.sampled_from([None, 1, 3]))
def test_reader_matches_kseq_on_record_shaped_streams(tmp_path, recs, chunk):
    out = bytearray()
    for k, (hdr, lines, eol) in enumerate(recs):
        out += hdr + b"s%d some text" % k + eol
        for ln in lines:
            out += ln + eol
    p = tmp_path / "fuzz2.fa"
    p.write_bytes(bytes(out))
    names, seqs, _ = reference_view(str(p))
    check_same(str(p), (names, seqs), chunk)


def test_reader_matches_kseq_on_a_stored_sample_of_random_streams(tmp_path):
    """The two property tests above on a fixed seeded sample of their streams (make_golden_ref_cases.random_streams),
    inputs and the reference reader's views stored: the comparison runs where the compiled reader is not built too."""
    streams = [s[0] for s in GC.get_lists(GOLD, "random_in")]
    assert streams == GC.random_streams(2024, len(streams))
    for i, (data, want) in enumerate(zip(streams, stored_views("random"))):
        p = tmp_path / "sample.fa"
        p.write_bytes(data)
        expected_view(want, str(p))
        check_same(str(p), want, (None, 1, 2, 5)[i % 4])


def test_two_call_reader_agrees_with_the_single_call_one(tmp_path):
    from ldweaver_b200 import _lib
    L = _lib.lib()
    p = tmp_path / "x.fa"
    p.write_bytes(b">a d\r\nACGT\r\nAC\r\n>b\r\nTTTT\r\nGG\r\n")
    nseq, slen = C.c_int64(), C.c_int64()
    _lib.check(L.ldw_read_fasta(os.fsencode(str(p)), C.byref(nseq), C.byref(slen), None, 0, None, 0))
    assert (nseq.value, slen.value) == (2, 8)
    aln = np.empty((2, 8), dtype=np.uint8)
    names = C.create_string_buffer(64)
    _lib.check(L.ldw_read_fasta(os.fsencode(str(p)), C.byref(nseq), C.byref(slen), aln.ctypes.data_as(C.c_void_p), aln.size,
                                names, 64))
    assert bytes(aln[0]) == b"ACGT\rAC\r" and bytes(aln[1]) == b"TTTT\rGG\r" and names.raw.split(b"\0")[:2] == [b"a", b"b"]


def crlf_alignment_file():
    rng = np.random.default_rng(5)
    nseq, L = 40, 300
    base = rng.choice(list(b"ACGT"), size=L)
    out = bytearray()
    for k in range(nseq):
        r = base.copy()
        m = rng.random(L) < 0.2
        r[m] = rng.choice(list(b"ACGTacgtN-"), size=int(m.sum()))
        r = bytes(r.astype(np.uint8))
        out += b">s%d\r\n" % k
        for o in range(0, L, 70):
            out += r[o:o + 70] + b"\r\n"
    return bytes(out)


def test_whole_encode_chain_on_a_crlf_alignment_matches_the_reference_host_side(tmp_path):
    """POS/seq.length after the tokeniser: the reference's extractAlnParam on a CRLF file counts the CR columns (class
    'other'); the product's reader must hand the same matrix to the device kernels (checked here on the host: the
    matrix bytes equal what kseq gives, and the oracle's filter on that matrix equals the reference's POS)."""
    import ldw_oracle as O
    L = 300
    p = tmp_path / "crlf_aln.fa"
    p.write_bytes(crlf_alignment_file())
    ref = {"num.seqs": int(GOLD["crlf_shape"][0]), "seq.length": int(GOLD["crlf_shape"][1]), "pos": GOLD["crlf_pos"]}
    if HAVE_REF:
        live = ref_lib.extractAlnParam(str(p), 0, 0.15, 0.01)
        assert (live["num.seqs"], live["seq.length"]) == (ref["num.seqs"], ref["seq.length"])
        np.testing.assert_array_equal(live["pos"], ref["pos"])
    nseq_p, slen_p, names, aln = product_view(str(p))
    assert (nseq_p, slen_p) == (ref["num.seqs"], ref["seq.length"]) and slen_p == L + 5  # five CRs per record
    seqs = [aln[i * slen_p:(i + 1) * slen_p] for i in range(nseq_p)]
    par = O.extract_aln_param([n.decode() for n in names], seqs, 0, 0.15, 0.01)
    assert np.array_equal(np.asarray(par["pos"], dtype=np.int32), ref["pos"])
