"""Generates tests/golden/ref_cases.npz: what the reference's own compiled functions return on the fixed and seeded inputs of
tests/test_fasta_ref_cpu.py and tests/test_ref_pins_cpu.py, so that those comparisons also run where
oracle/_ref/libldw_ref.so cannot be built.  Where the library is built, the tests compare the stored values with it as
well, which keeps this file pinned to the reference.

    python tests/golden/make_golden_ref_cases.py

The values come from oracle/_ref/libldw_ref.so when it is built.  Otherwise they come from the repository's restatements
of the same functions, which those tests pinned to the library bit for bit:
- ldw_oracle.read_fasta for kseq_read as its callers see it;
- ldw_oracle.extract_aln_param / extract_snps / coo_triplets for .extractAlnParam / .extractSNPs;
- ldw_oracle.fast_hadamard for .fastHadamard;
- post_oracle for the ARACNE helpers.
`source` in the file says which was used.  The inputs of the random-stream sample are stored beside their outputs.
"""
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
PATH = os.path.join(HERE, "ref_cases.npz")
ALPHABET = [b">", b"@", b"+", b"\n", b"\n", b"\r", b" ", b"\t", b"A", b"c", b"N", b"-", b"\0", b"x"]
PARTS = [b"ACGT", b"acgtn-", b"", b"AC GT", b"\r", b"+", b"II"]


def pack(lists):
    """A list of lists of byte strings as three flat arrays (bytes, length of each string, strings per list)."""
    flat = [s for lst in lists for s in lst]
    return (np.frombuffer(b"".join(flat), dtype=np.uint8).copy(), np.array([len(s) for s in flat], dtype=np.int64),
            np.array([len(lst) for lst in lists], dtype=np.int64))


def unpack(data, lens, counts):
    raw = data.tobytes()
    ends = np.cumsum(lens)
    flat = [raw[e - n:e] for e, n in zip(ends.tolist(), lens.tolist())]
    cut = np.concatenate([[0], np.cumsum(counts)]).tolist()
    return [flat[a:b] for a, b in zip(cut[:-1], cut[1:])]


def put_lists(out, key, lists):
    out[key + "__data"], out[key + "__len"], out[key + "__count"] = pack(lists)


def get_lists(gold, key):
    return unpack(gold[key + "__data"], gold[key + "__len"], gold[key + "__count"])


def load():
    """The stored cases ({} before the first generation, which imports the tests for their inputs)."""
    return dict(np.load(PATH)) if os.path.exists(PATH) else {}


def random_streams(seed, n):
    """A fixed seeded sample of the streams the two property tests of tests/test_fasta_ref_cpu.py draw: byte soup over
    ALPHABET, and header/line-shaped records (rows 0..n-1 alternate between the two kinds)."""
    rng = np.random.default_rng(seed)
    out = []
    for i in range(n):
        if i % 2 == 0:
            out.append(b"".join(ALPHABET[k] for k in rng.integers(0, len(ALPHABET), size=int(rng.integers(0, 61)))))
        else:
            s = bytearray()
            for r in range(int(rng.integers(1, 7))):
                eol = [b"\n", b"\r\n"][int(rng.integers(0, 2))]
                s += [b">", b"@"][int(rng.integers(0, 2))] + b"s%d some text" % r + eol
                for k in rng.integers(0, len(PARTS), size=int(rng.integers(0, 6))):
                    s += PARTS[k] + eol
            out.append(bytes(s))
    return out


def main():
    for p in (ROOT, os.path.join(ROOT, "oracle"), os.path.join(ROOT, "tests"), HERE):
        if p not in sys.path:
            sys.path.insert(0, p)
    import tempfile

    import ldw_oracle as O
    import post_oracle as PO
    import ref_lib as R
    import test_fasta_ref_cpu as TF
    import test_ref_pins_cpu as TP

    live = R.available()
    out = {"source": np.array("oracle/_ref/libldw_ref.so" if live else "oracle restatements")}
    tmp = tempfile.mkdtemp()

    def view(data):
        p = os.path.join(tmp, "x.fa")
        with open(p, "wb") as fh:
            fh.write(data)
        if live:
            names, seqs, _ = TF.reference_view(p)
            return names, seqs
        names, seqs = O.read_fasta(p)
        return [n.encode("latin-1") for n in names], seqs

    groups = {"hand": [TF.CASES[k] for k in sorted(TF.CASES)], "edge16k": [TF.edge16k_stream(t) for t in TF.EDGE16K_TOTALS],
              "random": random_streams(2024, 400)}
    for g, inputs in groups.items():
        views = [view(d) for d in inputs]
        put_lists(out, g + "_in", [[d] for d in inputs])
        put_lists(out, g + "_names", [v[0] for v in views])
        put_lists(out, g + "_seqs", [v[1] for v in views])

    crlf = TF.crlf_alignment_file()
    p = os.path.join(tmp, "crlf.fa")
    with open(p, "wb") as fh:
        fh.write(crlf)
    if live:
        ref = R.extractAlnParam(p, 0, 0.15, 0.01)
    else:
        names, seqs = O.read_fasta(p)
        ref = O.extract_aln_param(names, seqs, 0, 0.15, 0.01)
    out["crlf_shape"] = np.array([ref["num.seqs"], ref["seq.length"]], dtype=np.int64)
    out["crlf_pos"] = np.asarray(ref["pos"], dtype=np.int32)

    for seed in TP.ENC_SEEDS:
        aln, names, settings_ = TP.random_alignment(seed)
        p = os.path.join(tmp, "r.fa")
        TP.write_fasta(p, aln)
        seqs = [bytes(r) for r in aln]
        for k, (filt, gap, maf) in enumerate(settings_):
            key = f"enc_s{seed}_k{k}"
            if live:
                par = R.extractAlnParam(p, filt, gap, maf)
            else:
                par = O.extract_aln_param(names, seqs, filt, gap, maf)
            out[key + "_shape"] = np.array([par["num.seqs"], par["num.snps"], par["seq.length"]], dtype=np.int64)
            out[key + "_pos"] = np.asarray(par["pos"], dtype=np.int32)
            if par["num.snps"]:
                if live:
                    sn = R.extractSNPs(p, len(aln), par["num.snps"], par["pos"])
                    codes, table = R.codes_from_coo(sn, par["num.snps"], len(aln)), sn["ACGTN_table"]
                    coo = {c: sn[c] for c in O.coo_triplets(codes)}
                else:
                    d = O.extract_snps(seqs, len(aln), par["num.snps"], par["pos"])
                    codes, table, coo = d["codes"], d["ACGTN_table"], O.coo_triplets(d["codes"])
                out[key + "_codes"] = codes
                out[key + "_table"] = table
                for c, v in coo.items():
                    out[f"{key}_coo_{c}"] = np.asarray(v, dtype=np.int32)

    for s, mats in enumerate(TP.hadamard_inputs()):
        a = [m.copy(order="F") for m in mats]
        (R.fastHadamard(*a, ncores=3) if live else O.fast_hadamard(*a))
        out[f"had{s}"] = a[0]

    cols = {"row1": [], "rowany": [], "inter": [], "vpm": [], "trip": []}
    for x, y, ys, a, b, xs, yv, m1, m2, mi0 in TP.aracne_helper_inputs():
        if live:
            cols["row1"].append(R.compareToRow(x, np.array([y])))
            cols["rowany"].append(R.compareToRow(x, ys))
            cols["inter"].append(R.fast_intersect(a, b))
            cols["vpm"].append(R.vecPosMatch(xs, yv))
            cols["trip"].append(np.array([R.compareTriplet(m1, m2, mi0)]))
        else:
            cols["row1"].append(np.asarray(PO.compare_to_row(x, y), dtype=bool))
            cols["rowany"].append(np.isin(x, ys).any(axis=1))
            cols["inter"].append(np.asarray(PO.fast_intersect(a, b)))
            cols["vpm"].append(np.asarray(PO.vec_pos_match(xs, yv), dtype=float))
            cols["trip"].append(np.array([PO.compare_triplet(m1, m2, mi0)]))
    for k, v in cols.items():
        out["aracne_" + k] = np.concatenate(v).astype(np.float64)
        out["aracne_" + k + "_len"] = np.array([len(a) for a in v], dtype=np.int64)

    for t, (p1, p2, mi, chk) in enumerate(TP.run_aracne_inputs()):
        if live:
            import pytest
            with pytest.MonkeyPatch.context() as m:
                TP.use_reference_helpers(m)
                out[f"run_aracne{t}"] = np.asarray(PO.run_aracne(p1[chk], p2[chk], mi[chk], p1, p2, mi))
        else:
            out[f"run_aracne{t}"] = np.asarray(PO.run_aracne(p1[chk], p2[chk], mi[chk], p1, p2, mi))

    np.savez_compressed(PATH, **out)
    print(PATH, os.path.getsize(PATH), "bytes, source:", out["source"])


if __name__ == "__main__":
    main()
