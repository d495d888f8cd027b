"""The MI scan across the range of its fixed-point count unit, and at the sequence-count edges of the K dimension.

The scan's epilogue rebuilds every joint allele table from int32 accumulators in a count unit of 2^sb weight units that
``build_plan`` sizes from the weights (ldweaver_b200/csrc/mi_scan.cu:171-199) so that a whole table fits 32 bits.  The
cases below put that arithmetic where it is thin:

 * all weights equal (``threshold = 0``, quirk Q7; or a population of isolated sequences, all weights 0.5), no N: the
   table total is 1.2-2 x 2^31 units and the corner cell (highest-coded class at both sites) of many pairs holds more
   than 2^31 units by itself;
 * ``sb = 0`` (2 and 3 sequences), ``sb`` capped at 14 with the pseudocount unit M halved (three clonal clusters of
   20 000), the largest supported sequence count 65 535 (512 K-blocks) and one over it;
 * 127 / 128 / 129 sequences (one pad column, none, a last K-block with one real sequence; S % 4 != 0 runs the
   scalar loop of the fp64 refinement) and the smallest block size, 128, next to 129.

Every case is checked against the fp64 C oracle: the dense fp32 epilogue cell by cell, the fp64 refinement on sampled
pairs, and a whole perform_MI_computation (short-range links, block thresholds, long-range link sets).
``test_cases_reach_their_regime`` restates the count-unit choice on the host and fails if a case no longer reaches the
regime it is here for (e.g. after the sizing rule is retuned); it needs no GPU.
"""
import math

import numpy as np
import pytest

import ldw_oracle as O
from util import compare_lr_sets

MI_TOL = 1e-6      # fp32 epilogue vs the fp64 reference (tests/test_gpu_mi.py)
EXACT_TOL = 1e-12  # fp64 refinement vs the fp64 reference
SR_DIST = 20000.0


# ------------------------------------------------------------------------------------------------ count-unit restatement
def count_unit(w):
    """Host restatement of build_plan's fixed-point count unit (ldweaver_b200/csrc/mi_scan.cu:163-199): the epilogue
    forms t = (H << sa) + (L >> sb), i.e. counts in units of 2^sb weight units, with the pseudocount 1/2 = M units and the
    weight scale = M * 2^(sb + 1) (weight units per unit of weight)."""
    w = np.asarray(w, dtype=np.float64)
    wmax, neff = float(w.max()), float(np.cumsum(w)[-1])     # summed in sequence order, as the host loop does
    total = (neff + 12.5) * 268435456.0 / wmax                # :176
    bits = 0
    while math.ldexp(1.0, bits) <= total:                     # :177-178
        bits += 1
    sb_raw = max(0, bits - 32)                                # :179
    sb = min(sb_raw, 14)                                      # :180
    unit2 = math.ldexp(1.0, sb + 1)                           # :187
    M0 = math.floor(268435455.0 / wmax / unit2)               # :188
    assert M0 >= 1
    M = min(M0, 1073741823)                                   # :190
    if (neff + 12.5) * (M * unit2) / math.ldexp(1.0, sb) >= 4294967295.0:   # :194-198
        while M > 1 and (neff + 12.5) * (M * unit2) / math.ldexp(1.0, sb) >= 4294967295.0:
            M >>= 1
    return dict(sb_raw=sb_raw, sb=sb, sa=14 - sb, M0=min(M0, 1073741823), M=M, scale=M * unit2, neff=neff, wmax=wmax,
                table_total=(neff + 12.5) * M * unit2 / math.ldexp(1.0, sb))


def fixed_point_weights(w, scale):
    """W_s = round(w_s * scale) with the error diffusion of build_plan (mi_scan.cu:218-235)."""
    W = np.zeros(len(w), dtype=np.int64)
    carry = 0.0
    for s in np.argsort(w, kind="stable"):
        x = float(w[s]) * scale + carry
        v = min(max(math.floor(x + 0.5), 0), 268435455)      # llround of a non-negative value
        carry = min(max(x - v, -1.0), 1.0)
        W[s] = v
    return W


def corner_units(codes, w, cu):
    """[nsnp, nsnp] corner cell of every pair in count units, including its pseudocount M: the cell of the two sites'
    complement classes (the highest class present, which owns no operand plane, mi_scan.cu:310-315), formed from the
    fixed-point weights' halves as the epilogue forms a cell.  The kernel derives the corner from marginals, which moves it
    by a few units (floor of the low halves) -- immaterial for the 2^31 count below."""
    W = fixed_point_weights(w, cu["scale"])
    H, L = (W >> 14).astype(np.float64), (W & 16383).astype(np.float64)
    top = np.array([max(np.unique(c)) for c in codes])
    A = (codes == top[:, None]).astype(np.float64)            # sums below stay < 2^40: exact in fp64
    return ((A * H) @ A.T).astype(np.int64) * (1 << cu["sa"]) + (((A * L) @ A.T).astype(np.int64) >> cu["sb"]) + cu["M"]


def overflowing_pairs(codes, w, cu):
    c = corner_units(codes, w, cu)
    iu = np.triu_indices(len(codes), 1)
    return int(np.count_nonzero(c[iu] >= 1 << 31)), len(iu[0])


# ------------------------------------------------------------------------------------------------ case inputs
def _positions(rng, n, g=2221315):
    return np.sort(rng.choice(np.arange(1, g + 1), size=n, replace=False)).astype(np.int32), g


def equal_weight_input(S, seed, nsnp=2000):
    """The benchmark's generator without N (every cell an A/C/G/T call)."""
    from ldweaver_b200 import synth
    sy = synth.generate(nseq=S, nsnp=nsnp, seed=seed, n_rate=0.0)
    return sy.codes, sy.POS, sy.g


def isolated_input(S=616, nsnp=2000, seed=5):
    """Independent N-free sites: every pair of sequences differs at ~30 % of the sites, far above 0.1 * nsnp, so every
    sequence is its own only neighbour (weight 0.5).  At half of the sites the highest-coded allele is the major one."""
    rng = np.random.default_rng(seed)
    maf = rng.uniform(0.02, 0.3, size=nsnp)
    pair = np.stack([np.sort(rng.choice(4, 2, replace=False)) for _ in range(nsnp)])
    major_hi = rng.random(nsnp) < 0.5
    major = np.where(major_hi, pair[:, 1], pair[:, 0])
    minor = np.where(major_hi, pair[:, 0], pair[:, 1])
    codes = np.where(rng.random((nsnp, S)) < maf[:, None], minor[:, None], major[:, None]).astype(np.uint8)
    POS, g = _positions(rng, nsnp)
    return codes, POS, g


def tiny_input(S, nsnp=300, seed=3):
    """S = 2 or 3 sequences, random N-free sites with at least two classes."""
    rng = np.random.default_rng(seed + S)
    codes = rng.integers(0, 4, size=(nsnp, S)).astype(np.uint8)
    for c in codes:
        while len(np.unique(c)) < 2:
            c[:] = rng.integers(0, 4, S)
    POS, g = _positions(rng, nsnp)
    return codes, POS, g


CLONE_SIZE, N_CLONES = 20000, 3


def clonal_input(nsnp=300, seed=9):
    """Three clusters of 20 000 sequences: founders >= 0.4 * nsnp apart, each sequence differs from its founder at <= 2 %
    of the sites.  Within a cluster distances are <= 4 % of the sites, across clusters >= 36 %, so at threshold 0.1 every
    sequence has exactly 20 000 neighbours counting itself: weight 1 / 20001 by construction."""
    rng = np.random.default_rng(seed)
    lo = rng.integers(0, 3, size=nsnp)
    hi = lo + 1 + rng.integers(0, 3 - lo)                      # two distinct classes per site, lo < hi <= 3
    # every site polymorphic among the founders: one founder (the odd one out) carries the other class
    odd = rng.integers(0, N_CLONES, size=nsnp)
    pick = (np.arange(N_CLONES)[None, :] == odd[:, None]) ^ (rng.random(nsnp) < 0.5)[:, None]
    f = np.where(pick, hi[:, None], lo[:, None])
    S = CLONE_SIZE * N_CLONES
    codes = np.repeat(f, CLONE_SIZE, axis=1)
    k = int(0.02 * nsnp)
    sites = np.argsort(rng.random((S, nsnp)), axis=1)[:, :k].ravel()   # k distinct sites per sequence
    seqs = np.repeat(np.arange(S), k)
    # a mutation takes the founders' other class, or (one in five) a third class: sites with r = 2 and r = 3
    third = np.array([min({0, 1, 2, 3} - {a, b}) for a, b in zip(lo, hi)])
    other = np.where(codes[sites, seqs] == lo[sites], hi[sites], lo[sites])
    codes[sites, seqs] = np.where(rng.random(len(sites)) < 0.2, third[sites], other)
    POS, g = _positions(rng, nsnp)
    return np.ascontiguousarray(codes.astype(np.uint8)), POS, g, f


def max_s_input(S=65535, nsnp=256, seed=65535):
    codes, POS, g = equal_weight_input(S, seed, nsnp)
    w = np.ones(S)
    w[S // 2 + 1:] = 0.5                                       # half 1, half 0.5
    return codes, POS, g, w


def multiallelic_nrich_input(nsnp=3 * 128 + 1, S=300, seed=42):
    """Multi-allelic, N-rich data (as tests/test_gpu_mi.py::test_multiallelic_nrich_vs_oracle), SNPs ordered so that the
    first 129 all have r = 3: with blk = 129 the first range's 2-plane group has 129 members (two row tiles, the second
    with one real row); with blk = 128 the last range holds one SNP."""
    rng = np.random.default_rng(seed)
    m = 4 * nsnp
    nall = rng.choice([2, 3, 4], size=m, p=[0.5, 0.3, 0.2])
    founders = np.stack([rng.integers(0, k, size=10) for k in nall]).astype(np.uint8)
    codes = founders[:, rng.integers(0, 10, size=S)]
    flip = rng.random((m, S)) < 0.05
    codes[flip] = (codes[flip] + 1) % np.repeat(nall, S).reshape(m, S)[flip]
    codes[rng.random((m, S)) < 0.08] = 4
    r = np.array([len(np.unique(c)) for c in codes])
    r3, rest = np.nonzero(r == 3)[0], np.nonzero((r >= 2) & (r != 3))[0]
    take = np.concatenate([r3[:129], np.sort(np.concatenate([r3[129:], rest]))[:nsnp - 129]])
    POS, g = _positions(rng, nsnp, 100000)
    return np.ascontiguousarray(codes[take]), POS, g


# ------------------------------------------------------------------------------------------------ regime test (no GPU)
def _hdw_host(codes, threshold):
    snp = O.snp_dat_from_codes(codes, np.arange(1, len(codes) + 1), None)
    return O.estimate_Hamming_distance_weights(snp, threshold)


def test_cases_reach_their_regime():
    report = {}
    # equal weights, no N: corner >= 2^31 units for a share of the pairs
    for name, S, seed, lo, hi in (("uniform", 300, 11, 1.1, 1.25), ("top", 499, 12, 1.9, 2.0)):
        codes, _, _ = equal_weight_input(S, seed)
        assert np.all(codes < 4)
        w = _hdw_host(codes, 0.0)
        assert np.all(w == 1.0)                                # quirk Q7: threshold 0 -> every weight 1
        cu = count_unit(w)
        n_over, n_pairs = overflowing_pairs(codes, w, cu)
        report[name] = (cu["sb"], cu["table_total"] / 2 ** 31, n_over / n_pairs)
        assert cu["sb"] >= 1 and lo < cu["table_total"] / 2 ** 31 < hi and n_over > 0
    codes, _, _ = isolated_input()
    w = _hdw_host(codes, 0.1)
    assert np.all(w == 0.5)
    cu = count_unit(w)
    n_over, n_pairs = overflowing_pairs(codes, w, cu)
    report["isolated"] = (cu["sb"], cu["table_total"] / 2 ** 31, n_over / n_pairs)
    assert cu["table_total"] > 2 ** 31 and n_over > 0
    # sb = 0: the accumulators' high half is shifted by the full 14 bits
    for S in (2, 3):
        codes, _, _ = tiny_input(S)
        assert all(len(np.unique(c)) >= 2 for c in codes) and np.all(codes < 4) and S % 4 != 0
        cu = count_unit(np.ones(S))
        assert cu["sb"] == 0 and cu["sa"] == 14
    # sb capped at 14, then M halved until a table fits 32 bits
    codes, _, _, f = clonal_input()
    nsnp = len(codes)
    fd = [np.count_nonzero(f[:, a] != f[:, b]) for a in range(N_CLONES) for b in range(a + 1, N_CLONES)]
    own = np.repeat(f, CLONE_SIZE, axis=1)
    per_seq = np.count_nonzero(codes != own, axis=0)
    thresh = int(nsnp * 0.1)
    assert min(fd) - 2 * per_seq.max() >= thresh and 2 * per_seq.max() < thresh   # weight 1/20001 by construction
    assert np.all(codes < 4) and all(len(np.unique(c)) >= 2 for c in codes)
    cu = count_unit(np.full(CLONE_SIZE * N_CLONES, 1.0 / (CLONE_SIZE + 1)))
    report["clonal"] = (cu["sb_raw"], cu["sb"], cu["M0"], cu["M"])
    assert cu["sb_raw"] == 15 and cu["sb"] == 14 and cu["M"] == cu["M0"] >> 1
    # the largest supported sequence count
    codes, _, _, w = max_s_input()
    S = codes.shape[1]
    assert S == 65535 and S % 4 != 0 and -(-S // 128) == 512 and np.all(codes < 4)
    cu = count_unit(w)
    n_over, n_pairs = overflowing_pairs(codes, w, cu)
    report["max_s"] = (cu["sb"], cu["table_total"] / 2 ** 31, n_over / n_pairs)
    assert 1.4 < cu["table_total"] / 2 ** 31 < 1.6 and n_over > 0
    # smallest blocks: a one-SNP last range (blk 128) and a 129-member plane group (blk 129)
    codes, _, _ = multiallelic_nrich_input()
    r = np.array([len(np.unique(c)) for c in codes])
    assert len(codes) % 128 == 1 and np.all(r[:129] == 3) and set(r) >= {3, 4, 5}
    print("regimes:", report)


# ------------------------------------------------------------------------------------------------ GPU cases
def _paint(n):
    p = np.ones(n, dtype=np.int32)
    p[n // 3:] = 2
    p[2 * n // 3:] = 3
    return p


def _check_case(name, codes, POS, g, hdw, blk, retain, exact_sr=False, n_sample=4000, seed=0):
    """Every block of the plan (blk: make_blocks block size, off-diagonal blocks included): the dense fp32 epilogue cell by
    cell and the fp64 refinement on sampled pairs against the C oracle; then perform_MI_computation on the same plan:
    short-range links (positions exact, MI within MI_TOL, or EXACT_TOL with the in-scan fp64 values), block thresholds,
    probabilities and long-range link sets against the oracle's block_links."""
    import c_oracle as CO
    import ldweaver_b200 as ldw
    from ldweaver_b200 import synth
    n = len(codes)
    osnp = O.snp_dat_from_codes(codes, POS, g)
    snp = ldw.snp_dat_from_codes(codes, POS, g)
    paint = _paint(n)
    P = np.asarray(POS, dtype=np.float64)
    lra = synth.exact_lr_links_approx(POS, g, SR_DIST)
    rng = np.random.default_rng(seed)
    plan = ldw.MIPlan(snp, hdw, paint, blk)
    try:
        blocks, w32, w64 = [], 0.0, 0.0
        for bi, (fs, fe, ts, te) in enumerate(O.make_blocks(n, blk)):
            f, t = np.arange(fs - 1, fe), np.arange(ts - 1, te)
            ref = CO.block_mi(codes, hdw, osnp.r, osnp.uqe, f, t)
            MI = plan.block_dense(bi)
            assert MI.shape == ref.shape
            w32 = max(w32, float(np.abs(MI - ref).max()))
            il, jl = rng.integers(0, len(f), n_sample), rng.integers(0, len(t), n_sample)
            w64 = max(w64, float(np.abs(plan.pairs_exact(bi, il, jl) - ref[il, jl]).max()))
            blocks.append((f, t, CO.block_links(ref, P, f, t, float(g), SR_DIST, retain, lra)))
        res = ldw.perform_MI_computation(snp, hdw, ldw.CdsVar(paint, 3), sr_dist=SR_DIST, lr_retain_links=retain,
                                         lr_links_approx=lra, write_tsv=False, plan=plan,
                                         exact_sr="in_scan" if exact_sr else None)
    finally:
        plan.close()
    wsr, wthr = 0.0, 0.0
    for bi, (f, t, L) in enumerate(blocks):
        k = res.sr["block"] == bi
        np.testing.assert_array_equal(res.sr["pos1"][k], P[t[L["col"]]][L["is_sr"]].astype(np.int32))
        np.testing.assert_array_equal(res.sr["pos2"][k], P[f[L["row"]]][L["is_sr"]].astype(np.int32))
        if k.any():
            wsr = max(wsr, float(np.abs(res.sr["MI"][k] - L["MI"][L["is_sr"]]).max()))
        if not np.isnan(L["thr"]) and not np.isnan(res.thr[bi]):
            wthr = max(wthr, abs(res.thr[bi] - L["thr"]))
    st = res.stats
    print(f"\n{name}: S={codes.shape[1]} nsnp={n} blk={blk} blocks={len(blocks)}: max |dMI| dense fp32 {w32:.3e}, "
          f"pairs_exact {w64:.3e}, short-range {'fp64 in-scan' if exact_sr else 'fp32'} {wsr:.3e}; max |dthr| {wthr:.3e}; "
          f"eps_obs_max {st['eps_obs_max']:.3e}; n_reruns {st['n_reruns']}; sr {len(res.sr['MI'])} lr {len(res.lr['MI'])}")
    assert w32 < MI_TOL, f"dense fp32 epilogue: {w32}"
    assert w64 < EXACT_TOL, f"pairs_exact: {w64}"
    assert wsr < (EXACT_TOL if exact_sr else MI_TOL), f"short-range MI: {wsr}"
    nb = 0
    for bi, (f, t, L) in enumerate(blocks):
        if np.isnan(L["thr"]):
            assert np.isnan(res.thr[bi])
            continue
        assert abs(res.thr[bi] - L["thr"]) < EXACT_TOL, (bi, res.thr[bi], L["thr"])
        assert res.prob[bi] == L["prob"]
        kk = res.lr["block"] == bi
        _, a, b = compare_lr_sets(P[t[L["col"]]][L["lr_keep"]], P[f[L["row"]]][L["lr_keep"]], L["MI"][L["lr_keep"]],
                                  res.lr["pos1"][kk], res.lr["pos2"][kk], res.lr["MI"][kk], L["thr"])
        nb += len(a) + len(b)
    assert st["eps_obs_max"] < MI_TOL
    return res, nb


@pytest.fixture(scope="module")
def uniform_case():
    """300 sequences, no N, weights through the device HDW at threshold 0 (quirk Q7: every weight 1)."""
    import ldweaver_b200 as ldw
    codes, POS, g = equal_weight_input(300, 11)
    hdw = ldw.estimate_Hamming_distance_weights(ldw.snp_dat_from_codes(codes, POS, g), 0.0)
    assert np.all(hdw == 1.0)
    return codes, POS, g, hdw


@pytest.mark.gpu
def test_equal_weights_corner_above_2_31(uniform_case):
    codes, POS, g, hdw = uniform_case
    _check_case("uniform 300, weights 1", codes, POS, g, hdw, 1000, 5e4)


@pytest.mark.gpu
def test_equal_weights_in_scan_exact_short_range(uniform_case):
    """LDW_SCAN_SR_EXACT on the same input: the fp64 corner-from-marginals path (refine_pair) at its heaviest corner."""
    codes, POS, g, hdw = uniform_case
    _check_case("uniform 300, in-scan exact SR", codes, POS, g, hdw, 1000, 5e4, exact_sr=True)


@pytest.mark.gpu
def test_equal_weights_top_of_the_bracket():
    """499 sequences of weight 1: the table total is just below 2^32 units, so t reaches ~2^32 in the fp32 conversion."""
    codes, POS, g = equal_weight_input(499, 12)
    _check_case("top of the bracket 499, weights 1", codes, POS, g, np.ones(499), 1000, 5e4)


@pytest.mark.gpu
def test_all_sequences_isolated():
    """A diverse population (no two sequences within 0.1 * nsnp): every weight 0.5, the equal-weight regime reached the
    way real data reaches it."""
    import ldweaver_b200 as ldw
    codes, POS, g = isolated_input()
    hdw = ldw.estimate_Hamming_distance_weights(ldw.snp_dat_from_codes(codes, POS, g), 0.1)
    assert np.all(hdw == 0.5)
    _check_case("all isolated 616, weights 0.5", codes, POS, g, hdw, 1000, 5e4)


@pytest.mark.gpu
@pytest.mark.parametrize("S", [2, 3])
def test_count_unit_sb0(S):
    codes, POS, g = tiny_input(S)
    _check_case(f"sb = 0, S = {S}", codes, POS, g, np.ones(S), 128, 2000)


@pytest.mark.gpu
@pytest.mark.parametrize("S", [127, 128, 129])
def test_k_block_edges(S):
    """One pad column (127), none (128), a last K-block holding one real sequence (129); weights through the device HDW
    (checked against the C oracle at these counts too)."""
    import c_oracle as CO
    import ldweaver_b200 as ldw
    from ldweaver_b200 import synth
    sy = synth.generate(nseq=S, nsnp=2000, seed=S)
    hdw = ldw.estimate_Hamming_distance_weights(ldw.snp_dat_from_codes(sy.codes, sy.POS, sy.g), 0.1)
    np.testing.assert_array_equal(hdw, CO.hdw(sy.codes, 0.1)[0])
    _check_case(f"K-block edge S = {S}", sy.codes, sy.POS, sy.g, hdw, 1000, 5e4)


@pytest.mark.gpu
def test_count_unit_cap_and_pseudocount_shrink():
    """60 000 sequences in three clonal clusters: (neff + 12.5) / max(w) > 2^18, so sb is capped at 14 and M halved.
    The weights come from the device HDW's fused path (no distance matrix) at 6 x the sequences of C3 and must be
    exactly 1/20001 (by construction, see clonal_input)."""
    import ldweaver_b200 as ldw
    codes, POS, g, _ = clonal_input()
    hdw = ldw.estimate_Hamming_distance_weights(ldw.snp_dat_from_codes(codes, POS, g), 0.1)
    np.testing.assert_array_equal(hdw, np.full(CLONE_SIZE * N_CLONES, 1.0 / (CLONE_SIZE + 1)))
    _check_case("sb cap + M shrink, 3 x 20000 clonal", codes, POS, g, hdw, 128, 2000, n_sample=2000)


@pytest.mark.gpu
def test_largest_supported_sequence_count():
    """65 535 sequences (512 K-blocks, S % 4 != 0), half of weight 1 and half of weight 0.5: the int32 accumulation at
    its documented limit and corner cells above 2^31 units."""
    codes, POS, g, w = max_s_input()
    _check_case("nseq = 65535", codes, POS, g, w, 128, 2000, n_sample=2000)


@pytest.mark.gpu
def test_one_sequence_over_the_limit_is_refused():
    import ldweaver_b200 as ldw
    from ldweaver_b200 import _lib
    rng = np.random.default_rng(1)
    codes = rng.integers(0, 2, size=(4, 65536)).astype(np.uint8)
    snp = ldw.snp_dat_from_codes(codes, np.array([10, 20, 30, 40]), 1000)
    with pytest.raises(_lib.LdwError, match="nseq > 65535") as e:
        ldw.MIPlan(snp, np.ones(65536), np.ones(4, dtype=np.int32), 128)
    assert e.value.code == 4   # LDW_ERR_UNSUPPORTED


@pytest.mark.gpu
@pytest.mark.parametrize("blk", [128, 129])
def test_smallest_blocks(blk):
    """blk = 128 (the minimum): a last range of one SNP (a 128 x 1 off-diagonal block, quirk Q1 ragged, Q2 drop) and a
    plane group of one member; blk = 129: a plane group of 129 members (a row tile with one real row)."""
    import c_oracle as CO
    codes, POS, g = multiallelic_nrich_input()
    hdw = CO.hdw(codes, 0.1)[0]
    _check_case(f"smallest blocks blk = {blk}", codes, POS, g, hdw, blk, 2000)
