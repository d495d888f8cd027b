"""The Hamming-distance weights on both epilogues of ``hdw_gemm_kernel``, at their tile, K-split and threshold edges.

``hdw_device`` (ldweaver_b200/csrc/hdw.cu) counts neighbours in one of two ways, and the input's shape decides which:

 * split-K (``p.fused = 0``): the partial products go to an ``S_pad x S_pad`` buffer and ``hdw_finish_kernel`` counts
   from it.  It runs when the upper triangle of the tile grid holds at most ``num_sms`` tiles and there is more than one
   K-block (S <= 2816 with more than 128 planes on 148 SMs), and whenever the distance matrix is requested;
 * fused (``p.fused = 1``): neighbours are counted straight out of TMEM, a pair ``s < t`` for both sequences (the row
   side in registers, the column side through warp ballots into shared memory), the diagonal once.  It runs from
   S = 2817 on 148 SMs (two or more tiles per CTA, three or more from S ~ 5000) and at any S with at most 128 planes.

Every case is checked against a reference that counts code equality, independently of the plane formulation:
``dist(s, t) = n - sum_a M_a^T M_a`` over the five one-hot class matrices, in float32 on the host (exact while
n < 2^24), then ``cnt = (dist < thresh).sum(0)`` and ``hdw = 1 / (cnt + 1)``.  ``test_reference_matches_the_c_oracle``
ties that reference to the C oracle.  Each case makes three calls: ``estimate_Hamming_distance_weights`` (fused where the
rule says so), the same with ``return_parts=True`` (never fused; the whole distance matrix is compared) and a one-member
``DeviceGroup`` (the path of the benchmark's C3 configuration).  Counts, weights and distances must agree bit for bit.

``test_cases_reach_their_regime`` restates the path choice of ``hdw_device`` and fails if a case stops reaching the
regime it is here for; it needs no GPU.  The class-matrix validation of ``ldw_hdw`` and ``ldw_group_load_codes`` is
tested at the end.

On one B200 the module runs in about a minute, most of it in the host reference at S ~ 6000.
"""
import numpy as np
import pytest

# ------------------------------------------------------------------------------------------------ path restatement
BM, BN, BK = 128, 256, 128   # HDW_BM, HDW_BN, HDW_BK of hdw.cu (BK in int8 planes)
HDW_STAGES = 4
B200_SMS = 148


def plane_count(codes):
    """Planes of the distance GEMM (hdw_plane_count_kernel): none for a monomorphic site, one for a biallelic site and
    r for a site with r >= 3 classes."""
    r = np.stack([(codes == a).any(axis=1) for a in range(5)]).sum(axis=0)
    return int(np.where(r <= 1, 0, np.where(r == 2, 1, r)).sum())


def hdw_regime(S, kh_real, num_sms, want_dist=False):
    """Restatement of the path choice of ``hdw_device`` (ldweaver_b200/csrc/hdw.cu, single device): the tile list of the
    upper triangle, the split count ``ks``, the loop that makes every split own a K-block, ``fused`` and the tiles each
    CTA of the persistent grid takes.  It follows hdw.cu and must be updated with it."""
    Kh = -(-max(kh_real, 1) // BK) * BK
    nkb = Kh // BK
    tiles_m, tiles_n = -(-S // BM), -(-S // BN)
    tiles = sum(1 for tn in range(tiles_n) for tm in range(tiles_m) if tm * BM <= tn * BN + BN - 1)
    ks = (2 * num_sms) // tiles if tiles > 0 else 1
    ks = min(max(ks, 1), nkb)
    while ks > 1 and (ks - 1) * (-(-nkb // ks)) >= nkb:
        ks -= 1
    grid = min(tiles * ks, num_sms)
    return dict(nkb=nkb, tiles=tiles, ks=ks, fused=(ks == 1 and not want_dist), grid=grid,
                work_per_cta=-(-tiles * ks // grid), last_tile_cols=S - (tiles_n - 1) * BN)


def fused_boundary(num_sms):
    """Smallest S whose many-plane input takes the fused path (the tile count first exceeds num_sms; monotone in S)."""
    lo, hi = 1, 1 << 16
    while lo < hi:
        mid = (lo + hi) // 2
        if hdw_regime(mid, 2 * BK, num_sms)["fused"]:
            hi = mid
        else:
            lo = mid + 1
    return lo


def pack_fallback_tiles(codes):
    """64-plane tiles of hdw_pack_kernel whose planes span 64 or more SNPs: those read the codes from global memory
    instead of the shared-memory tile."""
    r = np.stack([(codes == a).any(axis=1) for a in range(5)]).sum(axis=0)
    snp_of_plane = np.repeat(np.arange(len(codes)), np.where(r <= 1, 0, np.where(r == 2, 1, r)))
    return sum(1 for p0 in range(0, len(snp_of_plane), 64) if snp_of_plane[p0:p0 + 64][-1] - snp_of_plane[p0] >= 64)


# ------------------------------------------------------------------------------------------------ host reference
def reference_dist(codes, block=512):
    """dist(s, t) = n - sum_a M_a^T M_a over the five one-hot class matrices, float32 products in row blocks."""
    codes = np.ascontiguousarray(codes, dtype=np.uint8)
    n, S = codes.shape
    assert n < 2 ** 24 and codes.max(initial=0) <= 4      # float32 sums of 0/1 products are exact below 2^24
    X = np.empty((5 * n, S), dtype=np.float32)
    for a in range(5):
        X[a * n:(a + 1) * n] = codes == a
    dist = np.empty((S, S), dtype=np.int16 if n < 2 ** 15 else np.int32)
    for lo in range(0, S, block):
        dist[lo:lo + block] = n - X[:, lo:lo + block].T @ X
    return dist


def reference_counts(dist, thresh):
    cnt = (dist < thresh).sum(axis=0, dtype=np.int32)     # strict <, the sequence itself included (quirk Q7)
    return cnt, 1.0 / (cnt + 1.0)


def threshold_for(thresh, n):
    """A threshold fraction whose truncation n * threshold gives thresh."""
    thr = 0.0 if thresh == 0 else (thresh + 0.5) / n
    assert int(n * thr) == thresh
    return thr


def pick_thresh(dist, q=3.0):
    """A distance at the q-th percentile of the off-diagonal distances of the first rows: a dense part of the
    distribution, so that many pairs sit at thresh - 1, thresh and thresh + 1."""
    rows = dist[:256].astype(np.int64)
    off = rows[np.arange(len(rows))[:, None] != np.arange(dist.shape[1])[None, :]]
    return int(np.percentile(off, q))


# ------------------------------------------------------------------------------------------------ case inputs
def prefix_input(S, n, thresh, seed):
    """Sequence s carries the alternate allele at the sites {0 .. k_s - 1} and the base allele elsewhere, so
    dist(s, t) = |k_s - k_t| exactly.  k_s is drawn from {m * thresh + d : d in -1, 0, 1}, which puts many pairs at
    thresh - 1, thresh and thresh + 1 (and at 0: identical sequences), spread over every tile at random.  No k_s is below
    thresh - 1 or above n - thresh + 1, so the sites outside leave runs of monomorphic sites.  Alternate alleles come from
    {1, 2, 3, 4} (4 = N); the site order is shuffled."""
    rng = np.random.default_rng(seed)
    values = sorted({m * thresh + d for m in range(1, n // thresh) for d in (-1, 0, 1)} & set(range(0, n + 1)))
    k = rng.choice(values, size=S).astype(np.int64)
    alt = rng.integers(1, 5, size=n)
    base = (alt + rng.integers(1, 5, size=n)) % 5
    codes = np.where(np.arange(n)[:, None] < k[None, :], alt[:, None], base[:, None]).astype(np.uint8)
    return np.ascontiguousarray(codes[rng.permutation(n)]), k


def prefix_closed_form(k, thresh):
    d = np.abs(k[:, None] - k[None, :])
    return d, (d < thresh).sum(axis=0, dtype=np.int32)


def nrich_input(S, n, seed, n_rate=0.2):
    """Multi-allelic, N-rich founder codes; the last sequence is a copy of the first, so that the last real column has a
    neighbour in an earlier row."""
    from ldweaver_b200 import synth
    codes = synth.cheap_codes(S, n, seed, n_rate, (0.3, 0.4, 0.3))
    codes[:, S - 1] = codes[:, 0]
    return np.ascontiguousarray(codes)


def biallelic_input(S, n_planes, seed, n_mono=8):
    """n_planes biallelic sites (classes drawn from 0..4) copied from six founders with 5 % flips, every one of them
    polymorphic, and n_mono monomorphic sites among them."""
    rng = np.random.default_rng(seed)
    pairs = np.array([rng.choice(5, 2, replace=False) for _ in range(n_planes)], dtype=np.int64).reshape(n_planes, 2)
    side = rng.integers(0, 2, size=(n_planes, 6))[:, rng.integers(0, 6, size=S)]
    side ^= (rng.random((n_planes, S)) < 0.05)
    for j in range(n_planes):
        if S > 1 and side[j].min() == side[j].max():
            side[j, rng.integers(0, S)] ^= 1
    poly = np.take_along_axis(pairs, side, axis=1)
    mono = np.repeat(rng.integers(0, 5, size=(n_mono, 1)), S, axis=1)
    codes = np.concatenate([poly, mono])[rng.permutation(n_planes + n_mono)]
    return np.ascontiguousarray(codes.astype(np.uint8))


def multi_r_input(S, n_r, seed):
    """n_r = (sites with r = 3, 4, 5).  Some sites with r = 3 or 4 hold N, the highest class, which then owns the
    complement plane; the others end on a nucleotide."""
    rng = np.random.default_rng(seed)
    rows = []
    for r, m in zip((3, 4, 5), n_r):
        for j in range(m):
            classes = np.arange(5) if r == 5 else np.sort(rng.choice(5 if j % 2 else 4, r, replace=False))
            c = classes[rng.integers(0, 6, size=6)[rng.integers(0, 6, size=S)] % r]
            c[rng.choice(S, r, replace=False)] = classes                 # every class of the site present
            rows.append(c)
    return np.ascontiguousarray(np.stack(rows)[rng.permutation(len(rows))].astype(np.uint8))


def gap_input(S, seed, n_runs=4, run=(100, 150)):
    """Blocks of multi-allelic, N-rich sites separated by runs of 100-150 monomorphic sites: the 64-plane pack tiles that
    straddle a run span 64 or more SNPs."""
    rng = np.random.default_rng(seed)
    poly = nrich_input(S, 60 * (n_runs + 1), seed, n_rate=0.1)
    parts = []
    for b in range(n_runs + 1):
        parts.append(poly[60 * b:60 * (b + 1)])
        if b < n_runs:
            parts.append(np.repeat(rng.integers(0, 5, size=(int(rng.integers(*run)), 1)), S, axis=1).astype(np.uint8))
    return np.ascontiguousarray(np.concatenate(parts))


def duplicate_input(S, n, seed):
    """N-rich codes in which a tenth of the sequences are copies of others (some copied twice)."""
    rng = np.random.default_rng(seed)
    codes = nrich_input(S, n, seed)
    for i in rng.choice(S, S // 10, replace=False):
        codes[:, i] = codes[:, rng.integers(0, S)]
    return codes


def complement_input(S, n, seed):
    """Two founders that differ at every site, a fifth of the sequences copying each; the rest mix them site by site.
    Copies of different founders are at distance n."""
    rng = np.random.default_rng(seed)
    a = rng.integers(0, 5, size=n)
    b = (a + rng.integers(1, 5, size=n)) % 5
    kind = rng.integers(0, 5, size=S)
    take_a = np.where(kind[None, :] == 0, True, np.where(kind[None, :] == 1, False, rng.random((n, S)) < 0.5))
    return np.ascontiguousarray(np.where(take_a, a[:, None], b[:, None]).astype(np.uint8))


# (S, plane count) of the plane-count edges; S = 1 can only hold monomorphic sites
SMALL_S = (2, 127, 128, 129, 255, 256, 257, 385)
SMALL_PLANES = (1, 127, 128, 129)
MULTI_R = {128: (11, 10, 11), 129: (13, 10, 10)}                      # 3a + 4b + 5c planes
PREFIX_LARGE = ((2999, 2000), (6001, 2000))
PREFIX_SMALL = (300, 128)
DEEP = (6007, 3000)
GAP_S = (700, 3000)


# ------------------------------------------------------------------------------------------------ regime test (no GPU)
def _tile_positions(D, d):
    """Pairs at distance d by where the kernel meets them: (s < t in a tile that holds diagonal cells, s > t in a
    computed tile -- the mirror image the kernel must skip --, s < t in an off-diagonal tile)."""
    s, t = np.nonzero(D == d)
    tm, tn = s // BM, t // BN
    computed = tm * BM <= tn * BN + BN - 1
    diag = (tm * BM < (tn + 1) * BN) & (tn * BN < (tm + 1) * BM)
    return int(np.count_nonzero((s < t) & diag)), int(np.count_nonzero((s > t) & computed)), \
        int(np.count_nonzero((s < t) & ~diag))


def test_cases_reach_their_regime():
    R = lambda S, kh, want_dist=False: hdw_regime(S, kh, B200_SMS, want_dist)   # noqa: E731
    # the restated rule at the boundaries named in hdw.cu's comments and DESIGN.md section 4.3
    Sb = fused_boundary(B200_SMS)
    assert Sb == 2817 and R(2816, 4000)["tiles"] <= B200_SMS < R(2817, 4000)["tiles"] == 155
    assert R(Sb, 4000)["last_tile_cols"] == 1 and R(Sb - 1, 4000)["last_tile_cols"] == 256
    assert not R(Sb - 1, 4000)["fused"] and R(Sb - 1, 4000)["ks"] >= 2
    assert R(Sb, 4000)["fused"] and R(Sb, 4000)["work_per_cta"] == 2 and R(5000, 4000)["work_per_cta"] >= 3
    report = {}
    # 1. constructed ties, large S: fused without the distance matrix (>= 2 tiles per CTA, the stage ring wraps), never
    #    fused with it; pairs at thresh - 1, thresh, thresh + 1 at every tile position
    for S, n in PREFIX_LARGE + (PREFIX_SMALL,):
        thresh = int(n * 0.1)
        codes, k = prefix_input(S, n, thresh, seed=S)
        kh = plane_count(codes)
        reg = R(S, kh)
        report[f"prefix {S}"] = (kh, reg["ks"], reg["work_per_cta"])
        assert reg["fused"] and not R(S, kh, True)["fused"]
        if S == PREFIX_SMALL[0]:
            assert n <= 128 and reg["nkb"] == 1                          # fused through nkb = 1
        else:
            assert n >= 2000 and reg["work_per_cta"] >= 2 and reg["nkb"] > HDW_STAGES
        assert set(np.unique(codes)) == {0, 1, 2, 3, 4} and (codes == codes[:, :1]).all(axis=1).sum() > 0
        k16 = k.astype(np.int16)
        D = np.abs(k16[:, None] - k16[None, :])
        for d in (thresh - 1, thresh, thresh + 1):
            pos = _tile_positions(D, d)
            assert min(pos) > 0, (S, d, pos)
    assert R(6001, 2000)["work_per_cta"] >= 3
    # 2. the S boundary: multi-allelic, N-rich codes, one side split-K, the other fused with a one-column last tile
    for S in (Sb - 1, Sb):
        codes = nrich_input(S, 1000, seed=S)
        kh = plane_count(codes)
        assert kh > 2 * BK and R(S, kh)["fused"] == (S == Sb)
        assert (codes == 4).mean() > 0.15 and {3, 4, 5} <= set(np.stack([(codes == a).any(1) for a in range(5)]).sum(0))
    # 3. plane-count edges: <= 128 planes is one K-block (fused), 129 two (split-K)
    fused_planes = [p for p in SMALL_PLANES if R(385, p)["fused"]]
    assert max(fused_planes) == 128 and min(set(SMALL_PLANES) - set(fused_planes)) == 129 and min(SMALL_PLANES) == 1
    for S in SMALL_S:
        for p in SMALL_PLANES:
            codes = biallelic_input(S, p, seed=1000 * S + p)
            assert plane_count(codes) == p and R(S, p)["fused"] == (p <= 128)
            assert np.all([len(np.unique(c)) <= 2 for c in codes])
    codes = biallelic_input(1, 0, seed=1)
    assert plane_count(codes) == 0 and R(1, 0)["fused"]
    for p, n_r in MULTI_R.items():
        codes = multi_r_input(385, n_r, seed=p)
        r = np.array([len(np.unique(c)) for c in codes])
        assert plane_count(codes) == p and sorted(set(r)) == [3, 4, 5] and R(385, p)["fused"] == (p <= 128)
        top = np.array([c.max() for c in codes])
        assert np.any((r < 5) & (top == 4)) and np.any((r < 5) & (top < 4))   # N owns the complement plane at some sites
    # 4. pack-kernel fallback; the all-monomorphic matrix has no plane at all
    gap_fused = []
    for S in GAP_S:
        codes = gap_input(S, seed=S)
        kh = plane_count(codes)
        report[f"gap {S}"] = (kh, pack_fallback_tiles(codes), R(S, kh)["fused"])
        assert pack_fallback_tiles(codes) >= 2
        gap_fused.append(R(S, kh)["fused"])
    assert gap_fused == [False, True]                                     # one case on each path
    assert plane_count(np.full((50, 300), 2, dtype=np.uint8)) == 0
    # 5. thresholds: the truncation of n * threshold, pairs at distance n
    assert int(100 * 0.29) == 28 and int(100 * 0.07) == 7 and round(100 * 0.29) == 29
    codes = complement_input(300, 200, seed=5)
    assert np.count_nonzero(reference_dist(codes) == 200) > 0
    # 6. three or more tiles per CTA: both TMEM accumulators reused, their phases and the stage ring wrap
    S, n = DEEP
    codes = nrich_input(S, n, seed=S)
    kh = plane_count(codes)
    reg = R(S, kh)
    report["deep"] = (kh, reg["nkb"], reg["work_per_cta"])
    assert S % BM != 0 and reg["fused"] and reg["work_per_cta"] >= 3 and reg["nkb"] > HDW_STAGES
    print("regimes (planes, ...):", report)


def test_reference_matches_the_c_oracle():
    """The host reference against the C oracle (pinned to the reference's goldens), bit for bit, on N-rich multi-allelic
    codes and on the constructed ties."""
    import c_oracle as CO
    for codes, thresh in ((nrich_input(257, 400, seed=7), None), (prefix_input(300, 128, 12, seed=3)[0], 12)):
        n = len(codes)
        dist = reference_dist(codes)
        thresh = pick_thresh(dist) if thresh is None else thresh
        thr = threshold_for(thresh, n)
        w_o, cnt_o, dist_o = CO.hdw(codes, thr, want_dist=True)
        cnt, w = reference_counts(dist, thresh)
        np.testing.assert_array_equal(dist, dist_o)
        np.testing.assert_array_equal(cnt, cnt_o)
        np.testing.assert_array_equal(w, w_o)
        assert 1 < cnt.max() and cnt.min() < cnt.max()


# ------------------------------------------------------------------------------------------------ GPU cases
@pytest.fixture(scope="module")
def group():
    import ldweaver_b200 as ldw
    g = ldw.DeviceGroup([0])
    yield g
    g.close()


def _num_sms():
    import torch
    return torch.cuda.get_device_properties(0).multi_processor_count


def _first_diff(a, b):
    i = np.argwhere(np.asarray(a) != np.asarray(b))
    return f"{len(i)} differ, first at {tuple(i[0])}: {np.asarray(a)[tuple(i[0])]} != {np.asarray(b)[tuple(i[0])]}" if len(i) else ""


def check_case(name, codes, thresholds, group, dist=None):
    """The three calls against the host reference at every threshold: cnt, hdw and (return_parts) dist bit for bit."""
    import ldweaver_b200 as ldw
    n, S = codes.shape
    if dist is None:
        dist = reference_dist(codes)
    snp = ldw.snp_dat_from_codes(codes, np.arange(1, n + 1, dtype=np.int32), n)
    group.load_codes(codes)
    for thr in thresholds:
        thresh = int(n * thr)
        cnt_ref, w_ref = reference_counts(dist, thresh)
        what = f"{name} (S={S}, n={n}, thresh={thresh}, {plane_count(codes)} planes)"
        w1 = ldw.estimate_Hamming_distance_weights(snp, thr, devices=[0])
        w2, cnt2, dist2 = ldw.estimate_Hamming_distance_weights(snp, thr, return_parts=True, devices=[0])
        w3, cnt3, sharded = group.hdw(thr, return_parts=True)
        assert not sharded
        assert np.array_equal(dist2, dist), f"{what}: return_parts distances: {_first_diff(dist2, dist)}"
        assert np.array_equal(cnt2, cnt_ref), f"{what}: return_parts counts: {_first_diff(cnt2, cnt_ref)}"
        assert np.array_equal(cnt3, cnt_ref), f"{what}: device-group counts: {_first_diff(cnt3, cnt_ref)}"
        for label, w in (("weights", w1), ("return_parts weights", w2), ("device-group weights", w3)):
            assert np.array_equal(w, w_ref), f"{what}: {label}: {_first_diff(w, w_ref)}"
    return dist


@pytest.mark.gpu
@pytest.mark.parametrize("S,n", PREFIX_LARGE + (PREFIX_SMALL,))
def test_ties_at_the_threshold(S, n, group):
    """Constructed distances |k_s - k_t|: pairs at thresh - 1, thresh and thresh + 1 at every tile position, checked
    against the closed form too.  Large S: fused, and split-K with return_parts; S = 300 with <= 128 sites: fused
    through a single K-block."""
    thresh = int(n * 0.1)
    codes, k = prefix_input(S, n, thresh, seed=S)
    dist = reference_dist(codes)
    d_cf, cnt_cf = prefix_closed_form(k, thresh)
    assert np.array_equal(dist, d_cf)
    del d_cf
    assert np.array_equal(reference_counts(dist, thresh)[0], cnt_cf)
    check_case("ties", codes, (0.1, threshold_for(thresh - 1, n), threshold_for(thresh + 1, n)), group, dist)


@pytest.mark.gpu
@pytest.mark.parametrize("side", ["split-K", "fused"])
def test_fused_boundary(side, group):
    """The smallest S that takes the fused path on this device (2817 on 148 SMs: a last column tile with one real
    column), and one sequence fewer (split-K); multi-allelic, N-rich codes."""
    num_sms = _num_sms()
    S = fused_boundary(num_sms) - (side == "split-K")
    codes = nrich_input(S, 1000, seed=S)
    reg = hdw_regime(S, plane_count(codes), num_sms)
    assert reg["fused"] == (side == "fused")
    dist = reference_dist(codes)
    thresh = pick_thresh(dist)
    assert min(np.count_nonzero(dist == d) for d in (thresh - 1, thresh, thresh + 1)) > 100
    assert reference_counts(dist, thresh)[0][S - 1] > 1
    check_case(f"boundary {side}", codes, (threshold_for(thresh, len(codes)), 0.0), group, dist)


@pytest.mark.gpu
@pytest.mark.parametrize("S", SMALL_S)
def test_plane_count_edges(S, group):
    """1, 127, 128 (one K-block: fused) and 129 planes (two K-blocks: split-K), at a distance that occurs and one
    above it."""
    for p in SMALL_PLANES:
        codes = biallelic_input(S, p, seed=1000 * S + p)
        dist = reference_dist(codes)
        off = dist[~np.eye(S, dtype=bool)]
        t0 = max(1, int(np.median(off)))
        check_case(f"{p} planes", codes, (threshold_for(t0, len(codes)), threshold_for(t0 + 1, len(codes))), group, dist)


@pytest.mark.gpu
def test_one_sequence(group):
    codes = biallelic_input(1, 0, seed=1)
    check_case("one sequence", codes, (0.0, threshold_for(1, len(codes))), group)


@pytest.mark.gpu
@pytest.mark.parametrize("planes", sorted(MULTI_R))
def test_sites_with_three_to_five_classes(planes, group):
    codes = multi_r_input(385, MULTI_R[planes], seed=planes)
    dist = reference_dist(codes)
    t0 = int(np.median(dist[~np.eye(385, dtype=bool)]))
    check_case("r = 3, 4, 5", codes, (threshold_for(t0, len(codes)), threshold_for(t0 + 1, len(codes))), group, dist)


@pytest.mark.gpu
@pytest.mark.parametrize("S", GAP_S)
def test_pack_tiles_across_monomorphic_runs(S, group):
    codes = gap_input(S, seed=S)
    dist = reference_dist(codes)
    check_case("monomorphic runs", codes, (threshold_for(pick_thresh(dist), len(codes)),), group, dist)


@pytest.mark.gpu
@pytest.mark.parametrize("S", [300, 3000])
def test_all_sites_monomorphic(S, group):
    """No plane at all (kh_real = 0): every distance 0, every sequence a neighbour of every other."""
    codes = np.repeat(np.random.default_rng(S).integers(0, 5, size=(50, 1)), S, axis=1).astype(np.uint8)
    dist = check_case("monomorphic", codes, (0.1, 0.0), group)
    assert not dist.any() and np.all(reference_counts(dist, 5)[0] == S)


@pytest.mark.gpu
@pytest.mark.parametrize("S", [700, "boundary"])
def test_threshold_zero_and_one_difference(S, group):
    """threshold = 0: every weight 1 (quirk Q7), also on the fused path; thresh = 1: only identical sequences count,
    with duplicated sequences present."""
    S = fused_boundary(_num_sms()) if S == "boundary" else S
    codes = duplicate_input(S, 1000, seed=S)
    dist = reference_dist(codes)
    cnt1 = reference_counts(dist, 1)[0]
    assert cnt1.max() >= 3 and np.count_nonzero(cnt1 >= 2) >= S // 10
    check_case("threshold 0 / thresh 1", codes, (0.0, threshold_for(1, len(codes))), group, dist)


@pytest.mark.gpu
@pytest.mark.parametrize("S", [300, "boundary"])
def test_threshold_one_excludes_pairs_differing_everywhere(S, group):
    S = fused_boundary(_num_sms()) if S == "boundary" else S
    codes = complement_input(S, 200, seed=S)
    dist = reference_dist(codes)
    assert np.count_nonzero(dist == 200) > 0 and reference_counts(dist, 200)[0].min() < S
    check_case("threshold 1.0", codes, (1.0,), group, dist)


@pytest.mark.gpu
def test_truncation_of_n_times_threshold(group):
    """n = 100: 100 * 0.29 = 28.999999999999996 truncates to 28, 100 * 0.07 = 7.000000000000001 to 7 (R's
    as.integer); constructed distances put pairs at 27..29 and 6..8."""
    codes, k = prefix_input(300, 100, 7, seed=29)
    assert int(100 * 0.29) == 28 and int(100 * 0.07) == 7
    dist = reference_dist(codes)
    assert all(np.count_nonzero(dist == d) > 0 for d in (6, 7, 8, 27, 28, 29))
    check_case("truncation", codes, (0.29, 0.07), group, dist)


@pytest.mark.gpu
def test_fused_three_or_more_tiles_per_cta(group):
    """S = 6007 (not a multiple of 128), 3000 N-rich multi-allelic sites: every CTA takes three or more tiles, so both
    TMEM accumulators are reused with wrapped phases and the stage ring wraps within and across tiles."""
    S, n = DEEP
    codes = nrich_input(S, n, seed=S)
    dist = reference_dist(codes)
    thresh = pick_thresh(dist)
    assert reference_counts(dist, thresh)[0][S - 1] > 1
    check_case("three tiles per CTA", codes, (threshold_for(thresh, n),), group, dist)


# ------------------------------------------------------------------------------------------------ class validation
BAD_SHAPE = (37, 131)       # 4847 bytes: 302 16-byte words in the vectorised body, a scalar tail of 15 bytes
# (word of the 16-byte load, byte lane) pairs covering every lane and every word, plus the first and last tail bytes
BAD_BODY = [16 * 150 + 4 * w + b for w, b in ((0, 0), (1, 1), (2, 2), (3, 3), (0, 3), (1, 2), (2, 1), (3, 0))]
BAD_TAIL = [302 * 16, BAD_SHAPE[0] * BAD_SHAPE[1] - 1]


def _valid_codes():
    return np.random.default_rng(37).integers(0, 5, size=BAD_SHAPE).astype(np.uint8)


@pytest.mark.gpu
@pytest.mark.parametrize("where", BAD_BODY + BAD_TAIL)
def test_hdw_refuses_a_class_above_4(where):
    import ldweaver_b200 as ldw
    from ldweaver_b200 import _lib
    good = _valid_codes()
    n = good.shape[0]
    bad = good.copy()
    bad.reshape(-1)[where] = 5
    with pytest.raises(_lib.LdwError, match="class 5 outside 0..4") as e:
        ldw.estimate_Hamming_distance_weights(ldw.snp_dat_from_codes(bad, np.arange(1, n + 1), n), 0.1, devices=[0])
    assert e.value.code == 1   # LDW_ERR_ARG
    # the same context still computes the right weights
    dist = reference_dist(good)
    thr = threshold_for(pick_thresh(dist, 50), n)
    w = ldw.estimate_Hamming_distance_weights(ldw.snp_dat_from_codes(good, np.arange(1, n + 1), n), thr, devices=[0])
    np.testing.assert_array_equal(w, reference_counts(dist, int(n * thr))[1])


@pytest.mark.gpu
@pytest.mark.parametrize("where", BAD_BODY + BAD_TAIL)
def test_group_load_codes_refuses_a_class_above_4(where, group):
    from ldweaver_b200 import _lib
    good = _valid_codes()
    bad = good.copy()
    bad.reshape(-1)[where] = 5
    with pytest.raises(_lib.LdwError, match="class 5 outside 0..4") as e:
        group.load_codes(bad)
    assert e.value.code == 1
    dist = reference_dist(good)
    check_case("after a refused matrix", good, (threshold_for(pick_thresh(dist, 50), len(good)),), group, dist)
