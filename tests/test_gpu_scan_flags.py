"""ldw_mi_scan under every LDW_SCAN_* flag and entry path.

The value flags (0, IDEAL_Q, SR_EXACT, SR_ONLY and their combinations) choose what is computed; the output flags (NO_D2H,
NO_LINKS, LR_ONLY, SR_ON_DEVICE) choose what comes back.  Every combination runs through MIPlan.scan, the n_parts / part
split, a one-member DeviceGroup and an in-process group over every device, and is checked against an fp64 reference of
the same operation (the compiled C oracle for the reference's quirk Q1, a restatement of the closed form with the ideal
Q = 0.25 r_i r_j for IDEAL_Q, the literal restatement for SR_ONLY) and against the same value flags without output
flags, bit for bit.  What each output flag returns is the table in include/ldw.h.

Two inputs: A, shaped like the benchmark workload (10 blocks of blk 1000, one ragged 700-row range, short-range links in
the diagonal blocks, next to them and across the circular wrap); B, multi-allelic and N-rich (every r from 2 to 5, a
square off-diagonal block and ragged ones), where the ideal Q and quirk Q1 differ.  The GPU tests are marked one by one:
the header and oracle checks at the end run without a device."""
import ctypes as C
import functools
import os
import re

import numpy as np
import pytest

from util import compare_lr_sets

from ldweaver_b200 import api

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
MI_TOL = 1e-6       # fp32 epilogue against the fp64 reference
EXACT_TOL = 1e-12   # fp64 refinement (SR_EXACT short-range MI, thresholds, long-range MI)

SR_ONLY, IDEAL_Q, NO_LINKS, NO_D2H = api.SCAN_SR_ONLY, api.SCAN_IDEAL_Q, api.SCAN_NO_LINKS, api.SCAN_NO_D2H
SR_EXACT, LR_ONLY, SR_ON_DEVICE = api.SCAN_SR_EXACT, api.SCAN_LR_ONLY, api.SCAN_SR_ON_DEVICE
VALUE_FLAGS = (0, IDEAL_Q, SR_EXACT, IDEAL_Q | SR_EXACT, SR_ONLY, SR_ONLY | SR_EXACT)
OUTPUT_FLAGS = (0, NO_D2H, NO_LINKS, LR_ONLY, LR_ONLY | NO_D2H, SR_ON_DEVICE)
COLS = ("pos1", "pos2", "clust1", "clust2", "len", "MI", "block")
COUNTS = ("n_pairs", "n_sr", "n_lr_total", "n_lr_kept")   # n_candidates / n_reruns follow the unordered chain seed


def flag_name(flags: int) -> str:
    names = [n for n in ("SR_ONLY", "IDEAL_Q", "NO_LINKS", "NO_D2H", "SR_EXACT", "LR_ONLY", "SR_ON_DEVICE")
             if flags & getattr(api, "SCAN_" + n)]
    return "+".join(names) or "0"


def refused(flags: int) -> bool:
    """SR_ONLY asks for no long-range table, LR_ONLY for no short-range one: together they ask for nothing."""
    return bool(flags & SR_ONLY) and bool(flags & LR_ONLY)


def n_devices():
    import torch
    return torch.cuda.device_count()


# ---------------------------------------------------------------------------------------------------------- the inputs
def ideal_q_block_mi(osnp, hdw, from_idx, to_idx):
    """MI of one block with the ideal Q = 0.25 r_i r_j on every block (LDW_SCAN_IDEAL_Q): ldw_oracle.block_mi_closed_form
    without quirk Q1, which reads the off-diagonal blocks' Q at the transposed linear index.  fp64."""
    w = np.asarray(hdw, dtype=np.float64)
    rf, rt = osnp.r[from_idx].astype(np.float64), osnp.r[to_idx].astype(np.float64)
    den = w.sum() + 0.5 * np.outer(rf, rt)
    Q = 0.25 * np.outer(rf, rt)
    Xf = [(osnp.codes[from_idx] == a).astype(np.float64) for a in range(5)]
    Xt = [(osnp.codes[to_idx] == a).astype(np.float64) for a in range(5)]
    pf, pt = [x @ w for x in Xf], [x @ w for x in Xt]
    MI = np.zeros((len(from_idx), len(to_idx)))
    for a in range(5):
        for b in range(5):
            u = np.outer(osnp.uqe[from_idx, a], osnp.uqe[to_idx, b])
            if not u.any():
                continue
            cab = (Xf[a] * w[None, :]) @ Xt[b].T + 0.5
            D = np.outer(pf[a], pt[b]) + 0.5 * (pf[a] * rf)[:, None] + 0.5 * (pt[b] * rt)[None, :] + Q
            MI += u * cab / den * np.log(cab * den / D)
    return MI


class Ref:
    """What a scan must return, in reference order: short-range rows, per-block long-range sets, thresholds, probabilities."""

    def __init__(self, sr, lr_sets, thr, prob):
        self.sr, self.lr_sets, self.thr, self.prob = sr, lr_sets, thr, prob


class Case:
    blk = 1000
    sr_dist = 20000.0

    def __init__(self, name, codes, POS, g, retain):
        import c_oracle as CO
        import ldw_oracle as O
        from ldweaver_b200 import synth
        self.name, self.codes, self.POS, self.g, self.retain = name, np.ascontiguousarray(codes), np.asarray(POS, np.int32), int(g), retain
        n = len(self.POS)
        self.paint = np.ones(n, dtype=np.int32)        # three contiguous clusters, as synth.generate paints them
        self.paint[n // 3:] = 2
        self.paint[2 * n // 3:] = 3
        self.nclust = 3
        self.hdw = CO.hdw(self.codes, 0.1)[0]
        self.osnp = O.snp_dat_from_codes(self.codes, self.POS, self.g)
        self.lra = synth.exact_lr_links_approx(self.POS, self.g, self.sr_dist)
        self.blocks = O.make_blocks(n, self.blk)
        self.diag = np.array([fs == ts for fs, _, ts, _ in self.blocks])

    def block_idx(self, bi):
        fs, fe, ts, te = self.blocks[bi]
        return np.arange(fs - 1, fe), np.arange(ts - 1, te)

    def _links_ref(self, block_mi) -> Ref:
        import c_oracle as CO
        POS = self.POS.astype(np.float64)
        sr = {k: [] for k in COLS}
        lr_sets, thr, prob = {}, np.full(len(self.blocks), np.nan), np.full(len(self.blocks), np.nan)
        for bi in range(len(self.blocks)):
            f, t = self.block_idx(bi)
            L = CO.block_links(block_mi(f, t), POS, f, t, float(self.g), self.sr_dist, self.retain, self.lra)
            gi, gj = f[L["row"]], t[L["col"]]
            s = L["is_sr"]
            for k, v in (("pos1", self.POS[gj]), ("pos2", self.POS[gi]), ("clust1", self.paint[gj]), ("clust2", self.paint[gi]),
                         ("len", L["len"].astype(np.int32)), ("MI", L["MI"]), ("block", np.full(len(s), bi, np.int32))):
                sr[k].append(v[s])
            thr[bi], prob[bi] = L["thr"], L["prob"]
            k = L["lr_keep"]
            lr_sets[bi] = (self.POS[gj][k], self.POS[gi][k], L["MI"][k])
        return Ref({k: np.concatenate(v) for k, v in sr.items()}, lr_sets, thr, prob)

    @functools.cached_property
    def ref_q1(self) -> Ref:
        """The reference's arithmetic, quirk Q1 included: the compiled C oracle, block by block."""
        import c_oracle as CO
        return self._links_ref(lambda f, t: CO.block_mi(self.codes, self.hdw, self.osnp.r, self.osnp.uqe, f, t))

    @functools.cached_property
    def ref_ideal(self) -> Ref:
        return self._links_ref(lambda f, t: ideal_q_block_mi(self.osnp, self.hdw, f, t))

    @functools.cached_property
    def ref_sr_only(self) -> Ref:
        """perform_SR_analysis_only = TRUE (quirk Q12: far SNPs dropped before the MI, so Q1 acts on the reduced lists)."""
        import ldw_oracle as O
        res = O.perform_MI_scan(self.osnp, self.hdw, self.paint, self.nclust, sr_dist=self.sr_dist, lr_retain_links=self.retain,
                                max_blk_sz=self.blk, perform_SR_analysis_only=True, keep_blocks=True)
        sr = {k: np.asarray(res.sr[k]) for k in COLS if k != "block"}
        sr["block"] = np.concatenate([np.full(int(b.sr_mask.sum()), b.block, np.int32) for b in res.blocks])
        nb = len(self.blocks)
        return Ref(sr, {}, np.full(nb, np.nan), np.full(nb, np.nan))

    def ref(self, vflags) -> Ref:
        if vflags & SR_ONLY:
            return self.ref_sr_only
        return self.ref_ideal if vflags & IDEAL_Q else self.ref_q1


@functools.lru_cache(maxsize=None)
def case(name) -> Case:
    if name == "A":
        from ldweaver_b200 import synth
        sy = synth.generate(nseq=300, nsnp=3700, seed=31)
        return Case("A", sy.codes, sy.POS, sy.g, 5e4)
    # B: multi-allelic and N-rich (as test_gpu_mi.py::test_multiallelic_nrich_vs_oracle), 3 row blocks of 1000, 1000 and
    # the rest
    rng = np.random.default_rng(42)
    S, n, g = 300, 2600, 1_000_000
    nall = rng.choice([2, 3, 4], size=n, p=[0.5, 0.3, 0.2])
    founders = np.stack([rng.integers(0, k, size=10) for k in nall]).astype(np.uint8)
    codes = founders[:, rng.integers(0, 10, size=S)]
    flip = rng.random((n, S)) < 0.05
    codes[flip] = (codes[flip] + 1) % np.repeat(nall, S).reshape(n, S)[flip]
    nrich = rng.random((n, S)) < 0.08       # N / gap class, on all sites but a fifth (so that bi-allelic sites give r = 2)
    nrich[rng.random(n) < 0.2] = False
    codes[nrich] = 4
    POS = np.sort(rng.choice(np.arange(1, g), n, replace=False)).astype(np.int32)
    r = np.stack([(codes == a).any(axis=1) for a in range(5)], axis=1).sum(axis=1)
    keep = r >= 2
    return Case("B", codes[keep], POS[keep], g, 3e4)


# ------------------------------------------------------------------------------------------------- running the scans
def take(sr, lr, bd, thr, prob, st) -> dict:
    """A scan's outputs as arrays this test owns (the library's tables live until the next scan on the same context).
    A table whose columns came back NULL is None; its row count is kept either way."""
    if isinstance(st, list):   # device group: one entry per local member
        st = {k: sum(d[k] for d in st) for k in COUNTS}
    out = {"thr": thr.copy(), "prob": prob.copy(), "stats": {k: int(st[k]) for k in COUNTS}}
    for name, t in (("sr", sr), ("lr", lr), ("bd", bd)):
        n = int(t.n)
        present = {bool(getattr(t, k)) for k in COLS}
        assert n == 0 or len(present) == 1, f"{name}: some columns NULL, others not"
        out[name + "_n"] = n
        out[name] = t.to_dict() if (n == 0 or present == {True}) else None
    return out


class FlagSet:
    """One case and one set of value flags: a plan, and the whole-job scans under each output flag (memoised)."""

    def __init__(self, c: Case, vflags: int):
        import ldweaver_b200 as ldw
        self.case, self.v = c, vflags
        self.plan = ldw.MIPlan(ldw.snp_dat_from_codes(c.codes, c.POS, c.g), c.hdw, c.paint, c.blk)
        self._memo = {}

    def fresh(self, flags, n_parts=1, part=0) -> dict:
        c = self.case
        return take(*self.plan.scan(float(c.g), c.sr_dist, c.retain, c.lra, flags, n_parts, part, copy=False))

    def scan(self, flags) -> dict:
        if flags not in self._memo:
            self._memo[flags] = self.fresh(flags)
        return self._memo[flags]

    def group(self, grp, flags) -> dict:
        c = self.case
        return take(*grp.mi_scan(c.hdw, c.POS, c.paint, c.blk, float(c.g), c.sr_dist, c.retain, c.lra, flags, copy=False))


@pytest.fixture(scope="module", params=[(c, v) for c in ("A", "B") for v in VALUE_FLAGS], ids=lambda p: f"{p[0]}-{flag_name(p[1])}")
def flagset(request):
    fs = FlagSet(case(request.param[0]), request.param[1])
    yield fs
    fs.plan.close()


@pytest.fixture(scope="module")
def groups():
    """In-process device groups by device list, the case's matrix loaded (NCCL set-up is paid once per group)."""
    made = {}

    def get(devices, c: Case):
        key = tuple(devices)
        if key not in made:
            made[key] = [api.DeviceGroup(list(key)), None]
        if made[key][1] != c.name:
            made[key][0].load_codes(c.codes)
            made[key][1] = c.name
        return made[key][0]
    yield get
    for g, _ in made.values():
        g.close()


# --------------------------------------------------------------------------------------------------------- the checks
def same_table(a, b, what):
    for k in COLS:
        np.testing.assert_array_equal(a[k], b[k], err_msg=f"{what}: {k}")


def assert_same(a, b, what):
    """Two scans' outputs bit for bit: row counts, which tables came back, their rows, thr / prob, the counts of the stats."""
    for name in ("sr", "lr", "bd"):
        assert a[name + "_n"] == b[name + "_n"], f"{what}: {name} rows {a[name + '_n']} vs {b[name + '_n']}"
        assert (a[name] is None) == (b[name] is None), f"{what}: {name} columns NULL in one of them only"
        if a[name] is not None:
            same_table(a[name], b[name], f"{what}: {name}")
    np.testing.assert_array_equal(a["thr"], b["thr"], err_msg=f"{what}: thr")
    np.testing.assert_array_equal(a["prob"], b["prob"], err_msg=f"{what}: prob")
    assert a["stats"] == b["stats"], what


def assert_refused(call, what):
    with pytest.raises(api._lib.LdwError) as ei:
        call()
    msg = str(ei.value)
    assert ei.value.code == 1 and "LDW_SCAN_SR_ONLY" in msg and "LDW_SCAN_LR_ONLY" in msg, f"{what}: {msg}"


def check_contract(got, base, o, what):
    """What output flags `o` return (include/ldw.h), against the scan of the same value flags without output flags."""
    no_host = bool(o & (NO_D2H | NO_LINKS))
    sr_n = 0 if o & LR_ONLY else base["sr_n"]
    assert got["sr_n"] == sr_n, f"{what}: short-range rows {got['sr_n']}, expected {sr_n}"
    if sr_n:
        sr_cols = not (no_host or o & SR_ON_DEVICE)
        assert (got["sr"] is not None) == sr_cols, f"{what}: short-range columns {'missing' if sr_cols else 'not NULL'}"
        if sr_cols:
            same_table(got["sr"], base["sr"], f"{what}: sr")
    assert got["lr_n"] == base["lr_n"], f"{what}: long-range rows"
    if base["lr_n"]:
        assert (got["lr"] is not None) == (not no_host), f"{what}: long-range columns"
        if not no_host:
            same_table(got["lr"], base["lr"], f"{what}: lr")
    assert got["bd_n"] == (0 if no_host else base["bd_n"]), f"{what}: borderline rows"
    if got["bd_n"]:
        same_table(got["bd"], base["bd"], f"{what}: borderline")
    np.testing.assert_array_equal(got["thr"], base["thr"], err_msg=f"{what}: thr")
    np.testing.assert_array_equal(got["prob"], base["prob"], err_msg=f"{what}: prob")
    assert got["stats"] == base["stats"], what


def check_against_reference(got, c: Case, v, o, what):
    ref = c.ref(v)
    assert np.array_equal(np.isnan(got["thr"]), np.isnan(ref.thr)), f"{what}: blocks with a long-range branch"
    ok = ~np.isnan(ref.thr)
    if ok.any():
        assert np.abs(got["thr"][ok] - ref.thr[ok]).max() <= EXACT_TOL, f"{what}: thr"
    np.testing.assert_array_equal(got["prob"], ref.prob, err_msg=f"{what}: prob")
    assert got["sr_n"] == (0 if o & LR_ONLY else len(ref.sr["MI"])), f"{what}: short-range rows"
    if got["sr"] is not None and got["sr_n"]:
        for k in ("pos1", "pos2", "len", "block", "clust1", "clust2"):
            np.testing.assert_array_equal(got["sr"][k], ref.sr[k], err_msg=f"{what}: sr {k}")
        err = float(np.abs(got["sr"]["MI"] - ref.sr["MI"]).max())
        assert err <= (EXACT_TOL if v & SR_EXACT else MI_TOL), f"{what}: short-range MI off by {err}"
    if v & SR_ONLY:
        assert got["lr_n"] == 0 and got["stats"]["n_lr_total"] == 0, what
    lr = got["lr"]
    if lr is None:
        return
    assert np.all(np.diff(lr["block"]) >= 0), f"{what}: long-range rows out of block order"
    at = np.searchsorted(c.POS, lr["pos1"]), np.searchsorted(c.POS, lr["pos2"])
    np.testing.assert_array_equal(c.POS[at[0]], lr["pos1"])
    np.testing.assert_array_equal(lr["clust1"], c.paint[at[0]], err_msg=f"{what}: lr clust1")
    np.testing.assert_array_equal(lr["clust2"], c.paint[at[1]], err_msg=f"{what}: lr clust2")
    d = np.mod(lr["pos1"].astype(np.float64) - lr["pos2"], c.g)
    np.testing.assert_array_equal(lr["len"], (0.5 * c.g - np.abs(d - 0.5 * c.g)).astype(np.int64), err_msg=f"{what}: lr len")
    for bi in range(len(c.blocks)):
        k = lr["block"] == bi
        if np.isnan(ref.thr[bi]):
            assert not k.any(), f"{what}: long-range rows in block {bi}, which has no long-range branch"
        else:
            compare_lr_sets(*ref.lr_sets[bi], lr["pos1"][k], lr["pos2"][k], lr["MI"][k], ref.thr[bi])
    if got["bd"] is not None:
        near = np.abs(lr["MI"] - got["thr"][lr["block"]]) <= 1e-9
        same_table(got["bd"], {k: lr[k][near] for k in COLS}, f"{what}: borderline rows")


@pytest.mark.gpu
def test_every_output_flag_against_the_fp64_reference(flagset):
    """Whatever comes back -- short-range rows (exact, in reference order; MI to 1e-6, 1e-12 with SR_EXACT),
    thresholds (1e-12, NaN where no long-range branch), probabilities (exact), long-range sets, borderline rows -- against
    the fp64 reference of the value flags."""
    c, v = flagset.case, flagset.v
    for o in OUTPUT_FLAGS:
        what = f"case {c.name}, {flag_name(v | o)}"
        if refused(v | o):
            assert_refused(lambda: flagset.fresh(v | o), what)
            continue
        check_against_reference(flagset.scan(v | o), c, v, o, what)


@pytest.mark.gpu
def test_output_flags_change_what_comes_back_not_the_values(flagset):
    """Every output flag against the same value flags without it, bit for bit, under the header's table."""
    v = flagset.v
    base = flagset.scan(v)
    assert base["sr_n"] == base["stats"]["n_sr"] and base["lr_n"] == base["stats"]["n_lr_kept"]
    assert base["sr"] is not None and base["lr"] is not None and base["bd"] is not None
    assert base["sr_n"] > 0 and (v & SR_ONLY or base["lr_n"] > 0)
    for o in OUTPUT_FLAGS[1:]:
        if not refused(v | o):
            check_contract(flagset.scan(v | o), base, o, f"case {flagset.case.name}, {flag_name(v | o)}")


@pytest.mark.gpu
def test_partition_union_equals_the_whole_job(flagset):
    """Split n_parts = 3 ways: the parts' rows, ordered by block, are the whole job's bit for bit, and their counts sum to it."""
    c, v = flagset.case, flagset.v
    for o in OUTPUT_FLAGS:
        what = f"case {c.name}, {flag_name(v | o)}, 3 parts"
        if refused(v | o):
            assert_refused(lambda: flagset.fresh(v | o, 3, 1), what)
            continue
        whole = flagset.scan(v | o)
        parts = [flagset.fresh(v | o, 3, p) for p in range(3)]
        for name in ("sr", "lr", "bd"):
            assert sum(p[name + "_n"] for p in parts) == whole[name + "_n"], f"{what}: {name} rows"
            if whole[name] is not None:
                tabs = [p[name] for p in parts]
                assert all(t is not None for t in tabs), f"{what}: {name} columns"
                order = np.argsort(np.concatenate([t["block"] for t in tabs]), kind="stable")
                same_table({k: np.concatenate([t[k] for t in tabs])[order] for k in COLS}, whole[name], f"{what}: {name}")
        for key in ("thr", "prob"):
            merged = np.full_like(whole[key], np.nan)
            for p in parts:
                m = ~np.isnan(p[key])
                assert np.all(np.isnan(merged[m])), f"{what}: {key} of one block from two parts"
                merged[m] = p[key][m]
            np.testing.assert_array_equal(merged, whole[key], err_msg=f"{what}: {key}")
        for k in COUNTS:
            assert sum(p["stats"][k] for p in parts) == whole["stats"][k], f"{what}: {k}"


@pytest.mark.gpu
def test_one_member_group_equals_the_plan(flagset, groups):
    """DeviceGroup([0]) returns what MIPlan.scan returns, for every flag set, counts and NULL columns included."""
    c, v = flagset.case, flagset.v
    grp = groups([0], c)
    for o in OUTPUT_FLAGS:
        what = f"case {c.name}, {flag_name(v | o)}, one-member group"
        if refused(v | o):
            assert_refused(lambda: flagset.group(grp, v | o), what)
            continue
        assert_same(flagset.group(grp, v | o), flagset.scan(v | o), what)


@pytest.mark.gpu
def test_repeated_scan_is_bit_identical(flagset):
    """A second identical call returns the same thing bit for bit (what bench.py --dump-outputs relies on)."""
    c, v = flagset.case, flagset.v
    for o in OUTPUT_FLAGS:
        if not refused(v | o):
            assert_same(flagset.fresh(v | o), flagset.scan(v | o), f"case {c.name}, {flag_name(v | o)}, repeated")


def _device_post(c: Case):
    """mergeNsort_sr_links_device on what the last scan left on device 0: its arrays, or the error message."""
    try:
        r = api.mergeNsort_sr_links_device(api.CdsVar(c.paint, c.nclust), c.sr_dist, None, 3.0)
    except api._lib.LdwError as e:
        return str(e)
    out = {"red": r.red, "chk": r.chk, **{"df_" + k: v for k, v in r.df.items()}}
    for i, f in enumerate(r.fits):
        out.update({f"fit{i}_{k}": np.asarray(f[k]) for k in ("len", "max", "fit", "coef", "shape", "start", "n_pos")})
    return out


@pytest.mark.gpu
def test_device_post_processing_after_each_scan_kind(flagset):
    """mergeNsort_sr_links_device after a NO_D2H scan equals its result after an SR_ON_DEVICE scan; after an
    LR_ONLY, a NO_LINKS or an n_parts > 1 scan no device holds the job's table and it is refused with LDW_ERR_ARG."""
    c, v = flagset.case, flagset.v
    flagset.fresh(v | NO_D2H)
    a = _device_post(c)
    flagset.fresh(v | SR_ON_DEVICE)
    b = _device_post(c)
    assert type(a) is type(b), (a if isinstance(a, str) else b)
    if isinstance(a, str):
        assert a == b
    else:
        assert a.keys() == b.keys()
        for k in a:
            np.testing.assert_array_equal(a[k], b[k], err_msg=k)
    if v & SR_EXACT:
        # fp64 short-range MI: the fits succeed or fail as the host implementation's on the reference's table (with quirk
        # Q1 on these inputs, cluster 1 keeps fewer than two links above its decay fit; with the ideal Q they succeed)
        try:
            host = api.mergeNsort_sr_links(api.CdsVar(c.paint, c.nclust), c.ref(v).sr, c.sr_dist, None, 3.0)
        except api._lib.LdwError as e:
            assert a == str(e)
        else:
            assert not isinstance(a, str), a
            assert len(a["red"]) > 0 and [len(f["len"]) for f in host.fits] == [len(a[f"fit{i}_len"]) for i in range(c.nclust)]
    for flags, n_parts in ((v | NO_LINKS, 1), (v, 3)) + (() if v & SR_ONLY else ((v | LR_ONLY, 1),)):
        flagset.fresh(flags, n_parts, 0)
        with pytest.raises(api._lib.LdwError) as ei:
            api.mergeNsort_sr_links_device(api.CdsVar(c.paint, c.nclust), c.sr_dist, None, 3.0)
        assert ei.value.code == 1 and "no short-range table" in str(ei.value), (flag_name(flags), n_parts, str(ei.value))


@pytest.mark.gpu
@pytest.mark.skipif("n_devices() < 2")
def test_in_process_group_over_all_devices(flagset, groups):
    """A group over every device returns what one device returns, for every flag set -- with SR_ON_DEVICE the
    job's short-range count and NULL columns, with LR_ONLY | NO_D2H no short-range rows."""
    c, v = flagset.case, flagset.v
    grp = groups(range(n_devices()), c)
    base = flagset.group(grp, v)
    for o in OUTPUT_FLAGS:
        what = f"case {c.name}, {flag_name(v | o)}, group over {n_devices()} devices"
        if refused(v | o):
            assert_refused(lambda: flagset.group(grp, v | o), what)
            continue
        got = base if o == 0 else flagset.group(grp, v | o)
        assert_same(got, flagset.scan(v | o), what)
        check_contract(got, base, o, what)


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["A", "B"])
@pytest.mark.parametrize("exact", [False, True], ids=["fp32", "SR_EXACT"])
def test_ideal_q_equals_flag_0_on_diagonal_blocks(name, exact):
    """On a diagonal block quirk Q1 and the ideal Q are the same exact product, so IDEAL_Q must give flag 0's rows,
    MI, thresholds and long-range rows there bit for bit -- and differ on the off-diagonal blocks, as the references do."""
    c = case(name)
    extra = SR_EXACT if exact else 0
    fs = FlagSet(c, IDEAL_Q | extra)
    try:
        ideal, q1 = fs.scan(IDEAL_Q | extra), fs.scan(extra)
    finally:
        fs.plan.close()
    for tab in ("sr", "lr"):
        a, b = ideal[tab], q1[tab]
        ma, mb = c.diag[a["block"]], c.diag[b["block"]]
        same_table({k: a[k][ma] for k in COLS}, {k: b[k][mb] for k in COLS}, f"case {name}: {tab} rows of diagonal blocks")
    np.testing.assert_array_equal(ideal["thr"][c.diag], q1["thr"][c.diag])
    np.testing.assert_array_equal(ideal["prob"][c.diag], q1["prob"][c.diag])
    np.testing.assert_array_equal(ideal["sr"]["pos1"], q1["sr"]["pos1"])
    off, off_ref = ~c.diag[q1["sr"]["block"]], ~c.diag[c.ref_q1.sr["block"]]
    assert off.any() and off_ref.any()
    ref_gap = float(np.abs(c.ref_ideal.sr["MI"] - c.ref_q1.sr["MI"])[off_ref].max())
    got_gap = float(np.abs(ideal["sr"]["MI"] - q1["sr"]["MI"])[off].max())
    print(f"case {name}: |ideal Q - Q1| over off-diagonal short-range MI: reference {ref_gap:.3g}, scan {got_gap:.3g}")
    assert ref_gap > 1e-6 and got_gap > 1e-6


@pytest.mark.gpu
def test_sr_only_with_lr_only_is_refused_by_the_public_api():
    import ldweaver_b200 as ldw
    c = case("A")
    snp = ldw.snp_dat_from_codes(c.codes, c.POS, c.g)
    assert_refused(lambda: ldw.perform_MI_computation(snp, c.hdw, ldw.CdsVar(c.paint, c.nclust), sr_dist=c.sr_dist, max_blk_sz=c.blk,
                                                      perform_SR_analysis_only=True, scan_flags=api.SCAN_LR_ONLY, write_tsv=False),
                   "perform_MI_computation(perform_SR_analysis_only=True, scan_flags=SCAN_LR_ONLY)")


# ------------------------------------------------------------------------------------------------ without a device
def test_scan_flag_constants_match_the_header():
    with open(os.path.join(ROOT, "include", "ldw.h")) as f:
        enum = dict(re.findall(r"\bLDW_SCAN_(\w+)\s*=\s*(\d+)", f.read()))
    assert len(enum) == 7 and {int(x) for x in enum.values()} == {1, 2, 4, 8, 16, 32, 64}
    for name, value in enum.items():
        assert getattr(api, "SCAN_" + name) == int(value), name


def test_cases_cover_the_block_kinds():
    """A: ragged last range, short-range pairs across the circular wrap.  B: every r from 2 to 5, a square off-diagonal
    block and ragged ones."""
    a, b = case("A"), case("B")
    assert len(a.blocks) == 10 and a.blocks[-1][1] - a.blocks[-1][0] + 1 == 700
    assert a.POS[0] + a.g - a.POS[-1] <= a.sr_dist            # the first and last SNPs are short-range neighbours
    assert set(np.unique(b.osnp.r)) == {2.0, 3.0, 4.0, 5.0}
    sizes = [(fe - fs + 1, te - ts + 1) for fs, fe, ts, te in b.blocks if fs != ts]
    assert (1000, 1000) in sizes and any(nt < 1000 for _, nt in sizes)


def test_ideal_q_restatement_against_the_compiled_oracle():
    """The IDEAL_Q reference on diagonal blocks, where quirk Q1 and the ideal Q are the same product, agrees with the compiled
    C oracle to 1e-12; on case B's off-diagonal blocks the two differ by more than 1e-6 somewhere."""
    import c_oracle as CO
    worst_diag, gap_off = 0.0, 0.0
    for name in ("A", "B"):
        c = case(name)
        for bi in range(len(c.blocks)):
            if name == "A" and not (c.diag[bi] and bi == len(c.blocks) - 1):
                continue                                       # case A: its ragged diagonal block only
            f, t = c.block_idx(bi)
            d = np.abs(ideal_q_block_mi(c.osnp, c.hdw, f, t) - CO.block_mi(c.codes, c.hdw, c.osnp.r, c.osnp.uqe, f, t)).max()
            if c.diag[bi]:
                worst_diag = max(worst_diag, float(d))
            else:
                gap_off = max(gap_off, float(d))
    print("diagonal blocks: max |ideal - C oracle|", worst_diag, "; case B off-diagonal:", gap_off)
    assert worst_diag <= 1e-12 and gap_off > 1e-6


def test_sr_only_with_lr_only_is_refused_before_any_device_work():
    """The flag check comes first in both entry points, before the plan or group is looked at and before a device is
    bound: no plan, no group and no GPU are needed to see the refusal."""
    L = api._lib.lib()
    sr, lr, bd = api._lib.Links(), api._lib.Links(), api._lib.Links()
    st = api._lib.ScanStats()
    for flags in (SR_ONLY | LR_ONLY, SR_ONLY | SR_EXACT | LR_ONLY | NO_D2H):
        rc = L.ldw_mi_scan(None, 1e6, 2e4, 1e4, 1e5, flags, 1, 0, C.byref(sr), C.byref(lr), C.byref(bd), None, None, C.byref(st))
        msg = L.ldw_last_error().decode()
        assert rc == 1 and "LDW_SCAN_SR_ONLY" in msg and "LDW_SCAN_LR_ONLY" in msg, msg
        rc = L.ldw_group_mi_scan(None, None, None, None, 1000, 1e6, 2e4, 1e4, 1e5, flags, C.byref(sr), C.byref(lr), C.byref(bd),
                                 None, None, None, None)
        msg = L.ldw_last_error().decode()
        assert rc == 1 and "LDW_SCAN_SR_ONLY" in msg and "LDW_SCAN_LR_ONLY" in msg, msg
    for flags in (SR_ONLY | NO_D2H, LR_ONLY | NO_D2H):   # each alone is a valid request: the next check speaks
        assert L.ldw_mi_scan(None, 1e6, 2e4, 1e4, 1e5, flags, 1, 0, None, None, None, None, None, None) == 1
        assert L.ldw_last_error().decode() == "null plan"
