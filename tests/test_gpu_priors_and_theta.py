"""-F reference-panel priors (mcb_params.use_prior, mcb_batch.prior_an / prior_ac; mcall.c:1507-1527) and -P theta (mcall.c:397-416)
in every calling kernel, against the oracle.

Both inputs feed the allele-set choice of every kernel: the prior rescales the per-allele quality sums, with the sample count of
the group it is applied to, and theta is added once per non-REF allele to every set's log-likelihood.  The batches mix sites
whose decision a few log units can move (most samples REF/REF, a few carriers with weak evidence) with the adversarial sites of
parity.random_batch, and the priors cover AC spread over 0..AN, AN of a reference panel and of a biobank, REF without support,
an ALT that only the panel supports, missing AC entries, vector_end before nals-1 entries, absent / zero / negative AN, and
entries past nals-1 that a kernel must not read (they would make AN < sum(AC)).

The first tests need only the CPU oracle: they check that these inputs change the oracle's decisions, so that a kernel cannot
pass the device tests by ignoring them.  The device tests compare every kernel with the oracle ("port": PL >= 256 next to
missing values is undefined in the reference, mcall.c:522, and the reference error()s out on a bad prior), with its sibling
kernel, and check which kernel ran.

theta <= 0 is not covered: the library passes it to the kernels unchanged (init_theta), and what the reference does with it has
not been established.
"""
import ctypes as C

import numpy as np
import pytest

from bcftools_b200 import abi
from tests import parity

gpu = pytest.mark.gpu

FLAGS = [0, abi.CALL_VARONLY]
S_CLASS = [37, 130, 1000, 2504]     # odd lane tails, the sample counts of the class tests, 1000 Genomes
THETAS = [1e-6, 0.02, 0.3]          # 0.3 x aM is clamped at 0.99 for S = 2504
DEFAULT_THETA = 1.1e-3
SITE_BAD_PRIOR = 1 << 7             # MCB_SITE_BAD_PRIOR, include/mcall_b200.h
SITE_PL_RANGE = 1 << 6              # MCB_SITE_PL_RANGE: a PL > 2500 was seen, parity with the reference not guaranteed

K_BW = "mcall_biallelic_warp_kernel"
K_TILED = "mcall_site_kernel"
K_W3 = "mcall_triallelic_warp_kernel"
K_W4 = "mcall_multi_warp_kernel"
K_CTA = "mcall_multi_kernel"
K_GEN = "mcall_generic_kernel"
K_GRP = "mcall_groups_kernel"
K_BGRP = "mcall_biallelic_groups_kernel"


# ---- inputs ---------------------------------------------------------------------------------------------------------------

def near_boundary(rng, batch, i):
    """Site i becomes mpileup-shaped: most samples REF/REF, one to four carriers of ALT alleles, PL = w x (alleles that differ
    from the truth), QS from the carriers.  The carriers' w is chosen so that adding their ALT to REF gains 0..13 log units
    before theta (a carrier gains about w ln(10)/10 + log(2f), and every sample loses about 2f, f = carriers / 2S): which set
    wins turns on theta and on the prior."""
    A, S = int(batch.nals[i]), batch.nsmpl
    truth = np.zeros((S, 2), np.int64)
    w = rng.uniform(40, 60, S)
    if A > 1:
        k = min(S, int(rng.integers(1, 5)))
        who = rng.choice(S, size=k, replace=False)
        truth[who, 1] = rng.integers(1, A, k)
        gain = rng.uniform(0, 13)
        w[who] = (gain / k + 1 - np.log(k / S)) * 10 / np.log(10) * rng.uniform(0.9, 1.1, k)
    blk = batch.site_pl(i)
    j = 0
    for x in range(A):
        for y in range(x + 1):
            d = np.minimum((x != truth[:, 0]).astype(int) + (y != truth[:, 1]), (x != truth[:, 1]).astype(int) + (y != truth[:, 0]))
            blk[:, j] = np.minimum(255, np.round(w * d)).astype(np.int32)
            j += 1
    cnt = np.array([(truth == a).sum() for a in range(A)], np.float64)
    batch.qs[i, :A] = (cnt * rng.uniform(20, 30, A)).astype(np.float32)
    if batch.ad is not None:            # -G: read depths of the true alleles
        batch.site_ad(i)[...] = (np.arange(A)[None, :, None] == truth[:, None, :]).sum(2) * rng.integers(3, 12, (S, 1))
    batch.unseen[i] = 0


def make_batch(seed, R, S, maxA, minA=1):
    """parity.random_batch with three sites in four near the decision boundary"""
    rng = np.random.default_rng(seed)
    batch = parity.random_batch(rng, R, S, maxA, minA=minA)
    for i in range(R):
        if i % 4:
            near_boundary(rng, batch, i)
    return batch


def add_priors(rng, batch, bad=(), an_max=5008):
    """prior_an / prior_ac for every site, by case (i mod 8): AN up to an_max, about 1e6 on case 1.  The sites in `bad` get
    sum(AC) = AN + 1.  Entries past nals-1 hold values above AN: a kernel that reads them, or uses the wrong row stride, sees a
    bad prior."""
    R, M = batch.nsites, batch.max_nals
    an = np.zeros(R, np.int32)
    ac = np.zeros((R, M), np.int32)
    bad = set(map(int, bad))
    for i in range(R):
        A = int(batch.nals[i])
        n = A - 1
        case = i % 8
        N = int(rng.integers(900_000, 1_100_000)) if case == 1 else int(rng.integers(20, an_max + 1))
        counts = rng.multinomial(N, rng.dirichlet(np.full(A, 0.4)))          # AC spread over 0..AN
        row = N + 1 + rng.integers(0, 1000, M)                               # not the site's: never read
        row[:n] = counts[1:]
        if n and case == 2:             # AC = AN for one ALT: no panel support for REF, and REF without QS either
            row[:n] = 0
            row[rng.integers(n)] = N
            if batch.qs is not None:
                batch.qs[i, 0] = 0
        elif n and case == 3:           # an ALT without QS that the panel supports: a dead allele comes alive
            k = int(rng.integers(n))
            if batch.qs is not None:
                batch.qs[i, k + 1] = 0
            w = rng.dirichlet(np.full(A, 0.4))
            w[k + 1] += 1
            row[:n] = rng.multinomial(N, w / w.sum())[1:]
        elif n and case == 5:           # vector_end before nals-1 entries; what follows it is never read
            row[int(rng.integers(n))] = abi.INT32_VECTOR_END
        elif case == 6:                 # no prior applied: AN missing, 0 or negative
            N = [abi.INT32_MISSING, 0, -7][i // 8 % 3]
        if n and case != 6 and rng.random() < 0.6:      # a missing AC keeps its allele's raw QS: the scales mix
            m = int(rng.integers(n))
            if row[m] != abi.INT32_VECTOR_END:
                row[m] = abi.INT32_MISSING
        if i in bad:
            assert n and case != 6, i
            live = [j for j in range(n) if row[j] >= 0]
            if not live:
                live = [n - 1]
                row[n - 1] = 0
            row[n:] = N + 1
            row[:n][row[:n] == abi.INT32_VECTOR_END] = 0
            tot = int(row[live].sum())
            row[live[-1]] += N + 1 - tot                # sum(AC) = AN + 1, on the last live entry
        an[i], ac[i] = N, row
    batch.prior_an, batch.prior_ac = an, ac
    return batch


def pick_bad(batch, rng, per_class=2):
    """a few sites of every allele count > 1 that can carry a prior (AN > 0)"""
    out = []
    for A in range(2, int(batch.nals.max()) + 1):
        cand = [i for i in np.where(batch.nals == A)[0] if i % 8 != 6]
        out += list(rng.choice(cand, size=min(per_class, len(cand)), replace=False)) if cand else []
    return sorted(map(int, out))


def mixed_groups(S, seed):
    """big groups (whole-CTA path) next to small ones (warp path) with interleaved sample indices, as test_sample_groups"""
    perm = np.random.default_rng([S, seed]).permutation(S)
    cuts = [0, 150, 250, 290, S]
    return [sorted(perm[cuts[k]:cuts[k + 1]].tolist()) for k in range(4)]


def ploidy_012(rng, batch, S):
    tab = np.full((3, S), 2, np.uint8)
    tab[1, ::2] = 1
    tab[2, ::3] = 1
    tab[2, 1::5] = 0
    batch.ploidy_id = rng.integers(0, 3, batch.nsites).astype(np.uint16)
    return tab


def with_params(params, **kw):
    d = dict(nsmpl=params.nsmpl, max_nals=params.max_nals, theta=params.theta, init_ploidy=params.init_ploidy, flag=params.flag,
             output_tags=params.output_tags, groups=params.groups, use_prior=params.use_prior, tie_eps=params.tie_eps)
    d.update(kw)
    return abi.CallParams(**d)


def decided(res):
    """per site: the allele set chosen and the genotypes, for the discrimination checks"""
    return [(int(res.ret[i]), int(res.als_new[i]) if res.ret[i] > 0 else 0, res.gt[i].tobytes() if res.ret[i] > 0 else b"")
            for i in range(len(res.ret))]


def share_changed(a, b, res):
    called = res.ret > 0
    da, db = decided(a), decided(b)
    diff = np.array([x != y for x, y in zip(da, db)])
    return float((diff & called).sum()) / max(1, int(called.sum()))


def pad_groups_to_nsmpl(params, batch, tab):
    """The same -G call with every group padded to nsmpl samples by samples that carry no data (PL missing, AD 0, init ploidy 0):
    they change nothing but the sample count the prior divides by (mcall.c:1514, 1524), so the oracle on this batch computes
    what a kernel that used nsmpl in place of the group size would."""
    S, G = params.nsmpl, params.groups
    extra = [S - len(g) for g in G]
    S2 = S + sum(extra)
    groups, nxt = [], S
    for g, e in zip(G, extra):
        groups.append(list(g) + list(range(nxt, nxt + e)))
        nxt += e
    blocks, ads = [], []
    for i in range(batch.nsites):
        pl = batch.site_pl(i)
        pad = np.full((S2 - S, pl.shape[1]), abi.INT32_VECTOR_END, np.int32)
        pad[:, 0] = abi.INT32_MISSING
        blocks.append(np.vstack([pl, pad]))
        ad = batch.site_ad(i)
        ads.append(np.vstack([ad, np.zeros((S2 - S, ad.shape[1]), np.int32)]))
    b2 = abi.HostBatch(S2, batch.max_nals, batch.nals, pl_blocks=blocks, unseen=batch.unseen, ploidy_id=batch.ploidy_id,
                       qs=batch.qs, ad_blocks=ads, prior_an=batch.prior_an, prior_ac=batch.prior_ac)
    init = np.r_[np.full(S, 2), np.zeros(S2 - S)].astype(np.uint8)
    p2 = abi.CallParams(S2, params.max_nals, theta=params.theta, init_ploidy=init, flag=params.flag, output_tags=params.output_tags,
                        groups=groups, use_prior=params.use_prior)
    t2 = None if tab is None else np.hstack([tab, np.full((tab.shape[0], S2 - S), 2, np.uint8)])
    return p2, b2, t2


# ---- the oracle alone: the inputs discriminate --------------------------------------------------------------------------

def prior_case(S=130, maxA=5, flag=0, seed=1):
    batch = add_priors(np.random.default_rng([S, seed]), make_batch([S, maxA, seed], 120, S, maxA))
    return abi.CallParams(S, maxA, flag=flag, output_tags=abi.CALL_FMT_GQ, use_prior=True), batch


def test_oracle_decisions_depend_on_the_prior(oracle_built):
    for S in (130, 1000):
        params, batch = prior_case(S)
        exp, _ = oracle_built.call("port", params, batch)
        off, _ = oracle_built.call("port", with_params(params, use_prior=False), batch)
        assert share_changed(exp, off, exp) >= 0.10, S
        zero = abi.HostBatch.subset(batch, range(batch.nsites))
        zero.prior_ac[zero.prior_ac == abi.INT32_MISSING] = 0
        z, _ = oracle_built.call("port", params, zero)
        assert share_changed(exp, z, exp) >= 0.10, S
        # REF-only and variant calls, at sites of 1..5 alleles
        called = exp.ret > 0
        assert ((exp.ret == 1) & (batch.nals > 1)).any() and (exp.ret > 1).any()
        assert set(batch.nals[called].tolist()) == {1, 2, 3, 4, 5}


def mixed_scale(batch):
    """sites whose prior leaves some allele's raw quality sum next to rescaled ones (a missing AC, or vector_end before nals-1
    entries): only there does the sample count the prior divides by reach the decision.  Elsewhere every allele is divided by
    the same number, which the normalisation (mcall.c:1530-1535) cancels."""
    out = np.zeros(batch.nsites, bool)
    for i in range(batch.nsites):
        r = batch.prior_ac[i, :int(batch.nals[i]) - 1]
        out[i] = batch.prior_an[i] > 0 and ((r == abi.INT32_MISSING) | (r == abi.INT32_VECTOR_END)).any()
    return out


GROUP_AN = 1000     # -G: a panel of 500 diploid samples, so that the group size weighs against AN / 2


def test_oracle_grouped_decisions_depend_on_the_group_size(oracle_built):
    S = 300
    rng = np.random.default_rng(3)
    batch = add_priors(rng, make_batch([S, 3], 120, S, 5), an_max=GROUP_AN)
    tab = ploidy_012(rng, batch, S)
    params = abi.CallParams(S, 5, output_tags=abi.CALL_FMT_GQ, groups=mixed_groups(S, 3), use_prior=True)
    exp, _ = oracle_built.call("port", params, batch, tab)
    p2, b2, t2 = pad_groups_to_nsmpl(params, batch, tab)
    padded, _ = oracle_built.call("port", p2, b2, t2)
    padded.gt = padded.gt[:, :S]
    m = mixed_scale(batch)
    assert m.sum() >= batch.nsites // 3
    changed = np.array([x != y for x, y in zip(decided(exp), decided(padded))])
    assert changed[m & (exp.ret > 0)].mean() >= 0.10
    # the padding itself changes nothing without a prior
    e0, _ = oracle_built.call("port", with_params(params, use_prior=False), batch, tab)
    p0, _ = oracle_built.call("port", with_params(p2, use_prior=False), b2, t2)
    p0.gt = p0.gt[:, :S]
    assert share_changed(e0, p0, e0) == 0.0


@pytest.mark.parametrize("theta", THETAS)
def test_oracle_decisions_depend_on_theta(theta, oracle_built):
    for S in (130, 2504):
        batch = theta_batch(S, 5)
        params = abi.CallParams(S, 5, theta=theta, output_tags=abi.CALL_FMT_GQ)
        exp, _ = oracle_built.call("port", params, batch)
        base, _ = oracle_built.call("port", with_params(params, theta=DEFAULT_THETA), batch)
        assert share_changed(exp, base, exp) >= 0.10, S


@pytest.mark.parametrize("grouped", [False, True])
def test_bad_priors_stop_the_oracle(grouped, oracle_built):
    params, batch, tab, bad = bad_prior_case(grouped)
    assert len(set(batch.nals[bad].tolist())) == 7          # 2..8 alleles
    with pytest.raises(RuntimeError, match=str(abi.MCB_EPRIOR)):
        oracle_built.call("port", params, batch, tab)
    for i in bad:                                           # each one alone stops it
        with pytest.raises(RuntimeError, match=str(abi.MCB_EPRIOR)):
            oracle_built.call("port", params, batch.subset([i]), tab)
    good = [i for i in range(batch.nsites) if i not in bad]
    oracle_built.call("port", params, batch.subset(good), tab)


# ---- device runs ------------------------------------------------------------------------------------------------------------

def run(params, batch, options, tab=None, compact=False, typed=False, want_gp=False):
    """call_host with the given options; returns (result, names of the CUDA kernels that ran, launches counted by the library)"""
    import torch
    from torch.profiler import ProfilerActivity, profile
    from bcftools_b200 import mcall
    with mcall.MCaller(params, ploidy_tab=tab, options=options) as mc:
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            got = mc.call_host(batch, compact=compact, typed=typed, want_gp=want_gp)
            torch.cuda.synchronize()
        launches = int(mc.stats()[0])
    return (got.widen() if typed else got), {e.name for e in prof.events()}, launches


def ran(names, kernel, targ=None):
    """some kernel of that name ran; with targ, the instance whose template argument is targ (allele count, PLOIDY)"""
    return any(kernel in n and (targ is None or f"<{targ}>" in n.replace(" ", "")) for n in names)


def assert_same_calls_off_ties(got, ref, params, near_share=0.05):
    """assert_same_calls on every site that neither run flags MCB_SITE_NEAR_TIE.  Sibling kernels sum a site's log-likelihoods in
    different orders, so the last bits of two nearly tied sets may order them differently: parity.compare exempts such sites
    against the oracle by the same rule.  Near ties must stay a small share of the sites."""
    tie = ((got.site_flags | ref.site_flags) & abi.SITE_NEAR_TIE) != 0
    assert tie.sum() <= near_share * len(tie) + 1, np.where(tie)[0]
    keep = np.where(~tie)[0]
    for name in ("ret", "als_new", "als_map", "ac", "an", "site_flags", "gt", "gq"):
        a, b = getattr(got, name)[keep], getattr(ref, name)[keep]
        assert (a == b).all(), (name, keep[np.argwhere(a != b)[:5, 0]])
    for i in keep:
        if ref.ret[i] > 0 and not (ref.site_flags[i] & abi.SITE_PL_DROPPED):
            assert (got.site_pl(i) == ref.site_pl(i)).all(), (i, "pl")
    a, b = got.qual[keep], ref.qual[keep]
    same = (a.view(np.uint32) == b.view(np.uint32)) | (np.isnan(a) & np.isnan(b))
    rel = np.where(same, 0.0, np.abs(a.astype(np.float64) - b) / np.maximum(np.abs(b.astype(np.float64)), 1e-30))
    assert rel.max(initial=0.0) <= parity.QUAL_RTOL, (int(keep[rel.argmax()]), rel.max())


def check(got, exp, params, near_share=0.05):
    st = parity.compare(got, exp, params)
    assert st["compared"] > 0, st
    assert len(st["near_ties"]) <= near_share * len(exp.ret) + 1, st["near_ties"]
    return st


def pooled_matrix(params, batch, exp, S, tab=None):
    """default kernels, the CTA kernel of 3-4 alleles and the tiled kernel, each against the oracle; the warp kernels of 3 and 4
    alleles against the CTA kernel"""
    multi = S % 2 == 0 and S >= 128 and tab is None
    got, names, _ = run(params, batch, {}, tab=tab, compact=True)
    check(got, exp, params)
    assert ran(names, K_BW, "false" if tab is None else "true"), sorted(names)      # the PLOIDY instance with a ploidy table
    if multi:
        assert ran(names, K_W3) and ran(names, K_CTA), sorted(names)
        assert ran(names, K_W4, 4) == (S <= 2504), sorted(names)
        cta, names, _ = run(params, batch, {"warp3": 0, "warp4": 0}, tab=tab, compact=True)
        assert ran(names, K_CTA) and not ran(names, K_W3) and not ran(names, K_W4), sorted(names)
        check(cta, exp, params)
        assert_same_calls_off_ties(got, cta, params)
    tiled, names, _ = run(params, batch, {"block": 128}, tab=tab)
    assert ran(names, K_TILED) and not ran(names, K_BW) and not ran(names, K_CTA), sorted(names)
    check(tiled, exp, params)


@gpu
@pytest.mark.parametrize("flag", FLAGS)
@pytest.mark.parametrize("S", S_CLASS)
def test_prior_pooled_kernels(S, flag, oracle_built):
    """1-5 alleles with priors: two-allele warp kernel, 3- and 4-allele warp kernels, CTA kernel (5 alleles, and 3-4 with
    warp3=0 / warp4=0), tiled kernel"""
    params, batch = prior_case(S, 5, flag, seed=2)
    if S > 1500:
        batch = batch.subset(range(60))
    exp, _ = oracle_built.call("port", params, batch)
    pooled_matrix(params, batch, exp, S)


@gpu
@pytest.mark.parametrize("S", [37, 1000])
def test_prior_two_allele_kernel_under_ploidy_vectors(S, oracle_built):
    """the PLOIDY instance of the two-allele warp kernel (ploidy 0 / 1 / 2) against the oracle and the tiled kernel"""
    rng = np.random.default_rng([S, 4])
    batch = add_priors(rng, make_batch([S, 4], 96, S, 2, minA=2))
    tab = ploidy_012(rng, batch, S)
    params = abi.CallParams(S, 2, output_tags=abi.CALL_FMT_GQ, use_prior=True)
    exp, _ = oracle_built.call("port", params, batch, tab)
    pooled_matrix(params, batch, exp, S, tab=tab)


@gpu
@pytest.mark.parametrize("flag", [0, abi.CALL_KEEPALT])
def test_prior_tiled_two_allele_kernel_above_8192_samples(flag, oracle_built):
    S = 8194
    batch = add_priors(np.random.default_rng([S, 5]), make_batch([S, 5], 24, S, 2, minA=2))
    params = abi.CallParams(S, 2, flag=flag, output_tags=abi.CALL_FMT_GQ, use_prior=True)
    exp, _ = oracle_built.call("port", params, batch)
    got, names, _ = run(params, batch, {}, compact=True)
    assert ran(names, K_TILED) and not ran(names, K_BW), sorted(names)
    check(got, exp, params)


@gpu
def test_prior_keepalt_on_the_tiled_kernel(oracle_built):
    """KEEPALT keeps 3-5 allele sites off the class kernels: every class on the tiled kernel"""
    params, batch = prior_case(130, 5, abi.CALL_KEEPALT, seed=6)
    exp, _ = oracle_built.call("port", params, batch)
    got, names, _ = run(params, batch, {})
    assert ran(names, K_TILED) and not ran(names, K_CTA) and not ran(names, K_W3), sorted(names)
    check(got, exp, params)


@gpu
@pytest.mark.parametrize("S,maxA,grouped", [(150, 8, False), (12, 32, False), (300, 8, True)])
def test_prior_more_than_five_alleles(S, maxA, grouped, oracle_built):
    """6..32 alleles with priors (mcall_generic.cu), mixed with 1..5 allele sites, pooled and -G"""
    rng = np.random.default_rng([S, maxA, 7])
    batch = add_priors(rng, make_batch([S, maxA, 7], 40 if maxA > 16 else 90, S, maxA), an_max=GROUP_AN if grouped else 5008)
    tab = ploidy_012(rng, batch, S)
    params = abi.CallParams(S, maxA, output_tags=abi.CALL_FMT_GQ, groups=mixed_groups(S, 7) if grouped else None, use_prior=True)
    exp, _ = oracle_built.call("port", params, batch, tab)
    got, names, _ = run(params, batch, {}, tab=tab)
    assert ran(names, K_GEN), sorted(names)
    assert (batch.nals[got.ret > 0] > 5).any()
    check(got, exp, params)


@gpu
@pytest.mark.parametrize("flag", FLAGS)
def test_prior_sample_groups(flag, oracle_built):
    """-G with groups of 150 / 100 / 40 / 10 samples: the group-per-warp and the whole-CTA paths of mcall_groups.cu, and the
    two-allele grouped warp kernel, each dividing by its own group's sample count"""
    S = 300
    rng = np.random.default_rng([S, flag, 8])
    batch = add_priors(rng, make_batch([S, flag, 8], 120, S, 5), an_max=GROUP_AN)
    tab = ploidy_012(rng, batch, S)
    params = abi.CallParams(S, 5, flag=flag, output_tags=abi.CALL_FMT_GQ, groups=mixed_groups(S, 8), use_prior=True)
    exp, _ = oracle_built.call("port", params, batch, tab)
    got, names, n_new = run(params, batch, {}, tab=tab)
    assert ran(names, K_GRP) and ran(names, K_BGRP), sorted(names)
    check(got, exp, params)
    old, names, n_old = run(params, batch, {"bgroups": 0}, tab=tab)
    assert not ran(names, K_BGRP) and n_new == n_old + 1
    check(old, exp, params)


@gpu
@pytest.mark.parametrize("S", [130, 1000])
@pytest.mark.parametrize("ng", [2, 3, 5])
def test_prior_two_allele_grouped_kernel(S, ng, oracle_built):
    """the warp-per-site kernel of mcall_biallelic_groups.cu (bgroups=1) with 2-5 groups, against the oracle and mcall_groups.cu"""
    rng = np.random.default_rng([S, ng, 9])
    batch = add_priors(rng, make_batch([S, ng, 9], 96, S, 2, minA=2), an_max=GROUP_AN)
    tab = ploidy_012(rng, batch, S)
    params = abi.CallParams(S, 2, output_tags=abi.CALL_FMT_GQ, groups=[list(range(k, S, ng)) for k in range(ng)], use_prior=True)
    exp, _ = oracle_built.call("port", params, batch, tab)
    got, names, n_new = run(params, batch, {"bgroups": 1}, tab=tab)
    assert ran(names, K_BGRP), sorted(names)
    check(got, exp, params)
    old, _, n_old = run(params, batch, {"bgroups": 0}, tab=tab)
    assert n_new == n_old + 1
    check(old, exp, params)


@gpu
@pytest.mark.parametrize("grouped", [False, True])
def test_prior_literal_phase1(grouped, oracle_built):
    """exact_phase1=1, and adjudicate=1 with every site a near tie (compacted output): the literal sums of logs with priors"""
    S = 300
    rng = np.random.default_rng([S, int(grouped), 10])
    batch = add_priors(rng, make_batch([S, int(grouped), 10], 80, S, 7), an_max=GROUP_AN if grouped else 5008)
    tab = ploidy_012(rng, batch, S)
    params = abi.CallParams(S, 7, output_tags=abi.CALL_FMT_GQ, groups=mixed_groups(S, 10) if grouped else None, use_prior=True)
    exp, _ = oracle_built.call("port", params, batch, tab)
    got, names, _ = run(params, batch, {"exact_phase1": 1}, tab=tab)
    assert not ran(names, K_BW) and not ran(names, K_BGRP), sorted(names)
    st = check(got, exp, params)
    assert not st["near_ties"], st
    adj, _, _ = run(with_params(params, tie_eps=1e30), batch, {"adjudicate": 1}, tab=tab, compact=True)
    st = parity.compare(adj, exp, params)
    assert st["compared"] > 0 and not st["near_ties"], st
    called = adj.ret > 0
    assert ((adj.site_flags[called] & abi.SITE_ADJUDICATED) != 0).mean() > 0.3


@gpu
def test_prior_transports(oracle_built):
    """int16 PL in, BCF typed int8 / int16 out, and FORMAT/GP, with priors"""
    params, batch = prior_case(130, 5, seed=11)
    exp, _ = oracle_built.call("port", params, batch)
    for typed in (False, True):
        got, _, _ = run(params, batch.to_int16(), {}, compact=True, typed=typed)
        check(got, exp, params)
    pg = with_params(params, output_tags=abi.CALL_FMT_GQ | abi.CALL_FMT_GP)
    exp, _ = oracle_built.call("port", pg, batch, want_gp=True)
    got, _, _ = run(pg, batch, {}, want_gp=True)
    check(got, exp, pg)


@gpu
@pytest.mark.parametrize("async_flush", [False, True])
def test_prior_host_batcher(async_flush, oracle_built):
    """b200_mcall with use_prior: the per-record AN / AC go through the batcher's slabs over several flushes"""
    from bcftools_b200 import host_call
    params, batch = prior_case(130, 5, seed=12)
    exp, _ = oracle_built.call("port", params, batch)
    got = host_call.replay(params, batch, None, max_records=37, async_flush=async_flush)
    check(got, exp, params)


# ---- bad priors: AN < sum(AC) ------------------------------------------------------------------------------------------------

def bad_prior_case(grouped):
    S, maxA = 300, 8
    rng = np.random.default_rng([S, int(grouped), 13])
    batch = make_batch([S, int(grouped), 13], 96, S, maxA)
    bad = pick_bad(batch, rng)
    add_priors(rng, batch, bad)
    tab = ploidy_012(rng, batch, S) if grouped else None       # pooled: every sample diploid, so that the 3-5 allele class kernels run
    params = abi.CallParams(S, maxA, output_tags=abi.CALL_FMT_GQ, groups=mixed_groups(S, 13) if grouped else None, use_prior=True)
    return params, batch, tab, bad


def take(res, batch, idx, sub):
    """the rows `idx` of an in-place result of `batch`, as a result of the batch `sub` = batch.subset(idx)"""
    out = abi.HostResult(sub)
    for name in ("ret", "als_new", "als_map", "qual", "ac", "an", "site_flags", "gt", "gq"):
        getattr(out, name)[...] = getattr(res, name)[idx]
    for k, i in enumerate(idx):
        n = batch.nsmpl * int(batch.ngt[i])
        out.pl[sub.pl_off[k]:sub.pl_off[k] + n] = res.pl[batch.pl_off[i]:batch.pl_off[i] + n]
    return out


BAD_RUNS = [(False, {}), (False, {"warp3": 0, "warp4": 0}), (False, {"block": 128}), (False, {"exact_phase1": 1}),
            (True, {}), (True, {"bgroups": 0}), (True, {"exact_phase1": 1})]


@gpu
@pytest.mark.parametrize("grouped,options", BAD_RUNS)
def test_bad_priors_are_flagged(grouped, options, oracle_built):
    """MCB_SITE_BAD_PRIOR on exactly the sites with AN < sum(AC) (2..8 alleles; never on a 1-allele site, whose AC entries are
    not read), and every other site as the oracle calls it without the bad ones"""
    params, batch, tab, bad = bad_prior_case(grouped)
    good = [i for i in range(batch.nsites) if i not in bad]
    sub = batch.subset(good)
    exp, _ = oracle_built.call("port", params, sub, tab)
    got, names, _ = run(params, batch, options, tab=tab)
    if not grouped and not options:
        assert ran(names, K_BW) and ran(names, K_W3) and ran(names, K_W4, 4) and ran(names, K_CTA) and ran(names, K_GEN), sorted(names)
    flagged = np.where(got.site_flags & SITE_BAD_PRIOR)[0].tolist()
    assert flagged == bad, (flagged, bad)
    check(take(got, batch, good, sub), exp, params)


@gpu
@pytest.mark.parametrize("async_flush", [False, True])
def test_bad_priors_reach_the_batcher_error_handler(async_flush, oracle_built):
    """the batcher reports every flagged record through the error handler (the reference stops there, mcall.c:1523); with a handler
    that returns, the other records still come back as the oracle calls them"""
    from bcftools_b200 import host_call, mcall
    params, batch, tab, bad = bad_prior_case(False)
    R = 16
    msgs = []
    HANDLER = C.CFUNCTYPE(None, C.c_char_p)
    handler = HANDLER(lambda m: msgs.append(m.decode()))
    set_handler = C.CFUNCTYPE(None, HANDLER)(("b200_set_error_handler", mcall.lib()))    # a local prototype: the shared handle stays as it is
    set_handler(handler)
    try:
        got = host_call.replay(params, batch, tab, max_records=R, async_flush=async_flush)
    finally:
        set_handler(HANDLER())                      # back to the default handler
    assert msgs == [f"Incorrect prior AN,AC values at record {i % R} of the batch\n" for i in bad], msgs
    good = [i for i in range(batch.nsites) if i not in bad]
    sub = batch.subset(good)
    exp, _ = oracle_built.call("port", params, sub, tab)
    check(take(got, batch, good, sub), exp, params)


# ---- theta --------------------------------------------------------------------------------------------------------------------

def oracle_theta_fn(pyoracle):
    lib = C.CDLL(pyoracle.PORT_SO)
    f = lib.oracle_theta
    f.restype = C.c_double
    f.argtypes = [C.c_double, C.c_void_p, C.c_int]
    return f


@gpu
def test_theta_is_the_oracles_bit_for_bit(oracle_built):
    """log(theta x aM), aM = sum 1/i over the ploidy sum at init, clamped at 0.99 (mcall.c:397-416)"""
    from bcftools_b200 import mcall
    f = oracle_theta_fn(oracle_built)
    clamped = 0
    for S in (1, 2, 2504):
        mixed = np.array([(0, 1, 2)[s % 3] for s in range(S)], np.uint8)
        for init in (None, np.full(S, 2, np.uint8), mixed):
            for theta in (1e-6, 1.1e-3, 0.02, 0.3, 0.99):
                params = abi.CallParams(S, 5, theta=theta, init_ploidy=init)
                with mcall.MCaller(params) as mc:
                    got = mc.theta
                want = f(theta, None if init is None else init.ctypes.data, S)
                assert np.float64(got).view(np.uint64) == np.float64(want).view(np.uint64), (S, init, theta, got, want)
                clamped += want == np.log(0.99)
    assert clamped >= 3


def theta_batch(S, maxA, minA=1):
    """make_batch with every tenth site a one-allele site with data: no variant set is evaluated there, so QUAL is
    -4.343 theta (mcall.c:1641)"""
    R = 60 if S > 1500 else 120
    b = make_batch([S, maxA, 14], R, S, maxA, minA=minA)
    one = np.arange(R) % 10 == 0
    nals = np.where(one, 1, b.nals)
    rng = np.random.default_rng([S, maxA, 15])
    blocks = [rng.integers(1, 60, (S, 1)) if one[i] else b.site_pl(i) for i in range(R)]
    ads = [rng.integers(1, 20, (S, 1)) if one[i] else b.site_ad(i) for i in range(R)]
    return abi.HostBatch(S, maxA, nals, pl_blocks=blocks, unseen=np.where(one, 0, b.unseen), qs=b.qs, ad_blocks=ads)


def check_theta_quals(got, exp, batch, theta_log):
    """the one-allele sites carry QUAL = -4.343 theta"""
    ref_only = [i for i in range(0, batch.nsites, 10) if exp.ret[i] > 0]
    assert ref_only
    for i in ref_only:
        assert exp.qual[i] == np.float32(-4.343 * theta_log), (i, exp.qual[i])
        assert got.qual.view(np.uint32)[i] == exp.qual.view(np.uint32)[i], (i, got.qual[i], exp.qual[i])


def no_variant_set_batch(S, grouped):
    """Sites of 2..5 and 7 alleles at which the reference evaluates no variant set, so that QUAL is -4.343 theta (mcall.c:1641):
    the ALTs have no QS (or, for -G, no read depth), so no set of two or three alleles is tried, and every ALT homozygote has
    PL 4000, whose likelihood 10^-400 is 0, so the one-ALT sets have no sample with data (mcall.c:608-613)."""
    rng = np.random.default_rng([S, int(grouped), 17])
    nals = np.resize(np.array([2, 3, 4, 5, 7], np.uint8), 25)
    blocks, ads = [], []
    for A in map(int, nals):
        pl = rng.integers(1, 60, (S, A * (A + 1) // 2)).astype(np.int32)
        pl[:, 0] = 0
        for a in range(1, A):
            pl[:, (a + 1) * (a + 2) // 2 - 1] = 4000
        blocks.append(pl)
        ad = np.zeros((S, A), np.int32)
        ad[:, 0] = rng.integers(1, 20, S)
        ads.append(ad)
    qs = np.zeros((len(nals), 7), np.float32)
    qs[:, 0] = rng.uniform(100, 1000, len(nals))
    return abi.HostBatch(S, 7, nals, pl_blocks=blocks, qs=qs, ad_blocks=ads)


@gpu
@pytest.mark.parametrize("theta", THETAS)
@pytest.mark.parametrize("grouped", [False, True])
def test_theta_qual_where_no_variant_set_is_evaluated(theta, grouped, oracle_built):
    """QUAL = -4.343 theta at sites of 2..7 alleles.  The literal phase 1 (exact_phase1: the general, 6..32-allele and -G kernels)
    leaves samples with likelihood 0 out of a set's sum of logs as the reference does, and must give the oracle's QUAL bit for bit.
    The class kernels sum the one-ALT sets from integer PL sums and do not; PL > 2500 is outside the range in which they claim
    parity (DESIGN.md, edge semantics), so there they must flag every such site MCB_SITE_PL_RANGE and still call REF only."""
    from bcftools_b200 import mcall
    S = 300
    batch = no_variant_set_batch(S, grouped)
    params = abi.CallParams(S, 7, theta=theta, output_tags=abi.CALL_FMT_GQ, groups=mixed_groups(S, 17) if grouped else None)
    exp, _ = oracle_built.call("port", params, batch)
    with mcall.MCaller(params) as mc:
        want = np.float32(-4.343 * mc.theta)
    assert (exp.ret == 1).all() and (exp.qual == want).all(), (exp.ret, exp.qual, want)
    got, names, _ = run(params, batch, {"exact_phase1": 1})
    assert ran(names, K_GRP if grouped else K_TILED) and (grouped or ran(names, K_GEN)), sorted(names)
    check(got, exp, params)
    assert (got.qual.view(np.uint32) == exp.qual.view(np.uint32)).all(), (got.qual, want)
    fast, names, _ = run(params, batch, {})
    assert ((fast.site_flags & SITE_PL_RANGE) != 0).all(), fast.site_flags
    assert (fast.ret == 1).all() and (fast.als_new == 1).all() and (fast.gt == exp.gt).all()


@gpu
@pytest.mark.parametrize("theta", THETAS)
@pytest.mark.parametrize("S", [130, 2504])
def test_theta_pooled_kernels(S, theta, oracle_built):
    """two-allele warp, 3- and 4-allele warp and CTA kernels, 5-allele CTA kernel, tiled kernel at non-default theta"""
    from bcftools_b200 import mcall
    batch = theta_batch(S, 5)
    params = abi.CallParams(S, 5, theta=theta, output_tags=abi.CALL_FMT_GQ)
    exp, _ = oracle_built.call("port", params, batch)
    pooled_matrix(params, batch, exp, S)
    got, _, _ = run(params, batch, {})
    with mcall.MCaller(params) as mc:
        check_theta_quals(got, exp, batch, mc.theta)


@gpu
@pytest.mark.parametrize("theta", THETAS)
def test_theta_generic_grouped_and_literal(theta, oracle_built):
    """6..8 alleles (generic kernel), -G with the mixed grouping, and exact_phase1, at non-default theta"""
    from bcftools_b200 import mcall
    S = 300
    rng = np.random.default_rng([S, 15])
    batch = theta_batch(S, 8)
    tab = ploidy_012(rng, batch, S)
    for groups, options, kernel in ((None, {}, K_GEN), (mixed_groups(S, 15), {}, K_GRP), (None, {"exact_phase1": 1}, K_TILED),
                                    (mixed_groups(S, 15), {"exact_phase1": 1}, K_GRP)):
        params = abi.CallParams(S, 8, theta=theta, output_tags=abi.CALL_FMT_GQ, groups=groups)
        exp, _ = oracle_built.call("port", params, batch, tab)
        got, names, _ = run(params, batch, options, tab=tab)
        assert ran(names, kernel), (options, sorted(names))
        check(got, exp, params)
        with mcall.MCaller(params) as mc:
            check_theta_quals(got, exp, batch, mc.theta)
