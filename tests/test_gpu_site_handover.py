"""Every persistent calling kernel over long runs of sites per warp or CTA, and one context over many calls, against the oracle.

The kernels claim sites from a work counter (or walk a static stride) until their class list is empty, and carry state from one
site to the next: the ring position and mbarrier parity of the tiled and CTA-per-site kernels, the set-up of the next site that
the CTA kernel prepares during the current one, the per-warp records and packed copies of the warp kernels, the per-CTA scratch
of the grouped and 6..32-allele kernels.  A device-sized grid gives almost every worker one site of a test batch, so option
max_ctas caps the launched grid (and nothing else: the same kernels run, with the same scratch) and every case asserts from its
own arguments that each worker calls at least MIN_RUN sites.  Neighbouring sites differ in everything that state depends on:
REF-only, pair, triple and no-REF outcomes, VARONLY sites that end early, sites without QS or with dead alleles, the unseen allele
selected, no listed rows / a few / more than the 32 the class kernels hold (those sites punt to the general kernel), PL >= 256,
good and bad -F priors, ploidy ids 0 / 1 / 2.

Each capped call is compared with the oracle and, bit for bit, with the same call without the cap, fallback counts included: a
hand-over slip that only sends sites to the fallback list changes nothing else.  The rest of the file runs the real dynamic claim
on 20,000-site batches of replicated sites, one context over a sequence of batches of changing size and shape, and two calls into
one result whose buffers start out poisoned.
"""
import numpy as np
import pytest

from bcftools_b200 import abi, synth
from tests import parity
from tests.test_gpu_parity import ORACLE
from tests.test_gpu_priors_and_theta import (K_BGRP, K_BW, K_CTA, K_GEN, K_GRP, K_TILED, K_W3, K_W4, SITE_BAD_PRIOR, add_priors,
                                            mixed_groups, near_boundary, pick_bad, ploidy_012, ran)

pytestmark = pytest.mark.gpu

MIN_RUN = 8             # sites per worker every capped case must reach
BW_MAXWARP, TW_MAXWARP, MW_MAXWARP, BG_WARPS = 14, 7, 8, 8      # warps per CTA of the warp kernels (mcall_biallelic.cu, ...)


# ---- inputs ---------------------------------------------------------------------------------------------------------------

def listed(rng, blk, n, kind):
    """n listed rows: missing (vector_end behind a missing value) or partially missing"""
    S, G = blk.shape
    rows = rng.choice(S, size=min(n, S), replace=False)
    for s in rows:
        if kind == "partial" and G > 1:
            blk[s, rng.integers(1, G)] = abi.INT32_MISSING
        else:
            blk[s] = abi.INT32_VECTOR_END
            blk[s, 0] = abi.INT32_MISSING


def handover_batch(seed, R, S, maxA, minA, priors=True):
    """R sites of minA..maxA alleles, kind by site index (the class lists are filled by atomics, so their order is not fixed):
    0 adversarial, with 40 listed rows (punts from the class kernels); 1 mpileup-shaped, no listed rows; 2 mpileup-shaped with a
    few listed rows; 3 no QS at all; 4 uniform PLs, a few listed rows, some QS zero (dead alleles), unseen allele kept; 5 clean
    uniform PLs.  Every fifth site has PL >= 256 entries.  With priors: -F AN / AC for every site and AN < sum(AC) on a few.
    Returns the batch and the sites with bad priors."""
    rng = np.random.default_rng(seed)
    batch = parity.random_batch(rng, R, S, maxA, minA=minA, miss=False)
    for i in range(R):
        blk = batch.site_pl(i)
        A = int(batch.nals[i])
        kind = i % 6
        if kind in (1, 2):
            near_boundary(rng, batch, i)
            if kind == 2:
                listed(rng, blk, int(rng.integers(1, 8)), "partial" if i % 4 else "missing")
        elif kind == 0:
            listed(rng, blk, 40, "missing")
        elif kind == 3:
            batch.qs[i] = 0
        elif kind == 4:
            listed(rng, blk, int(rng.integers(1, 6)), "partial")
        else:
            batch.unseen[i] = 0
            batch.qs[i, :A] = (1 + rng.random(A) * 10).astype(np.float32)
        if i % 5 == 0:
            ok = np.where(blk[:, 0] >= 0)[0]
            blk[rng.choice(ok, size=min(3, len(ok)), replace=False), rng.integers(0, blk.shape[1], min(3, len(ok)))] = 300
    bad = []
    if priors:
        bad = pick_bad(batch, rng)
        add_priors(rng, batch, bad)
    return batch, bad


def params_for(S, maxA, flag=0, priors=True, **kw):
    return abi.CallParams(S, maxA, flag=flag, output_tags=abi.CALL_FMT_GQ | kw.pop("tags", 0), use_prior=priors, **kw)


def restrict(res, idx, sub):
    """rows `idx` of a result (in place or compacted) as an in-place result of sub = batch.subset(idx)"""
    out = abi.HostResult(sub, want_gp=res.gp is not None)
    for name in ("ret", "als_new", "als_map", "qual", "ac", "an", "site_flags", "diag", "gt", "gq"):
        getattr(out, name)[...] = getattr(res, name)[idx]
    for k, i in enumerate(idx):
        if res.ret[i] > 0 and not (res.site_flags[i] & abi.SITE_PL_DROPPED):
            p = res.site_pl(i)
            out.pl[sub.pl_off[k]:sub.pl_off[k] + p.size] = p.reshape(-1)
            if res.gp is not None:
                g = res.site_gp(i)
                out.gp[sub.pl_off[k]:sub.pl_off[k] + g.size] = g.reshape(-1)
    return out


# ---- runs ---------------------------------------------------------------------------------------------------------------

def call(mc, batch, compact=False, want_gp=False, profile=False):
    """call_host (the result) then call_device on the same context (the fallback counts, which only the device path reports,
    and, in place, the same result again).  Returns (result, kernel names or None, fallback counts)."""
    import torch
    from torch.profiler import ProfilerActivity
    from torch.profiler import profile as prof_ctx
    from bcftools_b200 import device
    names = None
    if profile:
        with prof_ctx(activities=[ProfilerActivity.CUDA]) as prof:
            got = mc.call_host(batch, compact=compact, want_gp=want_gp)
            torch.cuda.synchronize()
        names = {e.name for e in prof.events()}
    else:
        got = mc.call_host(batch, compact=compact, want_gp=want_gp)
    if not batch.nsites:
        return got, names, None
    db = device.DeviceBatch(batch)
    dr = device.DeviceResult(db, want_gp=want_gp)
    mc.call_device(db.c_struct(), dr.c_struct(), torch.cuda.current_stream().cuda_stream)
    torch.cuda.synchronize()
    fb = mc.fallback_counts()
    if not compact:
        assert_identical(dr.to_host(), got)
    return got, names, fb


def run(params, batch, options, tab=None, compact=False, want_gp=False, profile=False):
    from bcftools_b200 import mcall
    with mcall.MCaller(params, ploidy_tab=tab, options=options) as mc:
        return call(mc, batch, compact=compact, want_gp=want_gp, profile=profile)


def assert_identical(got, ref):
    """ret, als_new and site_flags of every site, and every other output of every called site, bit for bit (QUAL included); PL
    (and GP) block by block, which also covers compacted output.  What a site that is not emitted leaves in the other arrays is
    not an output."""
    for name in ("ret", "als_new", "site_flags"):
        a, b = getattr(got, name), getattr(ref, name)
        assert (a == b).all(), (name, np.argwhere(a != b)[:5])
    called = np.where(ref.ret > 0)[0]
    for name, bits in (("als_map", np.int8), ("ac", np.int32), ("an", np.int32), ("gt", np.int32), ("gq", np.int32),
                       ("qual", np.uint32), ("diag", np.uint64)):
        a, b = getattr(got, name)[called].view(bits), getattr(ref, name)[called].view(bits)
        diff = (a != b).reshape(len(called), -1).any(1)
        if name == "gq":        # GQ of a site called REF-only from GT alone is not written (parity.compare skips it too)
            diff &= (ref.site_flags[called] & abi.SITE_REF_GT) == 0
        assert not diff.any(), (name, called[diff][:5])
    if got.pl_off_out is not None and ref.pl_off_out is not None:
        assert ((got.pl_off_out < 0) == (ref.pl_off_out < 0)).all()
    for i in called:
        if ref.site_flags[i] & abi.SITE_PL_DROPPED:      # no PL block
            continue
        assert (got.site_pl(i) == ref.site_pl(i)).all(), (i, "pl")
        if ref.gp is not None:
            assert (got.site_gp(i).view(np.uint32) == ref.site_gp(i).view(np.uint32)).all(), (i, "gp")


def against_oracle(got, expected, params, batch, bad):
    """parity.compare against every (sites, result) of oracle(); the sites with bad priors are flagged, and only they"""
    flagged = np.where(got.site_flags & SITE_BAD_PRIOR)[0].tolist()
    assert flagged == sorted(bad), (flagged, bad)
    for sites, exp in expected:
        sub = got if len(sites) == batch.nsites else restrict(got, sites, batch.subset(sites))
        st = parity.compare(sub, exp, params)
        assert st["compared"] > 0 or not len(sites), st
        assert len(st["near_ties"]) <= 0.05 * len(exp.ret) + 1, st["near_ties"]


def oracle(oracle_built, params, batch, bad, tab=None, want_gp=False):
    """[(sites, expected result)]: the compiled reference (where it is built) on the sites where it is defined, and the port on
    every site with a good prior.  The reference stops at a bad prior, PL >= 256 next to missing values is undefined in it
    (mcall.c:522), and FORMAT/GP is compared with the port only."""
    good = [i for i in range(batch.nsites) if i not in set(bad)]
    out = [(good, oracle_built.call("port", params, batch.subset(good), tab, want_gp=want_gp)[0])]
    if oracle_built.have_ref() and not want_gp:
        defined = [i for i in good if batch.site_pl(i).max(initial=0) < 256]
        out.append((defined, oracle_built.call("reference", params, batch.subset(defined), tab)[0]))
    return out


def class_count(batch, nals):
    return int((batch.nals == nals).sum()) if nals else int((batch.nals > 5).sum())


def capped_matrix(params, batch, bad, exp, rows, tab=None, want_gp=False):
    """rows: (options, max_ctas, compact, check(names)); each capped call against the oracle and the uncapped call.  A class
    without sites still has its kernels launched, so check(names) can only ask for the kernels that must have run."""
    uncapped = {}
    for options, cap, compact, check in rows:
        key = (tuple(sorted(options.items())), compact)
        if key not in uncapped:
            uncapped[key] = run(params, batch, options, tab=tab, compact=compact, want_gp=want_gp)
        got, names, fb = run(params, batch, dict(options, max_ctas=cap), tab=tab, compact=compact, want_gp=want_gp, profile=True)
        assert check(names), (options, cap, sorted(names))
        against_oracle(got, exp, params, batch, bad)
        ref, _, fb_ref = uncapped[key]
        assert_identical(got, ref)
        assert (fb == fb_ref).all(), (options, cap, fb, fb_ref)


# ---- the option ------------------------------------------------------------------------------------------------------------

def test_max_ctas_option_takes_non_negative_values():
    from bcftools_b200 import mcall
    with mcall.MCaller(abi.CallParams(64, 5)) as mc:
        for good in (0, 1, 3, 1 << 40):
            mc.set_option("max_ctas", good)
        for bad in (-1, -1 << 40):
            with pytest.raises(mcall.McallError):
                mc.set_option("max_ctas", bad)


# ---- the kernels, one by one -----------------------------------------------------------------------------------------------

@pytest.mark.parametrize("ploidy", [False, True])
def test_two_allele_warp_kernel(ploidy, oracle_built):
    S, R = 256, 240
    flag = abi.CALL_VARONLY if ploidy else 0
    batch, bad = handover_batch([S, 2, int(ploidy)], R, S, 2, 2)
    tab = ploidy_012(np.random.default_rng(5), batch, S) if ploidy else None
    params = params_for(S, 2, flag)
    exp = oracle(oracle_built, params, batch, bad, tab)
    rows = []
    for w in (1, BW_MAXWARP):
        for cap in (1, 2):
            assert class_count(batch, 2) >= MIN_RUN * w * cap
            for compact in (False, True):
                rows.append(({"warp2": w}, cap, compact, lambda n: ran(n, K_BW, "true" if ploidy else "false")))
    capped_matrix(params, batch, bad, exp, rows, tab=tab)


@pytest.mark.parametrize("flag", [0, abi.CALL_VARONLY])
def test_three_allele_warp_kernel(flag, oracle_built):
    S, R = 640, 132
    batch, bad = handover_batch([S, 3, flag], R, S, 3, 3)
    params = params_for(S, 3, flag)
    exp = oracle(oracle_built, params, batch, bad)
    assert class_count(batch, 3) >= MIN_RUN * TW_MAXWARP
    rows = [({"warp3": w}, 1, compact, lambda n: ran(n, K_W3)) for w in (1, -1) for compact in (False, True)]
    capped_matrix(params, batch, bad, exp, rows)


@pytest.mark.parametrize("S,w", [(2560, MW_MAXWARP), (256, 1)])
def test_four_allele_warp_kernel(S, w, oracle_built):
    """at 2,560 samples and eight warps the packed copies have a tail in L2"""
    import torch
    if w == MW_MAXWARP:     # the shared-memory head of a warp's copy (10 bytes a sample) is short of S even with no tables
        per_cta = torch.cuda.get_device_properties(0).shared_memory_per_multiprocessor // 2 - 1024
        assert per_cta // (w * 10) < S, per_cta
    batch, bad = handover_batch([S, 4], 72, S, 4, 4)
    params = params_for(S, 4, abi.CALL_VARONLY if w == 1 else 0)
    exp = oracle(oracle_built, params, batch, bad)
    assert class_count(batch, 4) >= MIN_RUN * w
    rows = [({"warp4": w}, 1, compact, lambda n: ran(n, K_W4, 4)) for compact in (False, True)]
    capped_matrix(params, batch, bad, exp, rows)


@pytest.mark.parametrize("S", [130, 1282, 2504])
def test_cta_multi_kernel(S, oracle_built):
    """classes 3-5 on the CTA-per-site kernel, every CTA size and ring depth: the tiles per warp are not a multiple of the ring
    depth, and the short last tile falls on different warps"""
    batch, bad = handover_batch([S, 5], 108, S, 5, 3)
    params = params_for(S, 5, abi.CALL_VARONLY if S == 1282 else 0)
    exp = oracle(oracle_built, params, batch, bad)
    for nals in (3, 4, 5):
        assert class_count(batch, nals) >= MIN_RUN * 3, nals
    rows = [({"warp3": 0, "warp4": 0, "mm_block": blk, "mm_nst": nst}, cap, (blk + nst) % 2 == 1,
             lambda n: ran(n, K_CTA) and not ran(n, K_W3) and not ran(n, K_W4))
            for blk in (64, 128, 256) for nst in (1, 2, 3, 4) for cap in (1, 3)]
    capped_matrix(params, batch, bad, exp, rows)


def tiled_instance(n, targs):
    """a tiled kernel whose template arguments (NALS, PLOIDY, BLOCK, PL type, GPOUT) contain `targs`"""
    return any(K_TILED in x and targs in x.replace(" ", "") for x in n)


def tiled_only(n):
    return ran(n, K_TILED) and not ran(n, K_BW) and not ran(n, K_CTA) and not ran(n, K_W3) and not ran(n, K_W4)


STREAM_S = 1000         # 256-sample tiles: 4 tiles per pass over a ring of 3 stages, so 2 x ntiles is not a multiple of nstage


def streaming(options):
    """tiles of 256 samples, a ring of 3 of them in every class"""
    o = dict(options, tile_bytes=1024)
    for A in range(1, 6):
        o[f"ring_bytes_{A}"] = 3 * 256 * 4 * A * (A + 1) // 2
    return o


@pytest.mark.parametrize("mode", ["resident", "streaming"])
def test_tiled_site_kernel(mode, oracle_built):
    """every class on the tiled kernel (an explicit CTA size), VARONLY: REF-only sites end early between variant sites"""
    S = 640 if mode == "resident" else STREAM_S
    batch, bad = handover_batch([S, 1, mode == "streaming"], 150, S, 5, 1)
    params = params_for(S, 5, abi.CALL_VARONLY)
    exp = oracle(oracle_built, params, batch, bad)
    for nals in range(1, 6):
        assert class_count(batch, nals) >= MIN_RUN * 2, nals
    assert ((exp[0][1].ret == 0) & (batch.nals[exp[0][0]] > 1)).sum() >= 10
    wrap = streaming if mode == "streaming" else dict
    rows = [(wrap({"block": blk}), cap, blk == 64, tiled_only) for blk in (32, 64, 128, 256) for cap in (1, 2)]
    capped_matrix(params, batch, bad, exp, rows)


@pytest.mark.parametrize("variant", ["int16", "gp", "ploidy"])
def test_tiled_site_kernel_instances(variant, oracle_built):
    S = 640
    batch, bad = handover_batch([S, 2, len(variant)], 120, S, 5, 2)
    tab = ploidy_012(np.random.default_rng(7), batch, S) if variant == "ploidy" else None
    want_gp = variant == "gp"
    params = params_for(S, 5, tags=abi.CALL_FMT_GP if want_gp else 0)
    exp = oracle(oracle_built, params, batch, bad, tab, want_gp=want_gp)
    for nals in range(2, 6):
        assert class_count(batch, nals) >= MIN_RUN * 2, nals
    if variant == "int16":
        batch = batch.to_int16()
    blocks = (64, 256) if variant == "ploidy" else (0,)
    targs = {"int16": ",short,", "gp": ",true>(", "ploidy": ",true,"}[variant]
    check = lambda n: tiled_only(n) and tiled_instance(n, targs)
    rows = [({"block": blk} if blk else {}, cap, cap == 2, check) for blk in blocks for cap in (1, 2)]
    capped_matrix(params, batch, bad, exp, rows, tab=tab, want_gp=want_gp)


def test_tiled_two_allele_streaming_above_8192_samples(oracle_built):
    S = 8194
    batch, bad = handover_batch([S, 2], 24, S, 2, 2)
    params = params_for(S, 2, abi.CALL_VARONLY)
    exp = oracle(oracle_built, params, batch, bad)
    assert class_count(batch, 2) >= MIN_RUN * 2
    rows = [({"tile_bytes": 4096, "ring_bytes": 8192}, cap, cap == 2, lambda n: tiled_instance(n, "<2,") and not ran(n, K_BW)) for cap in (1, 2)]
    capped_matrix(params, batch, bad, exp, rows)


@pytest.mark.parametrize("cap", [1, 3])
def test_general_kernel_on_fallback_lists(cap, oracle_built):
    """most sites have more than 32 listed rows: the class kernels hand them to the general kernel, whose capped grid walks
    many of them per CTA"""
    S = 640
    batch, bad = handover_batch([S, 3, 3], 96, S, 5, 3, priors=False)
    rng = np.random.default_rng(11)
    for i in range(batch.nsites):
        if i % 6 != 0 and i % 3:
            listed(rng, batch.site_pl(i), 40, "partial")
    params = params_for(S, 5, priors=False)
    exp = oracle(oracle_built, params, batch, bad)
    rows = [({}, cap, False, lambda n: ran(n, K_W3) and ran(n, K_TILED)), ({"warp3": 0, "warp4": 0}, cap, True, lambda n: ran(n, K_CTA) and ran(n, K_TILED))]
    for options, *_ in rows:
        _, _, fb = run(params, batch, options)
        for nals in (3, 4, 5):
            assert fb[nals] >= MIN_RUN * cap, (options, fb)
    capped_matrix(params, batch, bad, exp, rows)


def test_grouped_kernels(oracle_built):
    """-G: mcall_groups.cu with groups of 150 / 100 / 40 / the rest (whole-CTA and warp paths), and the two-allele grouped warp
    kernel, ploidy ids 0 / 1 / 2"""
    S = 400
    batch, bad = handover_batch([S, 6], 400, S, 5, 1)
    tab = ploidy_012(np.random.default_rng(6), batch, S)
    params = params_for(S, 5, groups=mixed_groups(S, 6))
    exp = oracle(oracle_built, params, batch, bad, tab)
    for nals in range(1, 6):
        assert class_count(batch, nals) >= MIN_RUN * 3, nals
    assert class_count(batch, 2) >= MIN_RUN * BG_WARPS
    rows = [({"bgroups": 0}, cap, False, lambda n: ran(n, K_GRP) and not ran(n, K_BGRP)) for cap in (1, 3)]
    rows.append(({"bgroups": 1}, 1, False, lambda n: ran(n, K_BGRP)))
    capped_matrix(params, batch, bad, exp, rows, tab=tab)


@pytest.mark.parametrize("grouped", [False, True])
def test_more_than_five_alleles(grouped, oracle_built):
    S = 300
    batch, bad = handover_batch([S, 8, int(grouped)], 150, S, 8, 1)
    tab = ploidy_012(np.random.default_rng(8), batch, S)
    params = params_for(S, 8, groups=mixed_groups(S, 8) if grouped else None)
    exp = oracle(oracle_built, params, batch, bad, tab)
    assert class_count(batch, 0) >= MIN_RUN
    capped_matrix(params, batch, bad, exp, [({}, 1, False, lambda n: ran(n, K_GEN))], tab=tab)


def test_literal_phase1_and_adjudication(oracle_built):
    """exact_phase1=1, and adjudicate=1 with every site a near tie (the literal kernels again, over the adjudication lists)"""
    S = 300
    batch, bad = handover_batch([S, 7], 150, S, 7, 1)
    params = params_for(S, 7)
    exp = oracle(oracle_built, params, batch, bad)
    for nals in range(1, 6):
        assert class_count(batch, nals) >= MIN_RUN, nals
    capped_matrix(params, batch, bad, exp, [({"exact_phase1": 1}, 1, False, lambda n: ran(n, K_TILED) and ran(n, K_GEN) and not ran(n, K_BW))])
    pt = params_for(S, 7, tie_eps=1e30)
    capped_matrix(pt, batch, bad, exp, [({"adjudicate": 1}, 1, True, lambda n: ran(n, K_TILED) and ran(n, K_GEN))])


# ---- the real dynamic claim, every warp contending ------------------------------------------------------------------------

@pytest.mark.parametrize("groups", [None, 5])
def test_replicated_sites_at_full_occupancy(groups, oracle_built):
    """C3 sites, 300 distinct two-allele ones and 250 of each of 3, 4 and 5 alleles, replicated to 21,000 and called in one
    call_device: every copy bit-identical to the first, and the first as the oracle calls it"""
    import torch
    from bcftools_b200 import device, mcall
    params, full, tab = synth.make_batch("C3", 9000, with_groups=groups or 0)
    pick = [np.where(full.nals == A)[0][:n] for A, n in ((2, 300), (3, 250), (4, 250), (5, 250))]
    assert all(len(p) == n for p, n in zip(pick, (300, 250, 250, 250)))
    batch = full.subset(np.sort(np.concatenate(pick)))
    r = 20
    db = device.DeviceBatch(batch, replicate=r)
    dr = device.DeviceResult(db)
    with mcall.MCaller(params, ploidy_tab=tab) as mc:
        mc.call_device(db.c_struct(), dr.c_struct(), torch.cuda.current_stream().cuda_stream)
        torch.cuda.synchronize()
    assert db.nsites >= 20000
    bits = {1: torch.int8, 4: torch.int32, 8: torch.int64}
    for name, t in dr.t.items():        # in place: copy k of every array (PL included) is its k-th slice
        if t is None:
            continue
        v = t.view(bits[t.element_size()]).view(r, -1)
        same = (v == v[0]).all(1)
        assert bool(same.all()), (name, torch.where(~same)[0][:5].tolist())
    exp, _ = oracle_built.call(ORACLE(oracle_built), params, batch, tab)
    st = parity.compare(dr.to_host(), exp, params)
    assert st["compared"] > 0 and not st["near_ties"], st


# ---- one context over many calls ------------------------------------------------------------------------------------------

@pytest.mark.parametrize("grouped", [False, True])
def test_one_context_over_many_calls(grouped, oracle_built):
    """a small batch, one several times larger (the lists and the scratch grow), one with classes absent, one site, an empty
    batch and the large one again, with max_ctas, warp3 / warp4 and adjudicate changed between calls"""
    from bcftools_b200 import mcall
    S, maxA = 300, 7
    params = params_for(S, maxA, groups=mixed_groups(S, 12) if grouped else None)
    small, bad_s = handover_batch([S, 12, 1], 40, S, maxA, 1)
    large, bad_l = handover_batch([S, 12, 2], 300, S, maxA, 1)
    keep = [i for i in range(large.nsites) if large.nals[i] in (2, 4)]
    absent = large.subset(keep)
    bad_a = [k for k, i in enumerate(keep) if i in set(bad_l)]
    one = small.subset([1])
    empty = abi.HostBatch(S, maxA, np.zeros(0, np.uint8), pl_blocks=[], qs=np.zeros((0, maxA), np.float32),
                          ad_blocks=[] if grouped else None)
    steps = [(small, bad_s, {"max_ctas": 1}), (large, bad_l, {"max_ctas": 3, "warp3": 0, "warp4": 0}),
             (absent, bad_a, {"max_ctas": 0, "warp3": -1, "warp4": -1, "adjudicate": 1}), (one, [], {"max_ctas": 2, "adjudicate": 0}),
             (empty, [], {}), (large, bad_l, {"max_ctas": 0})]
    with mcall.MCaller(params) as mc:
        for k, (batch, bad, options) in enumerate(steps):
            for key, v in options.items():
                mc.set_option(key, v)
            got, _, _ = call(mc, batch, compact=k % 2 == 1)
            if batch.nsites:
                against_oracle(got, oracle(oracle_built, params, batch, bad), params, batch, bad)


def same_shape_other_batch(batch, seed):
    """the same sites' shape (allele counts, sample count) with other PLs, QS and AD: rows permuted, QS shuffled"""
    rng = np.random.default_rng(seed)
    b = batch.subset(range(batch.nsites))
    for i in range(b.nsites):
        p = rng.permutation(b.nsmpl)
        b.site_pl(i)[...] = b.site_pl(i)[p]
        if b.ad is not None:
            b.site_ad(i)[...] = b.site_ad(i)[p]
    b.qs = b.qs[rng.permutation(b.nsites)]
    b.qs[b.nals[:, None] <= np.arange(b.max_nals)[None, :]] = 0
    return b


@pytest.mark.parametrize("grouped", [False, True])
def test_two_calls_into_one_poisoned_result(grouped, oracle_built):
    """every result buffer starts as 0x5A bytes: an output the kernels never write shows; the second call, on other sites of the
    same shape, overwrites everything the first wrote"""
    import torch
    from bcftools_b200 import device, mcall
    S = 300
    params = params_for(S, 7, groups=mixed_groups(S, 13) if grouped else None, priors=False)
    b1, _ = handover_batch([S, 13, int(grouped)], 120, S, 7, 1, priors=False)
    b2 = same_shape_other_batch(b1, 14)
    db1, db2 = device.DeviceBatch(b1), device.DeviceBatch(b2)
    dr = device.DeviceResult(db1)
    for t in dr.t.values():
        if t is not None:
            t.view(torch.uint8).fill_(0x5A)
    with mcall.MCaller(params) as mc:
        for db, b in ((db1, b1), (db2, b2)):
            mc.call_device(db.c_struct(), dr.c_struct(), torch.cuda.current_stream().cuda_stream)
            torch.cuda.synchronize()
            dr.dbatch = db
            against_oracle(dr.to_host(), oracle(oracle_built, params, b, []), params, b, [])
