"""The warp-per-site kernel of the 4-allele class (mcall_multi_warp.cu): against the oracle, against the CTA-per-site kernel of
mcall_multi.cu (option warp4=0) on the same sites, with listed rows in the shared-memory head of the packed copy, in its
L2-resident tail and at the boundary, and with in-call adjudication of near ties.  The 5-allele class stays on the CTA kernel."""
import numpy as np
import pytest

from bcftools_b200 import abi, synth
from tests import parity
from tests.test_gpu_three_allele_warp_kernel import assert_same_calls

pytestmark = pytest.mark.gpu

KERNEL = "mcall_multi_warp_kernel"


def run(params, batch, options, compact=False, tab=None):
    """call_host with the given options; returns (result, names of the CUDA kernels that ran)"""
    import torch
    from torch.profiler import ProfilerActivity, profile
    from bcftools_b200 import mcall
    with mcall.MCaller(params, ploidy_tab=tab, options=options) as mc:
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            got = mc.call_host(batch, compact=compact)
            torch.cuda.synchronize()
    return got, {e.name for e in prof.events()}


def ran_warp_kernel(names, nals):
    return any(KERNEL in n and f"<{nals}>" in n.replace(" ", "") for n in names)


OFF = {"warp4": 0}


def fallbacks(params, batch, options, nals):
    """sites of the class that the specialised kernel of one call_device handed back to the general kernel"""
    import torch
    from bcftools_b200 import device, mcall
    db = device.DeviceBatch(batch)
    dr = device.DeviceResult(db)
    with mcall.MCaller(params, options=options) as mc:
        mc.call_device(db.c_struct(), dr.c_struct(), torch.cuda.current_stream().cuda_stream)
        return int(mc.fallback_counts()[nals])


@pytest.fixture(scope="module")
def largest_nsmpl():
    """Largest (even) sample count for which the launcher picks the warp kernel: the tails of the packed copies that do not
    fit shared memory must stay within a share of L2, which depends on the device."""
    def takes(S, nals):
        rng = np.random.default_rng(S)
        batch = parity.random_batch(rng, 4, S, nals, minA=nals, miss=False)
        return ran_warp_kernel(run(abi.CallParams(S, nals, output_tags=abi.CALL_FMT_GQ), batch, {})[1], nals)
    lo, hi = 2504, 10240                # even counts: lo takes it, hi does not
    assert takes(lo, 4) and not takes(hi, 4)
    while hi - lo > 2:
        mid = (lo + hi) // 4 * 2
        lo, hi = (mid, hi) if takes(mid, 4) else (lo, mid)
    return lo


def adversarial_batch(S, nals, flag):
    """Sites of the class with missing and partially missing rows, zero QS, unseen alleles, PL >= 256, clean sites and
    mpileup-shaped ones, so that REF-only, pair, triple and set-without-REF outcomes all occur.  Returns the batch, the
    indices of its ordinary sites (mpileup-shaped with REF in the best set: no special values, every sample on the fast path)
    and those of the mpileup-shaped sites whose best allele set leaves REF out."""
    rng = np.random.default_rng([S, nals, flag, 41])
    G = nals * (nals + 1) // 2
    R = 60 if S > 1500 else 120
    batch = parity.random_batch(rng, R, S, nals, minA=nals, pl_max=256)
    for i in range(0, R, 5):            # PL >= 256 on some sites
        blk = batch.site_pl(i)
        blk[rng.integers(0, S, 3), rng.integers(0, G, 3)] = 300
    for i in range(3, R, 4):            # a handful of special rows per site: the list stays below its 32 entries
        blk = batch.site_pl(i)
        sp = (blk < 0).any(1)
        keep = rng.choice(np.where(sp)[0], size=min(int(sp.sum()), 7), replace=False) if sp.any() else []
        fix = sp.copy(); fix[keep] = False
        blk[fix] = rng.integers(0, 256, (int(fix.sum()), G))
        blk[fix, 0] = 0
    for i in range(1, R, 4):            # clean sites: every sample on the fast path, every allele live
        blk = batch.site_pl(i)
        blk[...] = rng.integers(0, 256, blk.shape)
        blk[np.arange(S), rng.integers(0, G, S)] = 0
        batch.qs[i, :nals] = (1 + rng.random(nals) * 10).astype(np.float32)
        batch.unseen[i] = 0
    mpileup = range(2, R, 7)
    # mpileup-shaped sites: most samples REF/REF, so that a triple, a pair {REF,ALT1}, REF alone and a set without REF win
    probs = [np.r_[0.8, 0.1, 0.1, np.zeros(nals - 3)], np.r_[0.8, 0.2, np.zeros(nals - 2)], np.r_[1.0, np.zeros(nals - 1)],
             np.r_[0.0, 0.0, 0.5, 0.5, np.zeros(nals - 4)]]
    for n, i in enumerate(mpileup):
        blk = batch.site_pl(i)
        truth = rng.choice(nals, size=(S, 2), p=probs[n % 4])
        k = 0
        for x in range(nals):
            for y in range(x + 1):
                m = ((truth[:, 0] == x) & (truth[:, 1] == y)) | ((truth[:, 0] == y) & (truth[:, 1] == x))
                one = (truth == x).any(1) | (truth == y).any(1)
                blk[:, k] = np.where(m, 0, np.where(one, 20 + rng.integers(0, 9, S), 200 + rng.integers(0, 50, S)))
                k += 1
        batch.qs[i, :nals] = np.array([(truth == x).sum() for x in range(nals)], np.float32)
        batch.unseen[i] = 0
    noref = list(mpileup)[3::4]
    return batch, sorted(set(mpileup) - set(noref)), noref


def boundary_batch(S, nals):
    """mpileup-shaped sites (the triple {REF,ALT1,ALT2} wins) with a few listed rows each: a partially missing row (filled,
    has data), a vector_end row and a row of missing values (no data) at samples 64k-1, 64k and 64k+1 for every k, plus
    one near the start and one near the end.  Whatever the head of the packed copy is (a multiple of 64 samples), some
    site has its listed rows on both sides of it."""
    rng = np.random.default_rng([S, nals, 7])
    G = nals * (nals + 1) // 2
    ks = list(range(1, (S - 2) // 64 + 1))
    batch = parity.random_batch(rng, len(ks), S, nals, minA=nals, miss=False, zq=False)
    for i, k in enumerate(ks):
        blk = batch.site_pl(i)
        truth = rng.choice(nals, size=(S, 2), p=np.r_[0.8, 0.1, 0.1, np.zeros(nals - 3)])
        j = 0
        for x in range(nals):
            for y in range(x + 1):
                m = ((truth[:, 0] == x) & (truth[:, 1] == y)) | ((truth[:, 0] == y) & (truth[:, 1] == x))
                one = (truth == x).any(1) | (truth == y).any(1)
                blk[:, j] = np.where(m, 0, np.where(one, 20 + rng.integers(0, 9, S), 200 + rng.integers(0, 50, S)))
                j += 1
        batch.qs[i, :nals] = np.array([(truth == x).sum() for x in range(nals)], np.float32)
        batch.unseen[i] = 0
        for s in (64 * k - 1, 3):
            blk[s, rng.integers(1, G)] = abi.INT32_MISSING
        for s in (64 * k, S - 2):
            blk[s] = abi.INT32_VECTOR_END
            blk[s, 0] = abi.INT32_MISSING
        if 64 * k + 1 < S:
            blk[64 * k + 1] = abi.INT32_MISSING
    return batch


@pytest.mark.parametrize("flag", [0, abi.CALL_VARONLY])
@pytest.mark.parametrize("S", [128, 130, 300, 1000, 2504, 2560, "largest", "largest+2"])
def test_four_allele_warp_kernel(S, flag, oracle_built, request):
    nals = 4
    if isinstance(S, str):
        S = request.getfixturevalue("largest_nsmpl") + (2 if S.endswith("+2") else 0)
    fits = S <= request.getfixturevalue("largest_nsmpl")
    batch, ordinary, noref = adversarial_batch(S, nals, flag)
    params = abi.CallParams(S, nals, flag=flag, output_tags=abi.CALL_FMT_GQ)
    exp, _ = oracle_built.call("port", params, batch, None)     # PL >= 256 next to missing values: undefined in the reference (mcall.c:522)
    # the outcomes phase 2 has straight-line code for are all in the batch (flag 0: REF only too), and a set without REF
    nsel = np.array([bin(int(x)).count("1") for x in exp.als_new])
    called = exp.ret > 0
    assert (called & (nsel == 2)).any() and (called & (nsel == 3)).any(), (exp.ret, nsel)
    assert flag or (called & (nsel == 1)).any(), (exp.ret, nsel)
    # the specialised kernels decide the ordinary sites themselves, and both hand back the same sites
    fb = fallbacks(params, batch, {}, nals)
    assert fb == fallbacks(params, batch, OFF, nals), fb
    sub = batch.subset(ordinary)
    fb_ordinary = fallbacks(params, sub, {}, nals)
    assert fb_ordinary <= len(ordinary) // 4 and fb_ordinary == fallbacks(params, sub, OFF, nals), (fb_ordinary, len(ordinary))
    # a best set without REF has no straight-line code: both kernels hand those sites back (random clean sites of 4-5 alleles
    # often end that way too, so only the mpileup-shaped sites count as ordinary)
    assert fallbacks(params, batch.subset(noref), {}, nals) == len(noref) == fallbacks(params, batch.subset(noref), OFF, nals)
    for compact in (False, True):
        got, names = run(params, batch, {}, compact=compact)
        assert ran_warp_kernel(names, nals) == fits, (S, sorted(names))
        st = parity.compare(got, exp, params)
        assert st["compared"] > 0, st
        cta, names = run(params, batch, OFF, compact=compact)
        assert not ran_warp_kernel(names, nals)
        assert_same_calls(got, cta, params)


@pytest.mark.parametrize("S", [2504, 2560])
def test_listed_rows_in_head_tail_and_boundary(S, oracle_built):
    """the sites stay on the warp kernel (almost no fallback), results as the oracle's and the CTA kernel's"""
    nals = 4
    batch = boundary_batch(S, nals)
    params = abi.CallParams(S, nals, output_tags=abi.CALL_FMT_GQ)
    exp, _ = oracle_built.call("port", params, batch, None)
    fb = fallbacks(params, batch, {}, nals)
    assert fb <= batch.nsites // 4 and fb == fallbacks(params, batch, OFF, nals), fb
    for compact in (False, True):
        got, names = run(params, batch, {}, compact=compact)
        assert ran_warp_kernel(names, nals), sorted(names)
        st = parity.compare(got, exp, params)
        assert st["compared"] > 0, st
        cta, _ = run(params, batch, OFF, compact=compact)
        assert_same_calls(got, cta, params)


def test_adjudication_with_the_warp_kernel(oracle_built):
    """adjudicate=1 with every site a near tie, compacted output: each flagged site reserves its full-G block in the warp
    kernel's finalisation and is evaluated again in place"""
    S, nals = 2504, 4
    rng = np.random.default_rng([nals, 99])
    batch = parity.random_batch(rng, 24, S, nals, minA=nals)
    params = abi.CallParams(S, nals, output_tags=abi.CALL_FMT_GQ, tie_eps=1e30)
    exp, _ = oracle_built.call("reference" if oracle_built.have_ref() else "port", params, batch, None)
    got, names = run(params, batch, {"adjudicate": 1}, compact=True)
    assert ran_warp_kernel(names, nals), sorted(names)
    st = parity.compare(got, exp, params)
    assert st["compared"] > 0 and not st["near_ties"], st
    called = got.ret > 0
    adj = (got.site_flags[called] & abi.SITE_ADJUDICATED) != 0
    assert adj.mean() > 0.3, adj.mean()


def test_warp4_option_is_validated():
    from bcftools_b200 import mcall
    with mcall.MCaller(abi.CallParams(130, 5)) as mc:
        for v in (-1, 0, 1, 8):
            mc.set_option("warp4", v)
        for v in (-2, 9):
            with pytest.raises(Exception):
                mc.set_option("warp4", v)


def test_four_allele_warp_kernel_on_the_bench_workload(oracle_built):
    """2,048 sites of the C3 mix against the compiled reference with the default kernels: the 4-allele class runs the warp
    kernel, the 5-allele class the CTA kernel, no near ties."""
    params, batch, tab = synth.make_batch("C3", 2048)
    exp, _ = oracle_built.call("reference" if oracle_built.have_ref() else "port", params, batch, tab)
    got, names = run(params, batch, {}, compact=True, tab=tab)
    assert ran_warp_kernel(names, 4) and not ran_warp_kernel(names, 5), sorted(names)
    st = parity.compare(got, exp, params)
    assert st["compared"] > 0 and not st["near_ties"], st
