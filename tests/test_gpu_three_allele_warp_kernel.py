"""The warp-per-site kernel of the 3-allele class (mcall_triallelic.cu): against the oracle, against the CTA-per-site kernel
of mcall_multi.cu (option warp3=0) on the same sites, and on the bench workload against the compiled reference."""
import numpy as np
import pytest

from bcftools_b200 import abi, synth
from tests import parity

pytestmark = pytest.mark.gpu

KERNEL = "mcall_triallelic_warp_kernel"


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


def ran_warp_kernel(names):
    return any(KERNEL in n for n in names)


def class3_fallbacks(params, batch, options):
    """3-allele sites that the specialised kernel of one call_device handed back to the general kernel"""
    import torch
    from bcftools_b200 import device, mcall
    db = device.DeviceBatch(batch)
    dr = device.DeviceResult(db)
    with mcall.MCaller(params, options=options) as mc:
        mc.call_device(db.c_struct(), dr.c_struct(), torch.cuda.current_stream().cuda_stream)
        return int(mc.fallback_counts()[3])


@pytest.fixture(scope="module")
def largest_nsmpl():
    """Largest (even) sample count for which the launcher picks the warp kernel: its packed copies must leave room for
    12 resident warps per SM, which depends on the device's shared memory."""
    def takes(S):
        rng = np.random.default_rng(S)
        batch = parity.random_batch(rng, 4, S, 3, minA=3, miss=False)
        return ran_warp_kernel(run(abi.CallParams(S, 3, output_tags=abi.CALL_FMT_GQ), batch, {})[1])
    lo, hi = 2560, 10240                # even counts: lo takes it, hi does not
    assert takes(lo) and not takes(hi)
    while hi - lo > 2:
        mid = (lo + hi) // 4 * 2
        lo, hi = (mid, hi) if takes(mid) else (lo, mid)
    return lo


def adversarial_batch(S, flag):
    """Three-allele sites of the shapes test_multi_allelic_kernel uses: missing and partially missing rows (more than the
    32-entry list holds on most random sites of >= 1,000 samples), zero QS, unseen alleles, PL >= 256, clean sites and
    mpileup-shaped ones, so that REF-only, pair, triple and set-without-REF outcomes all occur.  Returns the batch and the
    indices of its ordinary sites (clean and mpileup-shaped: no special values, every sample on the fast path)."""
    rng = np.random.default_rng([S, flag, 31])
    R = 60 if S > 1500 else 120
    batch = parity.random_batch(rng, R, S, 3, minA=3, pl_max=256)
    for i in range(0, R, 5):            # PL >= 256 on some sites
        blk = batch.site_pl(i)
        blk[rng.integers(0, S, 3), rng.integers(0, blk.shape[1], 3)] = 300
    for i in range(3, R, 4):            # a handful of special rows per site: the list stays below its 32 entries
        blk = batch.site_pl(i)
        sp = (blk < 0).any(1)
        keep = rng.choice(np.where(sp)[0], size=min(int(sp.sum()), 7), replace=False) if sp.any() else []
        fix = sp.copy(); fix[keep] = False
        blk[fix] = rng.integers(0, 256, (int(fix.sum()), blk.shape[1]))
        blk[fix, 0] = 0
    for i in range(1, R, 4):            # clean sites: every sample on the fast path, every allele live
        blk = batch.site_pl(i)
        blk[...] = rng.integers(0, 256, blk.shape)
        blk[np.arange(S), rng.integers(0, blk.shape[1], S)] = 0
        batch.qs[i, :3] = (1 + rng.random(3) * 10).astype(np.float32)
        batch.unseen[i] = 0
    mpileup = range(2, R, 9)
    for n, i in enumerate(mpileup):     # mpileup-shaped sites: most samples REF/REF, so that the triple, the pair {REF,ALT1} and REF alone win
        blk = batch.site_pl(i)
        truth = rng.choice(3, size=(S, 2), p=np.array([(0.8, 0.1, 0.1), (0.8, 0.2, 0.0), (1.0, 0.0, 0.0)][n % 3]))
        k = 0
        for x in range(3):
            for y in range(x + 1):
                m = ((truth[:, 0] == x) & (truth[:, 1] == y)) | ((truth[:, 0] == y) & (truth[:, 1] == x))
                one = (truth == x).any(1) | (truth == y).any(1)
                blk[:, k] = np.where(m, 0, np.where(one, 20 + rng.integers(0, 9, S), 200 + rng.integers(0, 50, S)))
                k += 1
        batch.qs[i, :3] = np.array([((truth == x).sum()) for x in range(3)], np.float32)
        batch.unseen[i] = 0
    return batch, sorted(set(range(1, R, 4)) | set(mpileup))


def assert_same_calls(got, ref, params):
    """GT, GQ, trimmed PL, AC, AN, ret, als_new, als_map, site flags (near ties included) bit-identical; QUAL within 1e-6."""
    for name in ("ret", "als_new", "als_map", "ac", "an", "site_flags", "gt", "gq"):
        a, b = getattr(got, name), getattr(ref, name)
        assert (a == b).all(), (name, np.argwhere(a != b)[:5])
    for i in range(len(ref.ret)):
        if ref.ret[i] > 0 and not (ref.site_flags[i] & abi.SITE_PL_DROPPED):
            assert (got.site_pl(i) == ref.site_pl(i)).all(), (i, "pl")
    a, b = got.qual.astype(np.float64), ref.qual.astype(np.float64)
    same = (got.qual.view(np.uint32) == ref.qual.view(np.uint32)) | (np.isnan(a) & np.isnan(b))
    rel = np.where(same, 0.0, np.abs(a - b) / np.maximum(np.abs(b), 1e-30))
    assert rel.max() <= 1e-6, (int(rel.argmax()), rel.max())


@pytest.mark.parametrize("flag", [0, abi.CALL_VARONLY])
@pytest.mark.parametrize("S", [128, 130, 300, 1000, 2504, 2560, "largest", "largest+2"])
def test_three_allele_warp_kernel(S, flag, oracle_built, request):
    if isinstance(S, str):
        S = request.getfixturevalue("largest_nsmpl") + (2 if S.endswith("+2") else 0)
    fits = S <= request.getfixturevalue("largest_nsmpl")
    batch, ordinary = adversarial_batch(S, flag)
    params = abi.CallParams(S, 3, flag=flag, output_tags=abi.CALL_FMT_GQ)
    exp, _ = oracle_built.call("port", params, batch, None)     # PL >= 256 next to missing values: undefined in the reference (mcall.c:522)
    # the outcomes phase 2 has straight-line code for are all in the batch: REF only (flag 0: VARONLY drops those sites), a pair, the triple
    nsel = np.array([bin(int(x)).count("1") for x in exp.als_new])
    called = exp.ret > 0
    assert (called & (nsel == 2)).any() and (called & (nsel == 3)).any(), (exp.ret, nsel)
    assert flag or (called & (nsel == 1)).any(), (exp.ret, nsel)
    # the specialised kernels decide the ordinary sites themselves, and both hand back the same sites
    fb = class3_fallbacks(params, batch, {})
    assert fb == class3_fallbacks(params, batch, {"warp3": 0}), fb
    sub = batch.subset(ordinary)
    fb_ordinary = class3_fallbacks(params, sub, {})
    assert fb_ordinary <= len(ordinary) // 4 and fb_ordinary == class3_fallbacks(params, sub, {"warp3": 0}), (fb_ordinary, len(ordinary))
    for compact in (False, True):
        got, names = run(params, batch, {}, compact=compact)
        assert ran_warp_kernel(names) == fits, (S, sorted(names))
        st = parity.compare(got, exp, params)
        assert st["compared"] > 0, st
        cta, names = run(params, batch, {"warp3": 0}, compact=compact)
        assert not ran_warp_kernel(names)
        assert_same_calls(got, cta, params)


def test_three_allele_warp_kernel_on_the_bench_workload(oracle_built):
    """2,048 sites of the C3 mix against the compiled reference with the default kernels: the 3-allele class runs the
    warp kernel, no near ties."""
    params, batch, tab = synth.make_batch("C3", 2048)
    exp, _ = oracle_built.call("reference" if oracle_built.have_ref() else "port", params, batch, tab)
    got, names = run(params, batch, {}, compact=True, tab=tab)
    assert ran_warp_kernel(names)
    st = parity.compare(got, exp, params)
    assert st["compared"] > 0 and not st["near_ties"], st
