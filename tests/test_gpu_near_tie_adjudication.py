"""In-call near-tie adjudication (mcb_set_option "adjudicate"): the sites of a call that come back with MCB_SITE_NEAR_TIE are
evaluated a second time on the device with the literal phase 1, in every calling mode.  With tie_eps = 1e30 every site that
has a runner-up set is flagged, so the whole batch goes through the literal path of its mode and must give the reference's
calls: pooled (general kernel, int32 and int16 PLs), grouped (mcall_groups.cu) and 6..32 alleles (mcall_generic.cu)."""
import numpy as np
import pytest

from bcftools_b200 import abi
from tests import parity

pytestmark = pytest.mark.gpu

ALL = 1e30          # tie_eps: every site with a runner-up set is a near tie


def oracle_kind(pyoracle):
    return "reference" if pyoracle.have_ref() else "port"


def groups_of(S, mode):
    if not mode:
        return None
    if mode == "-":                 # -G -: one group per sample
        return [[s] for s in range(S)]
    return [list(range(k, S, mode)) for k in range(mode)]


def mixed_ploidy(rng, batch, S):
    tab = np.full((3, S), 2, np.uint8)
    tab[1, ::2] = 1
    tab[2, ::3] = 1
    tab[2, 1::5] = 0
    batch.ploidy_id = rng.integers(0, 3, batch.nsites).astype(np.uint16)
    return tab


def check_flags(got):
    """every adjudicated site carries NEAR_TIE and ADJUDICATED, and no other site carries either"""
    called = got.ret > 0
    tie = (got.site_flags[called] & abi.SITE_NEAR_TIE) != 0
    adj = (got.site_flags[called] & abi.SITE_ADJUDICATED) != 0
    assert (tie == adj).all()
    return adj


def run(params, batch, tab, options, compact=False, typed=False, want_gp=False):
    from bcftools_b200 import mcall
    with mcall.MCaller(params, ploidy_tab=tab, options=options) as mc:
        got = mc.call_host(batch.to_int16() if typed else batch, compact=compact, typed=typed, want_gp=want_gp)
    return got.widen() if typed else got


# name: (S, minA, maxA, groups, flag, tags, ploidy, typed, compact, options)
MODES = {
    "pooled":          (37, 1, 5, None, 0, abi.CALL_FMT_GQ, False, False, False, {}),
    "pooled-2504":     (2504, 2, 5, None, 0, abi.CALL_FMT_GQ, False, False, False, {}),
    "int16":           (300, 1, 5, None, 0, abi.CALL_FMT_GQ, False, True, False, {}),
    "int16-compact":   (130, 1, 5, None, 0, abi.CALL_FMT_GQ, True, True, True, {"slab_bytes": 1 << 16}),
    "ploidy":          (40, 1, 5, None, 0, abi.CALL_FMT_GQ, True, False, False, {}),
    "gq-gp":           (33, 1, 5, None, 0, abi.CALL_FMT_GQ | abi.CALL_FMT_GP, True, False, False, {}),
    "varonly":         (64, 1, 5, None, abi.CALL_VARONLY, abi.CALL_FMT_GQ, False, False, False, {}),
    "keepalt":         (64, 1, 5, None, abi.CALL_KEEPALT, abi.CALL_FMT_GQ, False, False, False, {}),
    "compact":         (300, 1, 5, None, abi.CALL_VARONLY, abi.CALL_FMT_GQ, True, False, True, {"slab_bytes": 1 << 17}),
    "groups2-biallelic": (128, 2, 2, 2, 0, abi.CALL_FMT_GQ, False, False, False, {}),
    "groups5-biallelic": (1000, 2, 2, 5, abi.CALL_VARONLY, abi.CALL_FMT_GQ, True, False, True, {"slab_bytes": 1 << 20}),
    "groups26-biallelic": (260, 2, 2, 26, 0, abi.CALL_FMT_GQ, False, False, False, {}),
    "groups-each-biallelic": (7, 2, 2, "-", 0, abi.CALL_FMT_GQ, False, False, False, {}),
    "groups2-multi":   (90, 3, 5, 2, 0, abi.CALL_FMT_GQ, True, False, False, {}),
    "groups5-multi":   (2504, 3, 5, 5, 0, abi.CALL_FMT_GQ, False, False, True, {}),
    "groups26-multi":  (260, 3, 5, 26, abi.CALL_KEEPALT, abi.CALL_FMT_GQ, False, False, False, {}),
    "groups-each-multi": (9, 3, 5, "-", 0, abi.CALL_FMT_GQ, False, False, False, {}),
    "alleles6-32":     (12, 1, 32, None, 0, abi.CALL_FMT_GQ, False, False, False, {}),
    "alleles6-9-compact": (150, 6, 9, None, abi.CALL_VARONLY, abi.CALL_FMT_GQ, True, False, True, {"slab_bytes": 1 << 18}),
    "alleles6-9-groups": (25, 6, 9, 3, 0, abi.CALL_FMT_GQ, True, False, False, {}),
}


@pytest.mark.parametrize("mode", list(MODES))
def test_every_mode_through_the_literal_path(mode, oracle_built):
    S, minA, maxA, g, flag, tags, ploidy, typed, compact, opts = MODES[mode]
    rng = np.random.default_rng([S, minA, maxA, flag, 77])
    R = 24 if S >= 1000 else (40 if maxA > 16 else 90)
    gp = bool(tags & abi.CALL_FMT_GP)
    batch = parity.random_batch(rng, R, S, maxA, minA=minA, zq=not gp)
    tab = mixed_ploidy(rng, batch, S) if ploidy else None
    params = abi.CallParams(S, maxA, flag=flag, output_tags=tags, groups=groups_of(S, g), tie_eps=ALL)
    kind = "port" if gp else oracle_kind(oracle_built)          # GP: assert(max) in mcall.c:881
    exp, _ = oracle_built.call(kind, params, batch, tab, want_gp=gp)
    got = run(params, batch, tab, dict(opts, adjudicate=1), compact=compact, typed=typed, want_gp=gp)
    st = parity.compare(got, exp, params)
    assert st["compared"] > 0 and not st["near_ties"], st
    adj = check_flags(got)
    assert adj.mean() > 0.3, adj.mean()


def test_exact_phase1_with_groups(oracle_built):
    """exact_phase1 = 1 with -G groups: every site through the literal phase A (formerly refused with MCB_EINVAL)."""
    S = 150
    rng = np.random.default_rng(515)
    batch = parity.random_batch(rng, 90, S, 5)
    tab = mixed_ploidy(rng, batch, S)
    params = abi.CallParams(S, 5, flag=abi.CALL_VARONLY, output_tags=abi.CALL_FMT_GQ, groups=groups_of(S, 5))
    exp, _ = oracle_built.call(oracle_kind(oracle_built), params, batch, tab)
    got = run(params, batch, tab, {"exact_phase1": 1})
    st = parity.compare(got, exp, params)
    assert st["compared"] > 0 and not st["near_ties"], st


def subset(batch, idx):
    return abi.HostBatch(batch.nsmpl, batch.max_nals, batch.nals[idx], pl_blocks=[batch.site_pl(i) for i in idx],
                         unseen=batch.unseen[idx], qs=batch.qs[idx],
                         ploidy_id=None if batch.ploidy_id is None else batch.ploidy_id[idx])


@pytest.mark.parametrize("S", [40, 2504])
def test_device_adjudication_equals_a_second_exact_call(S):
    """Pooled int32 PLs, up to 5 alleles: the in-call second evaluation gives bit for bit what a second call with
    exact_phase1 = 1 on the flagged sites gives (the earlier host-side re-submission), QUAL included."""
    rng = np.random.default_rng([S, 4])
    batch = parity.random_batch(rng, 60 if S > 1000 else 200, S, 5)
    tab = mixed_ploidy(rng, batch, S)
    probe = run(abi.CallParams(S, 5, output_tags=abi.CALL_FMT_GQ), batch, tab, {})
    gaps = np.sort(probe.diag[:, 3][np.isfinite(probe.diag[:, 3])])
    params = abi.CallParams(S, 5, output_tags=abi.CALL_FMT_GQ, tie_eps=float(gaps[len(gaps) // 3]))    # about a third flagged
    plain = run(params, batch, tab, {})
    flagged = np.where(plain.site_flags & abi.SITE_NEAR_TIE)[0]
    assert 0 < len(flagged) < batch.nsites
    got = run(params, batch, tab, {"adjudicate": 1})
    again = run(params, subset(batch, flagged), tab, {"exact_phase1": 1})
    other = np.setdiff1d(np.arange(batch.nsites), flagged)
    for name in ("ret", "als_new", "an", "site_flags"):
        assert (getattr(got, name)[other] == getattr(plain, name)[other]).all(), name
    assert (got.qual[other].view(np.uint32) == plain.qual[other].view(np.uint32)).all()
    mask = ~np.uint32(abi.SITE_NEAR_TIE | abi.SITE_ADJUDICATED)
    assert (got.site_flags[flagged] & abi.SITE_ADJUDICATED).all()
    assert ((got.site_flags[flagged] & mask) == (again.site_flags & mask)).all()
    for k, i in enumerate(flagged):
        assert got.ret[i] == again.ret[k]
        if again.ret[k] <= 0:
            continue
        assert got.als_new[i] == again.als_new[k] and got.an[i] == again.an[k]
        assert got.qual[i:i + 1].view(np.uint32)[0] == again.qual[k:k + 1].view(np.uint32)[0], (i, got.qual[i], again.qual[k])
        assert (got.als_map[i] == again.als_map[k]).all() and (got.ac[i] == again.ac[k]).all()
        assert (got.gt[i] == again.gt[k]).all() and (got.gq[i] == again.gq[k]).all()
        if not (again.site_flags[k] & abi.SITE_PL_DROPPED):
            assert (parity.mask_after_end(got.site_pl(i)) == parity.mask_after_end(again.site_pl(k))).all()


def test_exact_ties_pick_the_first_strict_maximum(oracle_built):
    """Two ALT alleles with identical PL columns and QS: the single-allele sets {A} and {B} tie exactly.  Flagged at the
    default tie_eps, adjudicated, and the reference's first strict maximum in enumeration order ({A}) is kept."""
    S, R = 60, 40
    rng = np.random.default_rng(90210)
    blocks, qs = [], np.zeros((R, 5), np.float32)
    for i in range(R):
        pl = np.zeros((S, 6), np.int32)            # genotypes 0/0 0/1 1/1 0/2 1/2 2/2; A/A and B/B most likely
        pl[:, 0] = rng.integers(60, 200, S)
        pl[:, 1] = pl[:, 3] = rng.integers(20, 60, S)
        pl[:, 2] = pl[:, 5] = rng.integers(0, 4, S)
        pl[:, 4] = rng.integers(10, 60, S)
        blocks.append(pl)
        qs[i, :3] = [rng.random() * 5, 3.0, 3.0]
    batch = abi.HostBatch(S, 5, np.full(R, 3, np.uint8), pl_blocks=blocks, qs=qs)
    params = abi.CallParams(S, 5, output_tags=abi.CALL_FMT_GQ)
    exp, _ = oracle_built.call(oracle_kind(oracle_built), params, batch, None)
    got = run(params, batch, None, {"adjudicate": 1})
    st = parity.compare(got, exp, params)
    assert st["compared"] > 0 and not st["near_ties"], st
    check_flags(got)
    one = (got.ret > 0) & ((got.als_new == 0b011) | (got.als_new == 0b101))
    assert one.sum() > R // 2
    assert (got.site_flags[one] & abi.SITE_ADJUDICATED).all()
    assert (got.als_new[one] == 0b011).all()          # REF + the first ALT: {A} is the first of the tied sets


@pytest.mark.parametrize("groups", [None, 5])
def test_off_means_off(groups):
    """adjudicate = 0 (the default) changes nothing, and no site carries the ADJUDICATED bit."""
    from bcftools_b200 import mcall
    S = 200
    rng = np.random.default_rng([S, 8])
    batch = parity.random_batch(rng, 120, S, 5)
    params = abi.CallParams(S, 5, output_tags=abi.CALL_FMT_GQ, groups=groups_of(S, groups))
    a = run(params, batch, None, {}, compact=True)
    b = run(params, batch, None, {"adjudicate": 0}, compact=True)
    for name in ("ret", "als_new", "als_map", "ac", "an", "site_flags", "gt", "gq"):
        assert (getattr(a, name) == getattr(b, name)).all(), name
    assert (a.qual.view(np.uint32) == b.qual.view(np.uint32)).all()
    assert ((a.pl_off_out < 0) == (b.pl_off_out < 0)).all()      # compacted blocks are placed in no particular order
    for i in range(batch.nsites):
        if a.pl_off_out[i] >= 0:
            assert (a.site_pl(i) == b.site_pl(i)).all(), i
    assert not (a.site_flags & abi.SITE_ADJUDICATED).any()


def test_adjudicate_needs_site_flags():
    import torch
    from bcftools_b200 import device, mcall
    S = 16
    batch = parity.random_batch(np.random.default_rng(1), 8, S, 3)
    db = device.DeviceBatch(batch)
    dr = device.DeviceResult(db)
    rs = dr.c_struct()
    rs.site_flags = None
    with mcall.MCaller(abi.CallParams(S, 5), options={"adjudicate": 1}) as mc:
        with pytest.raises(mcall.McallError):
            mc.call_device(db.c_struct(), rs, torch.cuda.current_stream().cuda_stream)
        with pytest.raises(mcall.McallError):
            mc.set_option("adjudicate", 2)


@pytest.mark.parametrize("S,maxA,minA", [(300, 3, 3), (41, 5, 1), (20, 9, 6)])
def test_compacted_capacity_with_every_site_flagged(S, maxA, minA, oracle_built):
    """Every site flagged, compacted output over several slabs: the used prefix stays within sum_i pad4(S*G_i), the capacity
    mcall_b200.h documents, also where the second evaluation keeps more alleles than the first (3-allele pair -> triple)."""
    rng = np.random.default_rng([S, maxA, 12])
    batch = parity.random_batch(rng, 150, S, maxA, minA=minA)
    params = abi.CallParams(S, maxA, flag=abi.CALL_VARONLY, output_tags=abi.CALL_FMT_GQ, tie_eps=ALL)
    exp, _ = oracle_built.call(oracle_kind(oracle_built), params, batch, None)
    plain = run(params, batch, None, {"slab_bytes": 1 << 16}, compact=True)
    got = run(params, batch, None, {"slab_bytes": 1 << 16, "adjudicate": 1}, compact=True)
    st = parity.compare(got, exp, params)
    assert st["compared"] > 0 and not st["near_ties"], st
    check_flags(got)
    cap = int(sum(abi.pad4(S * int(g)) for g in batch.ngt))
    ends = [int(got.pl_off_out[i]) + abi.pad4(S * int(batch.ngt[i])) for i in range(batch.nsites) if got.pl_off_out[i] >= 0]
    assert ends and max(ends) <= cap
    blocks = sorted((int(got.pl_off_out[i]), i) for i in range(batch.nsites) if got.pl_off_out[i] >= 0)
    for (o1, i1), (o2, _) in zip(blocks, blocks[1:]):        # disjoint: a flagged site's block spans its full G
        n = got.ret[i1]
        assert o1 + abi.pad4(S * n * (n + 1) // 2) <= o2
    dropped = (got.site_flags & abi.SITE_PL_DROPPED) != 0
    assert (got.pl_off_out[(got.ret > 0) & ~dropped] >= 0).all()          # every site with PLs has its block
    assert (got.pl_off_out[dropped & (got.ret > 0)] < 0).all()
    if minA == 3 and maxA == 3:
        grew = (plain.ret > 0) & (got.ret > plain.ret)
        print("3-allele sites whose trimmed set grew:", int(grew.sum()))


@pytest.mark.parametrize("kind", ["grouped", "typed", "alleles6"])
def test_batcher_adjudicates_every_mode(kind, oracle_built):
    from bcftools_b200 import host_call
    rng = np.random.default_rng([len(kind), 6])
    S = 37
    if kind == "alleles6":
        batch = parity.random_batch(rng, 90, S, 6)
        params = abi.CallParams(S, 6, output_tags=abi.CALL_FMT_GQ)
    else:
        batch = parity.random_batch(rng, 150, S, 5)
        params = abi.CallParams(S, 5, output_tags=abi.CALL_FMT_GQ, groups=groups_of(S, 4) if kind == "grouped" else None)
    exp, _ = oracle_built.call(oracle_kind(oracle_built), params, batch, None)
    for async_flush in (False, True):
        got = host_call.replay(params, batch, None, max_records=64, typed=kind == "typed", async_flush=async_flush, tie_eps=ALL)
        st = parity.compare(got, exp, params)
        assert st["compared"] > 0 and not st["near_ties"], st
        assert check_flags(got).mean() > 0.3


def test_job_with_adjudication_equals_one_context(oracle_built):
    import torch
    from bcftools_b200 import mcall
    S = 64
    rng = np.random.default_rng(31)
    batch = parity.random_batch(rng, 160, S, 5)
    params = abi.CallParams(S, 5, output_tags=abi.CALL_FMT_GQ, tie_eps=ALL)
    one = run(params, batch, None, {"adjudicate": 1}, compact=True)
    devs = list(range(torch.cuda.device_count()))
    with mcall.MJob(params, devs, options={"adjudicate": 1}) as job:
        many = job.call_host(batch, compact=True)
    for name in ("ret", "als_new", "als_map", "ac", "an", "site_flags", "gt", "gq"):
        assert (getattr(one, name) == getattr(many, name)).all(), name
    assert (one.qual.view(np.uint32) == many.qual.view(np.uint32)).all()
    for i in range(batch.nsites):
        if one.ret[i] > 0 and not (one.site_flags[i] & abi.SITE_PL_DROPPED):
            assert (one.site_pl(i) == many.site_pl(i)).all(), i
    check_flags(many)


@pytest.mark.parametrize("S,maxA,minA,groups", [(2504, 5, 3, 5), (40, 12, 6, None)])
def test_against_the_compiled_reference(S, maxA, minA, groups, oracle_built):
    if not oracle_built.have_ref():
        pytest.skip("the compiled reference (oracle/_ref) is not built")
    rng = np.random.default_rng([S, maxA, 88])
    batch = parity.random_batch(rng, 24 if S > 1000 else 60, S, maxA, minA=minA)
    params = abi.CallParams(S, maxA, output_tags=abi.CALL_FMT_GQ, groups=groups_of(S, groups), tie_eps=ALL)
    exp, _ = oracle_built.call("reference", params, batch, None)
    got = run(params, batch, None, {"adjudicate": 1})
    st = parity.compare(got, exp, params)
    assert st["compared"] > 0 and not st["near_ties"], st
    check_flags(got)
