"""Host-side logic that needs no GPU: batch packing, synthetic generator, byte accounting, oracle cross-checks."""
import hashlib
import os

import numpy as np
import pytest

from bcftools_b200 import abi, synth
from tests import parity


def test_hostbatch_layout_is_16_byte_aligned_and_padded():
    rng = np.random.default_rng(0)
    b = parity.random_batch(rng, 50, 7, 5)
    assert (b.pl_off % 4 == 0).all()
    for i in range(b.nsites):
        g = int(b.ngt[i])
        assert b.site_pl(i).shape == (7, g)
        end = b.pl_off[i] + 7 * g
        nxt = b.pl_off[i + 1] if i + 1 < b.nsites else b.pl.size
        assert end <= nxt and (b.pl[end:nxt] == abi.INT32_VECTOR_END).all()


def test_subset_roundtrip():
    params, b, tab = synth.make_batch("C3", 40)
    sub = b.subset([3, 7, 11])
    for k, i in enumerate([3, 7, 11]):
        assert (sub.site_pl(k) == b.site_pl(i)).all() and sub.nals[k] == b.nals[i]
        assert (sub.qs[k] == b.qs[i]).all()


@pytest.mark.parametrize("cfg", ["C1", "C2", "C3", "C5"])
def test_synthetic_generator_is_seeded_and_mpileup_shaped(cfg):
    p1, b1, _ = synth.make_batch(cfg, 30)
    p2, b2, _ = synth.make_batch(cfg, 30)
    assert (b1.pl == b2.pl).all() and (b1.qs == b2.qs).all()
    for i in range(b1.nsites):
        pl = b1.site_pl(i)
        ok = pl[(pl != abi.INT32_MISSING) & (pl != abi.INT32_VECTOR_END)]
        assert ok.min() >= 0 and ok.max() <= 255           # bam2bcf.c:645-646
    assert b1.nsmpl == synth.CONFIGS[cfg]["nsmpl"]


RANDOM_REFERENCE = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "random_reference.npz")
RANDOM_REFERENCE_FIELDS = ("ret", "als_new", "als_map", "qual", "ac", "an", "site_flags", "gt", "gq", "pl", "gp")


def random_reference_cases():
    """The five seeded adversarial batches the port is compared with the reference on: -> [(params, batch, ploidy_tab, want_gp)]."""
    rng = np.random.default_rng(11)
    out = []
    for (R, S, A, flag, tags, groups) in [(150, 7, 5, 0, abi.CALL_FMT_GQ, None), (120, 33, 4, abi.CALL_KEEPALT, abi.CALL_FMT_GQ, None),
                                          (120, 40, 5, abi.CALL_VARONLY, abi.CALL_FMT_GQ | abi.CALL_FMT_GP, None),
                                          (100, 30, 5, 0, abi.CALL_FMT_GQ, 3), (60, 9, 4, abi.CALL_VARONLY, abi.CALL_FMT_GQ, "single")]:
        b = parity.random_batch(rng, R, S, A, zq=not (tags & abi.CALL_FMT_GP))
        g = None
        if groups == 3:
            g = [list(range(k, S, 3)) for k in range(3)]
        elif groups == "single":
            g = [[s] for s in range(S)]
        params = abi.CallParams(S, A, flag=flag, output_tags=tags, groups=g)
        tab = np.full((2, S), 2, np.uint8)
        tab[1, ::3] = 1
        tab[1, 1::7] = 0
        b.ploidy_id = rng.integers(0, 2, R).astype(np.uint16)
        out.append((params, b, tab, bool(tags & abi.CALL_FMT_GP)))
    return out


def inputs_digest(params, batch, tab):
    """sha256 over everything an oracle reads: a stored result is only compared on the very inputs it was computed from."""
    h = hashlib.sha256()
    h.update(np.array([params.nsmpl, params.max_nals, params.flag, params.output_tags, batch.nsites], np.int64).tobytes())
    h.update(np.float64(params.theta).tobytes())
    for a in [params.grp_off, params.grp_smpl, tab] + [getattr(batch, name) for name in abi.BATCH_FIELDS]:
        h.update(b"-" if a is None else np.ascontiguousarray(a).tobytes())
    return h.hexdigest()


def stored_result(gold, k, batch, want_gp):
    res = abi.HostResult(batch, want_gp=want_gp)
    for name in RANDOM_REFERENCE_FIELDS:
        if getattr(res, name) is not None:
            getattr(res, name)[...] = gold[f"{k}_{name}"]
    return res


def test_restatement_equals_compiled_reference_on_random_inputs(oracle_built):
    """The plain-C port against the reference's unmodified mcall.c on five seeded adversarial batches (GP, -G groups,
    -v / keep-alts, mixed ploidy): against the reference's results stored in tests/golden/random_reference.npz
    (tests/golden/make_random_reference.py), and against the compiled reference itself where oracle/_ref is built."""
    gold = np.load(RANDOM_REFERENCE)
    for k, (params, b, tab, want_gp) in enumerate(random_reference_cases()):
        assert str(gold[f"{k}_inputs"]) == inputs_digest(params, b, tab), f"batch {k}: not the inputs the stored results belong to"
        a, _ = oracle_built.call("port", params, b, tab, want_gp=want_gp)
        refs = [stored_result(gold, k, b, want_gp)]
        if oracle_built.have_ref():
            refs.append(oracle_built.call("reference", params, b, tab, want_gp=want_gp)[0])
        for r in refs:
            st = parity.compare(a, r, params, exact_qual=True)
            assert st["compared"] > 0 and not st["near_ties"]


def test_algorithmic_bytes_accounting(oracle_built):
    params, b, tab = synth.make_batch("C2", 20)
    res, _ = oracle_built.call("port", params, b, tab)
    rd, wr = synth.algorithmic_bytes(b, res, params.output_tags)
    S = params.nsmpl
    assert rd >= 20 * S * 3 * 4
    var = (res.ret == 2).sum()
    ref = (res.ret == 1).sum()
    assert wr == var * S * (8 + 4 + 12) + ref * S * 8       # SURVEY.md §8d: 36 B per biallelic call with GQ and PL kept
