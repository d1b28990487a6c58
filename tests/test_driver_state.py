"""include/b200_driver.h (SURVEY.md 8f N2): ploidy definitions + set_ploidy, -G group files, the unseen allele -- against
the committed golden cases (whose per-site ploidy vectors / unseen alleles / groups reproduce the reference's outputs),
the reference's own option files and expected outputs (bundled in tests/golden/vcf_text_cases.json.gz), its ploidy
presets (tests/golden/ploidy_presets.txt) and the quirks of ploidy.c / mcall.c."""
import os
import re

import numpy as np
import pytest

from bcftools_b200 import driver
from tests import golden_util, vcf_cases

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _ref_file(name):
    """Text of a file of the reference's test/ directory, from the committed bundle."""
    return vcf_cases.bundle()["files"][name]

# the definition the reference's chrX tests use (test/test.pl:281-283), in the format of ploidy.c:40-53
PLOIDY_X = "X 1 1000 M 1\nX 3104 5000 M 1\n* * * M 2\n* * * F 2\n"


def test_symbols_are_exported():
    from bcftools_b200 import mcall
    hdr = re.sub(r"/\*.*?\*/", "", open(os.path.join(ROOT, "include", "b200_driver.h")).read(), flags=re.S)
    syms = sorted(set(re.findall(r"\b(b200_[A-Za-z0-9_]+)\s*\(", hdr)))
    assert syms == sorted(driver.DRIVER_EXPORTS)
    assert all(hasattr(mcall.lib(), s) for s in syms)


def test_unseen_allele_of_every_golden_site():
    n = 0
    for name in golden_util.case_names():
        case = golden_util.load_case(name)[3]
        for s in case["sites"]:
            assert driver.unseen_allele(s["alleles"]) == s["unseen"], (name, s["alleles"])
            n += 1
    assert n > 100
    assert driver.unseen_allele(["A", "C", "<*>"]) == 2 and driver.unseen_allele(["A", "<X>"]) == 1
    assert driver.unseen_allele(["A", "X"]) == 1 and driver.unseen_allele(["A", "<NON_REF>", "C"]) == 0
    assert driver.unseen_allele(["<*>"]) == 0          # REF is never looked at (vcfcall.c:1103 starts at 1)


@pytest.mark.parametrize("name,sexes", [("mpileup.X", "FMF"), ("mpileup.X.ped", "FMF")])
def test_set_ploidy_replays_the_chrX_goldens(name, sexes):
    """vcfcall.c:807-825 over the records of the golden case: the ploidy vector in force at every site must be the one the
    golden was generated (and reproduces the reference's output) with."""
    case = golden_util.load_case(name)[3]
    pl = driver.Ploidy(PLOIDY_X, 2)
    assert pl.sexes == ["M", "F"] and (pl.min(), pl.max()) == (1, 2)
    s2s = np.array([pl.sex2id(s) for s in sexes], np.int32)
    prev = np.full(len(pl.sexes), pl.max(), np.int32)           # vcfcall.c:652-655
    ploidy = np.full(len(sexes), pl.max(), np.uint8)
    changes = 0
    for s in case["sites"]:
        changes += pl.set_ploidy(s["chrom"], s["pos"] - 1, s2s, prev, ploidy)
        assert ploidy.tolist() == case["ploidy_vectors"][s["ploidy_id"]], (s["pos"], ploidy)
    assert changes >= 2
    pl.close()


def test_ploidy_query_semantics():
    pl = driver.Ploidy("X 1 60000 M 1\nX 2699521 154931043 M 1\nY 1 59373566 M 1\nY 1 59373566 F 0\nMT 1 16569 M 1\nMT 1 16569 F 1\n"
                       "*  * *     M 2\n*  * *     F 2\n", 2)
    assert pl.sexes == ["M", "F"] and (pl.min(), pl.max()) == (0, 2)
    assert pl.query("X", 0) == (1, {"M": 1, "F": 2}, 1, 1)
    assert pl.query("X", 59999) == (1, {"M": 1, "F": 2}, 1, 1)      # 1-based inclusive end 60000 = 0-based 59999
    assert pl.query("X", 60000) == (0, {"M": 2, "F": 2}, 2, 2)
    assert pl.query("Y", 100) == (1, {"M": 1, "F": 0}, 0, 1)
    assert pl.query("MT", 5) == (1, {"M": 1, "F": 1}, 1, 1)
    assert pl.query("1", 5) == (0, {"M": 2, "F": 2}, 2, 2)
    assert pl.add_sex("U") == 2 and pl.query("Y", 100)[1] == {"M": 1, "F": 0, "U": 2}
    # a region whose ploidy equals the default does not count as a hit for min/max but still is an overlap (ploidy.c:214-226)
    p2 = driver.Ploidy("1 10 20 M 2\n* * * M 1\n", 2)
    assert p2.query("1", 10) == (1, {"M": 2}, 2, 2) and p2.query("1", 30) == (0, {"M": 1}, 2, 2)
    # SEX "*" sets the default of everything (ploidy.c:126)
    p3 = driver.Ploidy("* * * * 1\nX 1 5 F 2\n", 2)
    assert p3.query("2", 0)[1] == {"*": 1, "F": 1} and p3.query("X", 0)[1]["F"] == 2
    # ploidy.c:114-118 files a default under the most recently ADDED sex, not under the line's own: reproduced
    p4 = driver.Ploidy("X 1 5 M 1\nX 1 5 F 2\n* * * M 0\n", 2)
    assert p4.query("2", 0)[1] == {"M": 2, "F": 0}
    with pytest.raises(driver.DriverError):
        driver.Ploidy("X 1 5 M\n", 2)
    with pytest.raises(driver.DriverError):
        driver.Ploidy("X 9 5 M 1\n", 2)


def test_groups_parse_semantics():
    smp = ["s0", "s1", "s2", "s3", "s4"]
    off, g = driver.groups_parse("s3\tPOPB\nsX\tPOPC\ns0 \t POPA\ns1\tPOPB\ns4\tPOPA\ns2\tPOPB\n", smp)
    assert off.tolist() == [0, 3, 5] and g.tolist() == [1, 2, 3, 0, 4]      # first-appearance order of groups, header order inside
    off, g = driver.groups_parse("-", smp)
    assert off.tolist() == [0, 1, 2, 3, 4, 5] and g.tolist() == [0, 1, 2, 3, 4]
    # mcall.c:321-325 keys the populations WITHOUT their first character: "XEU" and "YEU" are one group
    off, g = driver.groups_parse("s0 XEU\ns1 YEU\ns2 ZRI\ns3 ZRI\ns4 XEU\n", smp)
    assert off.tolist() == [0, 3, 5] and g.tolist() == [0, 1, 4, 2, 3]
    with pytest.raises(driver.DriverError, match="listed twice"):
        driver.groups_parse("s0 A1\ns0 A2\n", smp)
    with pytest.raises(driver.DriverError, match="not listed"):
        driver.groups_parse("s0 A1\ns1 A1\n", smp)
    with pytest.raises(driver.DriverError, match="no matching samples"):
        driver.groups_parse("u0 A1\n", smp)
    with pytest.raises(driver.DriverError, match="expected a sample name"):
        driver.groups_parse("s0\n", smp)


@pytest.mark.parametrize("name,fname", [("call.af-fixation.2", "call.af-fixation.txt"), ("mpileup.hwe.4", "mpileup.hwe.samples")])
def test_groups_of_the_reference_option_files(name, fname):
    """The reference's own -G files (test/test.pl:287, 306): the parsed member lists must be the groups the golden case
    was generated with."""
    case = golden_util.load_case(name)[3]
    off, g = driver.groups_parse(_ref_file(fname), case["samples"])
    got = [g[off[k]:off[k + 1]].tolist() for k in range(len(off) - 1)]
    assert got == case["groups"]


def test_driver_state_feeds_the_c_abi_structs():
    """grp_off / grp_smpl go straight into mcb_params (abi.CallParams accepts member lists: same content)."""
    from bcftools_b200 import abi
    off, g = driver.groups_parse("a P1\nb Q2\nc P1\n", ["a", "b", "c"])
    p = abi.CallParams(3, 5, groups=[g[off[k]:off[k + 1]].tolist() for k in range(len(off) - 1)])
    assert p.ngroups == 2 and p.grp_off.tolist() == off.tolist() and p.grp_smpl.tolist() == g.tolist()


HDR3 = ["HG00100", "HG00101", "HG00102"]        # sample columns of the reference's test/mpileup*.vcf


def test_samples_parse_semantics():
    pl = driver.Ploidy(PLOIDY_X, 2)
    smap, s2s, warn = pl.samples_parse("HG00102 F\n# comment\nNA1 M\nHG00100\tM\nHG00102 M\nHG00101 1\n", HDR3)
    assert smap.tolist() == [2, 0, 1] and warn == 2                       # unknown sample + listed twice are skipped with a warning
    assert s2s.tolist() == [pl.sex2id("F"), pl.sex2id("M"), -1]            # literal ploidy 1 -> -1 (vcfcall.c:317-320)
    smap, s2s, _ = pl.samples_parse("HG00101\n", HDR3)
    assert smap.tolist() == [1] and s2s.tolist() == [-2]                   # no second column: ploidy 2
    smap, s2s, _ = pl.samples_parse("HG00100 U\n", HDR3)                   # a sex the ploidy file does not know is added with the default
    assert pl.sexes == ["M", "F", "U"] and s2s.tolist() == [2]
    # PED: >= 6 columns on every line; sex 1 = M, anything else F; named parents are added as M / F
    smap, s2s, _ = pl.samples_parse("f1 HG00102 HG00100 HG00101 2 0\n", HDR3)
    assert smap.tolist() == [2, 0, 1] and s2s.tolist() == [pl.sex2id("F"), pl.sex2id("M"), pl.sex2id("F")]
    with pytest.raises(driver.DriverError, match="not a PED"):
        pl.samples_parse("f1 HG00102 0 0 2 0\nHG00100 M\n", HDR3)
    smap, s2s = pl.samples_default(3)
    assert smap.tolist() == [0, 1, 2] and s2s.tolist() == [2, 2, 2]        # nsex-1 (vcfcall.c:645-649)
    pl.close()


@pytest.mark.parametrize("name,fname", [("mpileup.3", "mpileup.3.samples"), ("mpileup.4", "mpileup.4.samples"), ("mpileup.5", "mpileup.5.samples"),
                                        ("mpileup.X", "mpileup.samples"), ("mpileup.X.ped", "mpileup.ped"), ("mpileup.X.2", "mpileup.2.samples")])
def test_samples_of_the_reference_option_files(name, fname):
    """The reference's own -S files (test/test.pl:278-283): selected samples in the order of the golden case, and -- with the
    chrX ploidy definition -- the per-site ploidy vectors of the golden via set_ploidy."""
    case = golden_util.load_case(name)[3]
    pl = driver.Ploidy(PLOIDY_X if "X" in name else "* * * M 2\n* * * F 2\n", 2)
    smap, s2s, warn = pl.samples_parse(_ref_file(fname), HDR3)
    assert [HDR3[m] for m in smap] == case["samples"]
    prev = np.full(len(pl.sexes), pl.max(), np.int32)
    ploidy = np.full(len(smap), pl.max(), np.uint8)
    for s in case["sites"]:
        pl.set_ploidy(s["chrom"], s["pos"] - 1, s2s, prev, ploidy)
        assert ploidy.tolist() == case["ploidy_vectors"][s["ploidy_id"]], (s["pos"], ploidy)
    pl.close()


def _vcf_records(text):
    out = []
    for l in text.splitlines(True):
        if l.startswith("#"):
            continue
        f = l.rstrip("\n").split("\t")
        info = dict(kv.split("=", 1) if "=" in kv else (kv, "") for kv in f[7].split(";"))
        out.append(dict(chrom=f[0], pos=int(f[1]), ref=f[3], alt=f[4].split(","), info=info, fmt=f[8].split(":") if len(f) > 8 else [],
                        smpl=[x.split(":") for x in f[9:]]))
    return out


def test_trim_numberR_semantics():
    ad = np.array([[10, 3, 0, 7], [5, 0, 2, 1]], np.int32)                  # two samples, REF + 3 ALTs
    assert driver.trim_numberR(ad, [0, -1, -1, 1], 2).tolist() == [[10, 7], [5, 1]]
    assert driver.trim_numberR(ad, [0, 1, 2, -1], 3).tolist() == [[10, 3, 0], [5, 0, 2]]
    assert driver.trim_numberR(np.array([[0.5, 0.25, 0.125]], np.float32), [0, -1, 1], 2).tolist() == [[0.5, 0.125]]


@pytest.mark.parametrize("vcf,out", [("mpileup.vcf", "mpileup.1.out"), ("mpileup.X.vcf", "mpileup.X.out"), ("call-G.vcf", "call-G.1.out"),
                                     ("mpileup.hwe.vcf", "mpileup.hwe.2.out"), ("call.af-fixation.vcf", "call.af-fixation.1.out")])
def test_finaliser_pieces_against_the_reference_outputs(vcf, out):
    """DP4 / MQ from INFO/I16 (mcall.c:1660-1666) and the Number=R trimming of FORMAT/AD (mcall.c:1196-1265) against the records
    of the reference's own expected outputs."""
    src = {(r["chrom"], r["pos"], r["ref"]): r for r in _vcf_records(_ref_file(vcf))}
    n_dp4 = n_ad = 0
    for o in _vcf_records(_ref_file(out)):
        r = src.get((o["chrom"], o["pos"], o["ref"]))
        if r is None or "I16" not in r["info"]:
            continue
        dp4, mq = driver.i16_to_dp4_mq([float(x) for x in r["info"]["I16"].split(",")])
        assert ",".join(map(str, dp4)) == o["info"]["DP4"] and str(mq) == o["info"]["MQ"], (o["pos"], dp4, mq)
        n_dp4 += 1
        if "AD" in r["fmt"] and "AD" in o["fmt"]:
            old = [r["ref"]] + r["alt"]
            new = [o["ref"]] + [a for a in o["alt"] if a != "."]
            if len(new) == len(old):
                continue
            als_map = [new.index(a) if a in new else -1 for a in old]
            k, ko = r["fmt"].index("AD"), o["fmt"].index("AD")
            rows = [s[k].split(",") for s in r["smpl"]]
            if any(len(x) != len(old) or "." in x for x in rows):
                continue
            got = driver.trim_numberR(np.array(rows, np.int32), als_map, len(new))
            assert [",".join(map(str, g)) for g in got.tolist()] == [s[ko] for s in o["smpl"]], o["pos"]
            n_ad += 1
    assert n_dp4 >= 1 and (n_ad >= 1 or vcf.startswith("mpileup.") and "hwe" not in vcf)


def test_ploidy_aliases():
    g38 = driver.Ploidy(alias="grch38")                         # case-insensitive (vcfcall.c:834)
    assert g38.sexes == ["M", "F"] and (g38.min(), g38.max()) == (0, 2)
    assert g38.query("chrX", 9998)[1] == {"M": 1, "F": 2} and g38.query("chrX", 9999)[1] == {"M": 2, "F": 2}       # PAR1 starts behind 9,999
    assert g38.query("X", 2781479)[1] == {"M": 1, "F": 2} and g38.query("X", 2781478)[1] == {"M": 2, "F": 2}
    assert g38.query("chrY", 5)[1] == {"M": 1, "F": 0} and g38.query("chrM", 5)[1] == {"M": 1, "F": 1} and g38.query("MT", 5)[1] == {"M": 1, "F": 1}
    assert g38.query("chr1", 5)[1] == {"M": 2, "F": 2}
    g37 = driver.Ploidy(alias="GRCh37")
    assert g37.query("X", 59999)[1] == {"M": 1, "F": 2} and g37.query("X", 60000)[1] == {"M": 2, "F": 2} and g37.query("X", 2699520)[1]["M"] == 1
    assert driver.Ploidy(alias="X").query("7", 1)[1] == {"M": 1, "F": 2}
    assert driver.Ploidy(alias="Y").query("7", 1)[1] == {"M": 1, "F": 0}
    assert driver.Ploidy(alias="1").query("7", 1)[1] == {"*": 1}
    with pytest.raises(driver.DriverError):
        driver.Ploidy(alias="hg18")


def test_ploidy_aliases_against_the_reference_source():
    """Every preset of vcfcall.c:138-198 (its .ploidy strings, kept in tests/golden/ploidy_presets.txt under one '# alias'
    line each) answers the same per-sex ploidies as the alias on a grid of positions around all of its region boundaries."""
    text = open(os.path.join(ROOT, "tests", "golden", "ploidy_presets.txt")).read()
    n = 0
    for alias, body in re.findall(r"^# (\S+)\n((?:[^#].*\n)+)", text, flags=re.M):
        ref, mine = driver.Ploidy(body, 2), driver.Ploidy(alias=alias)
        assert ref.sexes == mine.sexes, alias
        probes = [("7", 100)]
        for l in body.splitlines():
            c = l.split()
            if c and c[0] != "*":
                probes += [(c[0], int(x) + d) for x in c[1:3] for d in (-2, -1, 0, 1)]
        for seq, pos in probes:
            assert ref.query(seq, max(0, pos)) == mine.query(seq, max(0, pos)), (alias, seq, pos)
        n += 1
    assert n == 5
