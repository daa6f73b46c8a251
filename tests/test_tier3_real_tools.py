"""Tier (iii) of SURVEY.md section 4: differential tests against the REAL third-party tools the reference calls --
cutadapt (imported by mirge/libs/digest.py:5-13) and bowtie 1.x (spawned by mirge/libs/manifoldAlign.py:47).  Neither
is installable in the build container (no network, not in the wheelhouse), so every test here skips cleanly there; on any
box that has them (`pip install cutadapt`, `bowtie` on PATH) they pin what the oracle only restates:

* cutadapt: Aligner / match_to trim points and the two quality trimmers, with the objective that matches the installed
  version (< 4: most matches, then cost -- compat "2-3"; >= 4: score -- compat "4");
* bowtie: for every round's command line (manifoldAlign.py:85) the reported alignment is a member of the oracle's valid
  hit set, has the oracle's best mismatch count where --best applies, equals the canonical pick when the set is a
  singleton, and reads without a valid alignment are reported unaligned.

CPU only (no GPU marker): what is held against the tools is the oracle; the GPU path is held against the oracle."""
import os
import shutil
import subprocess

import numpy as np
import pytest

from oracle import pyoracle as po

ILL = "TGGAATTCTCGGGTGCCAAGGAACTCCAG"
B = list("ACGT")


def _real_cutadapt():
    """The installed cutadapt, or skip -- also when the module in sys.modules is the stand-in other tests of this
    suite register to run the reference's own code (tests/golden/standins.py), which answers with the oracle."""
    cutadapt = pytest.importorskip("cutadapt")
    if "stand-in" in str(getattr(cutadapt, "__version__", "")) or not getattr(cutadapt, "__file__", None):
        pytest.skip("cutadapt in sys.modules is the stand-in of tests/golden/standins.py, not an install")
    return cutadapt


def _reads(rng, adapter, n):
    out = []
    for _ in range(n):
        ins = "".join(rng.choice(B, int(rng.integers(0, 40))))
        r = rng.random()
        if r < 0.6:  # adapter copy with substitutions / indels, random tail
            ad = []
            for c in adapter:
                x = rng.random()
                if x < 0.03:
                    continue
                if x < 0.06:
                    ad.append(str(rng.choice(B)))
                ad.append(str(rng.choice(B)) if rng.random() < 0.05 else c)
            s = ins + "".join(ad) + "".join(rng.choice(B, int(rng.integers(0, 15))))
        elif r < 0.8:  # partial adapter at the 3' end
            s = ins + adapter[: int(rng.integers(1, len(adapter)))]
        else:
            s = ins + "".join(rng.choice(B, int(rng.integers(0, 30))))
        if rng.random() < 0.05 and s:
            p = int(rng.integers(0, len(s)))
            s = s[:p] + "N" + s[p + 1:]
        out.append(s)
    return out


def _cutadapt_adapters(cutadapt, sequence, where, rate, overlap, indels):
    """A single adapter object across cutadapt 2.x / 3.x / 4.x APIs."""
    ad = cutadapt.adapters
    kw = dict(max_errors=rate, min_overlap=overlap, read_wildcards=False, adapter_wildcards=True, indels=indels)
    if hasattr(ad, "BackAdapter"):
        cls = ad.BackAdapter if where == "back" else ad.FrontAdapter
        try:
            return cls(sequence, **kw)
        except TypeError:
            kw["max_error_rate"] = kw.pop("max_errors")
            return cls(sequence, **kw)
    where_c = ad.Where.BACK if where == "back" else ad.Where.FRONT
    kw["max_error_rate"] = kw.pop("max_errors")
    return ad.Adapter(sequence, where=where_c, **kw)


@pytest.mark.parametrize("where", ["back", "front"])
@pytest.mark.parametrize("indels", [True, False])
def test_adapter_trim_points_match_cutadapt(where, indels):
    cutadapt = _real_cutadapt()
    import cutadapt.adapters  # noqa: F401

    major = int(str(cutadapt.__version__).split(".")[0])
    compat = "4" if major >= 4 else "2-3"
    rng = np.random.default_rng(7)
    for adapter, rate, overlap in ((ILL, 0.12, 3), ("AACTGTAGGCACCATCAAT", 0.1, 3), ("TGGAATTCNNGGGTGCCAAGGRACTCCAG", 0.2, 5)):
        real = _cutadapt_adapters(cutadapt, adapter, where, rate, overlap, indels)
        mine = po.Adapter(where, adapter, rate, overlap, indels, True)
        for read in _reads(rng, adapter.replace("N", "A").replace("R", "G"), 1500):
            try:
                m = real.match_to(read)
            except TypeError:  # 2.x wants a Sequence object
                from dnaio import Sequence

                m = real.match_to(Sequence("r", read))
            o = po.match_to(mine, read, compat)
            assert (m is None) == (o is None), (cutadapt.__version__, where, indels, adapter, read)
            if m is None:
                continue
            got = (m.rstart, m.rstop, m.errors)
            assert got == (o[2], o[3], o[5]), (cutadapt.__version__, where, indels, adapter, read, got, o)
            merit = getattr(m, "score", None) if compat == "4" else getattr(m, "matches", None)
            if merit is not None:
                assert merit == o[4], (cutadapt.__version__, read, merit, o)


SPEC_CASES = [  # (-a / -g arguments, --match-read-wildcards): the specification language beyond plain adapters
    ([("back", ILL + "$")], False), ([("front", "^GTTCAGAGTTCTAC")], False), ([("back", ILL + "X")], False),
    ([("front", "XGTTCAGAGTTCTAC")], False), ([("back", ILL + ";e=0.2;o=6")], False), ([("back", "TGGAA{3}TTCTCGG")], False),
    ([("front", "GTTCAGAGTTCTAC..." + ILL)], False), ([("back", "GTTCAGAGTTCTAC..." + ILL)], False),
    ([("back", "^GTTCAGAGTTCTAC..." + ILL)], False), ([("front", "GTTCAGAGTTCTAC;optional..." + ILL + ";e=0.2")], False),
    ([("back", "GTTCAGAGTTCTAC;required..." + ILL + "$")], False), ([("back", ILL)], True), ([("front", "GTTCAGAGTTCTAC"), ("back", ILL + "X")], True),
    # -a with non-internal halves: whether a non-internal half counts as "anchored" (= required) is the one point of
    # cutadapt's _parse_linked the restatement is unsure of (params.parse_adapter_spec: only ^ / $ make a half required)
    ([("back", "XGTTCAGAGTTCTAC..." + ILL)], False), ([("back", "GTTCAGAGTTCTAC..." + ILL + "X")], False),
]


@pytest.mark.parametrize("case", range(len(SPEC_CASES)))
def test_specification_language_matches_cutadapt(case):
    """The adapters exactly as the reference's stipulate() makes them (digest.py:66-85: cutadapt's own parser on
    args.adapters) and cutadapt's AdapterCutter on reads, against params.parse_adapter_specs + the oracle's modifier:
    placements, per-adapter parameters, linked pairs with required / optional halves, read wildcards."""
    cutadapt = _real_cutadapt()
    from cutadapt.modifiers import AdapterCutter

    from mirge_b200 import params as P
    from tests.util import py_params

    specs, read_wild = SPEC_CASES[case]
    search = dict(max_errors=0.12, min_overlap=3, read_wildcards=read_wild, adapter_wildcards=True, indels=True)
    try:
        from cutadapt.parser import make_adapters_from_specifications

        adapters = make_adapters_from_specifications(specs, search)
    except ImportError:
        from cutadapt.parser import AdapterParser

        search["max_error_rate"] = search.pop("max_errors")
        adapters = AdapterParser(**search).parse_multi(specs)
    cutter = AdapterCutter(adapters, 2, "trim")
    major = int(str(cutadapt.__version__).split(".")[0])
    cfg = P.TrimConfig(adapters=specs, times=2, quality_cutoff=None, match_read_wildcards=read_wild,
                       cutadapt_compat="4" if major >= 4 else "2-3")
    pp = py_params(cfg)
    mod = [m for m in pp.modifiers() if m[0] == "adapter"][0]
    from dnaio import Sequence

    rng = np.random.default_rng(100 + case)
    front = "GTTCAGAGTTCTAC"
    for read in _reads(rng, ILL, 1500):
        if rng.random() < 0.5:  # a 5' adapter (damaged, sometimes not at the very start) in front
            f = "".join(str(rng.choice(B)) if rng.random() < 0.05 else c for c in front)
            read = ("".join(rng.choice(B, int(rng.integers(1, 4)))) if rng.random() < 0.2 else "") + f + read
        if not read:
            continue
        rec = Sequence("r", read, "I" * len(read))
        try:
            out = cutter(rec, [])
        except TypeError:
            from cutadapt.info import ModificationInfo

            out = cutter(rec, ModificationInfo(rec))
        start, stop = po.apply_modifier(mod, read, "I" * len(read), 0, len(read), pp)
        assert out.sequence == read[start:stop], (cutadapt.__version__, specs, read_wild, read, out.sequence, read[start:stop])


def _reference_baking():
    """The unmodified reference's baking() running on the REAL cutadapt / dnaio / xopen: from the read-only checkout or an
    installed ``mirge`` package.  Skips unless all of them are there."""
    import sys

    _real_cutadapt()
    for mod in ("dnaio", "xopen"):
        m = pytest.importorskip(mod)
        if not getattr(m, "__file__", None):
            pytest.skip("%s in sys.modules is a stand-in" % mod)
    from tests.golden.make_reference_golden import REFERENCE

    ref = str(REFERENCE)
    if os.path.isdir(os.path.join(ref, "mirge")) and ref not in sys.path:
        sys.path.append(ref)
    try:
        from mirge.libs.digest import baking  # noqa: the reference's own code
    except Exception as e:  # not installed / its other imports are missing
        pytest.skip("the reference's mirge.libs.digest is not importable here: %s" % e)
    return baking


@pytest.mark.parametrize("name", ["ref_case2_umi", "ref_case3_umi_dedup", "ref_case4_qiagen", "ref_case5_nextseq_cuts",
                                  "ref_case6_front_back_noindels"])
def test_reference_baking_with_the_real_tools_reproduces_the_golden_files(name, tmp_path):
    """The committed golden files were written by the reference's code with stand-ins answering for cutadapt / dnaio
    (tests/golden/standins.py), so for the third-party arithmetic they are circular.  Here the same reference code runs
    on the same inputs with the REAL packages: equal files turn those goldens -- and with them the oracle and the GPU
    path, which reproduce them byte for byte -- into pinned ones."""
    import json
    from pathlib import Path

    from tests.golden.make_reference_golden import reference_args

    baking = _reference_baking()
    import cutadapt
    d = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", name)
    meta = json.load(open(os.path.join(d, "counters.json")))
    ov = dict(meta["args"])
    if "adapters" in ov:
        ov["adapters"] = [tuple(a) for a in ov["adapters"]]
    ver = tuple(str(cutadapt.__version__).split(".")[:2])
    args = reference_args(cutadaptVersion=ver, **ov)  # (digest.py:111-113 switches on the installed version)
    files = [os.path.join(d, s + ".fastq") for s in meta["samples"]]
    df, src, trc, tru = baking(args, files, meta["samples"], Path(tmp_path))
    got = df.sort_index(kind="stable").to_csv()
    assert src == meta["sampleReadCounts"], (cutadapt.__version__, src)
    assert trc == meta["trimmedReadCounts"] and tru == meta["trimmedReadCountsUnique"], (cutadapt.__version__, trc, tru)
    assert got == open(os.path.join(d, "complete_set.csv")).read(), "complete_set.csv differs with cutadapt %s" % cutadapt.__version__
    for extra in sorted(os.listdir(d)):
        if extra.endswith("_umiCounts.csv"):
            assert sorted(open(os.path.join(str(tmp_path), extra)).read().splitlines()) == sorted(open(os.path.join(d, extra)).read().splitlines()), extra


def test_quality_trimmers_match_cutadapt():
    _real_cutadapt()
    from cutadapt.qualtrim import nextseq_trim_index, quality_trim_index

    try:
        from dnaio import Sequence
    except ImportError:
        from cutadapt.seqio import Sequence  # very old releases
    rng = np.random.default_rng(11)
    for _ in range(3000):
        n = int(rng.integers(0, 80))
        seq = "".join(rng.choice(B + ["G", "G"], n))
        q0, q1 = int(rng.integers(20, 41)), int(rng.integers(0, 30))
        qual = "".join(chr(33 + int(np.clip(v + rng.integers(-6, 7), 0, 41))) for v in np.linspace(q0, q1, n))
        c5, c3 = int(rng.integers(0, 30)), int(rng.integers(0, 35))
        assert tuple(quality_trim_index(qual, c5, c3, 33)) == po.quality_trim_index(qual, c5, c3, 33)
        assert nextseq_trim_index(Sequence("r", seq, qual), c3, 33) == po.nextseq_trim_index(seq, qual, c3, 33)


# ------------------------------------------------------------------------------------------------ bowtie

ROUND_OPTS = ["-n 0", "-n 1", "-v 1 -a --best --strata", "-v 0 -a --best --strata", "-n 1", "-n 1", "-n 1", "-n 0",
              "-5 1 -3 2 -v 2 --best", "-n 0"]  # manifoldAlign.py:85 (plus -f --norc -S --threads N)


def _bowtie():
    b, bb = shutil.which("bowtie"), shutil.which("bowtie-build")
    if not b or not bb:
        pytest.skip("bowtie / bowtie-build not on PATH")
    return b, bb


@pytest.mark.parametrize("rnd", range(10))
def test_round_hits_match_bowtie(rnd, tmp_path):
    bowtie, bowtie_build = _bowtie()
    rng = np.random.default_rng(100 + rnd)
    refs = ["".join(rng.choice(B, int(rng.integers(18, 26) if rnd in (0, 8, 9) else rng.integers(60, 140)))) for _ in range(60)]
    refs += [refs[0][:10] + "A" + refs[0][11:], refs[1]]  # a near-duplicate and an exact duplicate: multi-hit sets
    refs[5] = refs[5][:30] + "N" + refs[5][31:] if len(refs[5]) > 31 else refs[5]
    names = ["ref%d" % i for i in range(len(refs))]
    fa = tmp_path / "lib.fa"
    fa.write_text("".join(">%s\n%s\n" % (n, s) for n, s in zip(names, refs)))
    subprocess.run([bowtie_build, "-q", str(fa), str(tmp_path / "lib")], check=True, stdout=subprocess.DEVNULL)
    lib = po.Library(names, [r.upper() for r in refs])
    pol = po.ROUND_POLICIES[rnd]
    queries = []
    for _ in range(400):
        r = refs[int(rng.integers(len(refs)))]
        L = int(rng.integers(16, min(len(r), 45) + 1))
        o = int(rng.integers(0, len(r) - L + 1))
        q = list(r[o : o + L])
        for _m in range(int(rng.integers(0, 4))):
            p = int(rng.integers(L))
            q[p] = str(rng.choice(B))
        q = "".join(q)
        if pol.strip_polyT:
            q += "T" * int(rng.integers(3, 6))
        elif pol.trim5 or pol.trim3:
            q = "A" * pol.trim5 + q + "C" * pol.trim3
        queries.append(q.replace("N", "A"))
    queries = sorted(set(queries))
    sent = [(q, po.round_query(q, rnd)) for q in queries]
    sent = [(q, s) for q, s in sent if s]
    # round 3: the reference submits the sequence without its poly-T tail under the full sequence's name (manifoldAlign.py:118-126)
    fq = tmp_path / "q.fa"
    fq.write_text("".join(">%s\n%s\n" % (q, s if pol.strip_polyT else q) for q, s in sent))
    cmd = [bowtie, str(tmp_path / "lib"), str(fq)] + ROUND_OPTS[rnd].split() + ["-f", "--norc", "-S", "--threads", "2"]
    sam = subprocess.run(cmd, check=True, capture_output=True, text=True).stdout
    reported = {}
    for line in sam.splitlines():
        if line.startswith("@"):
            continue
        f = line.split("\t")
        if int(f[1]) & 4:
            reported.setdefault(f[0], [])
            continue
        nm = [int(x[5:]) for x in f[11:] if x.startswith("NM:i:")]
        reported.setdefault(f[0], []).append((names.index(f[2]), int(f[3]) - 1, nm[0] if nm else None))
    for q, s in sent:
        valid = po.hits(s, lib, pol)
        got = reported.get(q)
        assert got is not None, q
        if not valid:
            assert got == [], (rnd, q, got)
            continue
        assert got, (rnd, q, "bowtie found nothing; oracle:", valid[:3])
        best_mm = min(h[0] for h in valid)
        vset = {(h[1], h[2]): h[0] for h in valid}
        for ref, off, nm in got:
            assert (ref, off) in vset, (rnd, q, (ref, off), sorted(vset)[:5])
            if nm is not None:
                assert nm == vset[(ref, off)]
        if "--best" in ROUND_OPTS[rnd]:
            assert all(vset[(r_, o_)] == best_mm for r_, o_, _ in got), (rnd, q)
        if "-a" in ROUND_OPTS[rnd].split():
            assert {(r_, o_) for r_, o_, _ in got} == {k for k, v in vset.items() if v == best_mm}, (rnd, q)
        if len(valid) == 1:
            assert (got[-1][0], got[-1][1]) == po.canonical_pick(valid)[1:], (rnd, q)


def test_ebwt_decoder_against_a_real_bowtie_build(tmp_path):
    """mirge_b200/ebwt.py (names + sequences straight from .1/.3/.4.ebwt) on an index a real bowtie-build wrote, and
    against what the real bowtie-inspect prints for it -- the validation the decoder is fenced for
    (MIRGE_B200_TRUST_EBWT) until it has passed here once."""
    _, bowtie_build = _bowtie()
    inspect = shutil.which("bowtie-inspect")
    from mirge_b200 import ebwt

    rng = np.random.default_rng(21)
    seqs = ["".join(rng.choice(B, int(rng.integers(18, 900)))) for _ in range(120)]
    seqs[3] = seqs[3][:10] + "NNN" + seqs[3][13:]
    seqs[7] = "NN" + seqs[7]
    names = ["ref%d some description" % i if i % 4 == 0 else "ref%d" % i for i in range(len(seqs))]
    fa = tmp_path / "lib.fa"
    fa.write_text("".join(">%s\n%s\n" % (n, s) for n, s in zip(names, seqs)))
    subprocess.run([bowtie_build, "-q", str(fa), str(tmp_path / "lib")], check=True, stdout=subprocess.DEVNULL)
    got_names, got = ebwt.decode_index(str(tmp_path / "lib"))
    assert got_names == [n.split()[0] for n in names]
    if inspect:
        out = subprocess.run([inspect, str(tmp_path / "lib")], check=True, capture_output=True, text=True).stdout
        lib = po.read_fasta(out)
        assert [s.decode() for s in got] == lib.seqs and got_names == lib.names
    else:
        assert [s.decode() for s in got] == [s.rstrip("N") for s in seqs]
