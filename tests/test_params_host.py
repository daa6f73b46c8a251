"""CPU tests of mirge_b200.params: the adapter specification subset, the flattened trim parameters (the product's
``stipulate()``), and -- when the read-only reference checkout is present -- the modifier pipeline held against the
list the reference's own ``stipulate(args)`` (mirge/libs/digest.py:59-101) builds for the same arguments."""
import os
import subprocess
import sys
import textwrap

import pytest

import mirge_b200  # noqa: F401
from mirge_b200 import abi
from mirge_b200 import params as P
from tests.golden import make_reference_golden as G

ILL_BACK = "TGGAATTCTCGGGTGCCAAGGAACTCCAG"
ILL_FRONT = "GTTCAGAGTTCTACAGTCCGACGATC"


def test_adapter_specification_language(tmp_path):
    """cutadapt's adapter specification language as it reaches stipulate() through -a / -g (parse.py:74-77)."""
    assert P.parse_adapter_spec("back", "illumina").sequence == ILL_BACK       # mirge/__main__.py:66-86
    assert P.parse_adapter_spec("front", "Illumina").sequence == ILL_FRONT
    assert P.parse_adapter_spec("back", "myname=acgu").sequence == "ACGT"      # name=, upper-casing, U -> T
    assert P.parse_adapter_spec("back", " ACGTN ").sequence == "ACGTN"
    w = lambda kind, spec: (lambda sp: (sp.where, sp.sequence, sp.params))(P.parse_adapter_spec(kind, spec))
    assert w("back", "ACGT$") == ("suffix", "ACGT", {})                        # anchored 3'
    assert w("front", "^ACGT") == ("prefix", "ACGT", {})                       # anchored 5'
    assert w("back", "ACGTX") == ("back_not_internal", "ACGT", {})
    assert w("front", "xxACGT") == ("front_not_internal", "ACGT", {})
    assert w("back", "AC{3}GT{2}") == ("back", "ACCCGTT", {})                  # x{n} repeats
    assert w("back", "n=ACGT;e=0.2;o=5") == ("back", "ACGT", {"max_error_rate": 0.2, "min_overlap": 5})
    assert w("back", "ACGT; max_error_rate = 0 ;noindels") == ("back", "ACGT", {"max_error_rate": 0, "indels": False})
    assert w("back", "...ACGT") == ("back", "ACGT", {})                        # -a ...ADAPTER: plain 3' adapter
    assert w("back", "ACGT...") == ("front", "ACGT", {})                       # -a ADAPTER...: plain 5' adapter
    assert w("front", "ACGT...") == ("front", "ACGT", {})
    fa = tmp_path / "adapters.fa"
    fa.write_text("# two adapters\n>first\nACGT\nACGT\n\n>second some text\n^TTTTGG;e=0.1\n")
    got = P.parse_adapter_specs("front", "file:%s" % fa)
    assert [(sp.where, sp.sequence, sp.params) for sp in got] == [("front", "ACGTACGT", {}), ("prefix", "TTTTGG", {"max_error_rate": 0.1})]
    for kind, spec in (("back", "file:/nonexistent/adapters.fa"), ("back", "^ACGT"), ("front", "ACGT$"), ("back", "XACGT"), ("front", "ACGTX"),
                       ("front", "^XACGT"), ("back", "ACGTX$"), ("back", "XXX"), ("back", ""), ("back", "ACGT;anywhere"),
                       ("back", "ACGT;foo=1"), ("back", "ACGT;e="), ("back", "ACGT;e=0.1;e=0.2"), ("back", "ACGT;e=2"), ("back", "ACGT;o=0"),
                       ("back", "ACGT;required"), ("back", "ACGT;optional"), ("back", "ACGT;indels;noindels"), ("back", "AC{GT"),
                       ("back", "{3}ACGT"), ("front", "...ACGT"),
                       ("back", "A" * (abi.MAX_ADAPTER_LEN + 1)), ("back", "ACGT-ACGT"), ("anywhere", "ACGT")):
        with pytest.raises(P.UnsupportedAdapterSpec):
            P.parse_adapter_specs(kind, spec)
    # per-adapter parameters reach the Aligner terms of that adapter only
    p = P.build_trim_params(P.TrimConfig(adapters=[("back", "ACGTACGTAC;e=0.3;o=7;noindels"), ("front", "^ACGTAC"), ("back", "TTTTTTTTX")]))
    a0, a1, a2 = p.adapters[0], p.adapters[1], p.adapters[2]
    assert (a0.where, a0.k, a0.min_overlap, a0.indel_cost, a0.max_err[10]) == (abi.WHERE["back"], 3, 7, 100000, 3)
    assert (a1.where, a1.k, a1.min_overlap, a1.indel_cost) == (abi.WHERE["prefix"], 0, 6, 1)      # anchored: the whole adapter
    assert (a2.where, a2.k, a2.min_overlap) == (abi.WHERE["back_not_internal"], 0, 3)
    assert [abi.WHERE[k] & 1 for k in ("back", "suffix", "back_not_internal", "front", "prefix", "front_not_internal")] == [0, 0, 0, 1, 1, 1]
    assert P.build_trim_params(P.TrimConfig(adapters=[("back", "ACGT")], match_read_wildcards=True)).adapters[0].wildcard_read == 1


def test_adapter_lists_beyond_the_bit_parallel_kernels(tmp_path):
    """A file: list of a whole kit: up to 16 adapters (a linked pair counts twice); more than four of them leave the
    bit-parallel kernels (one shared-memory match table per adapter) for the full-DP kernel."""
    fa = tmp_path / "kit.fa"
    seqs = ["ACGTACGTAC" + "ACGT"[i % 4] * 6 + "TTGCA"[: 1 + i % 5] for i in range(9)]
    fa.write_text("".join(">a%d\n%s\n" % (i, q) for i, q in enumerate(seqs)))
    p = P.build_trim_params(P.TrimConfig(adapters=[("back", "file:%s" % fa), ("back", "^GTTCAG...TGGAATTC")]))
    assert p.n_adapters == 11 and [bytes(p.adapters[i].ascii[: p.adapters[i].m]).decode() for i in range(9)] == seqs
    assert p.adapters[9].link == 11 | abi.LINK_BACK_OPTIONAL and p.adapters[10].link == abi.LINK_BACK_HALF
    with pytest.raises(RuntimeError):
        P.build_trim_params(P.TrimConfig(adapters=[("back", "ACGTACGT" + "ACGT"[i % 4] * (1 + i // 4)) for i in range(abi.MAX_ADAPTERS + 1)]))


def test_linked_adapter_specification():
    """"ADAPTER5...ADAPTER3" (docs/source/quick_start.md:208-220): a 5' half pointing at its 3' half in the flat adapter
    list.  -g: both halves required; -a: a half is required only when it is anchored; ;required / ;optional override."""
    sp = P.parse_adapter_spec("front", "TTAGGC...TGGAATTCTCGGGTGCCAAGGAACTCCAGT")
    assert (sp.where, sp.sequence, sp.sequence2, sp.where5, sp.where2, sp.front_required, sp.back_required) == \
        ("linked", "TTAGGC", "TGGAATTCTCGGGTGCCAAGGAACTCCAGT", "front", "back", True, True)
    p = P.build_trim_params(P.TrimConfig(adapters=[("back", "ACGTACGTAC"), ("front", "name=TTAGGC...ACGTTGCA")]))
    assert p.n_adapters == 3
    assert [p.adapters[i].where for i in range(3)] == [0, 1, 0]
    assert [p.adapters[i].link for i in range(3)] == [0, 3, abi.LINK_BACK_HALF]
    lk = lambda kind, spec: (lambda sp: (sp.where5, sp.where2, sp.front_required, sp.back_required))(P.parse_adapter_spec(kind, spec))
    assert lk("back", "^TTAGGC...ACGT") == ("prefix", "back", True, False)      # the documented -a form: anchored 5' half, optional 3' half
    assert lk("back", "TTAGGC...ACGT") == ("front", "back", False, False)
    assert lk("back", "TTAGGC...ACGT$") == ("front", "suffix", False, True)
    assert lk("front", "^TTAGGC...ACGTX") == ("prefix", "back_not_internal", True, True)
    assert lk("front", "TTAGGC;optional...ACGT;e=0.2") == ("front", "back", False, True)
    assert lk("back", "^TTAGGC...ACGT;required") == ("prefix", "back", True, True)
    sp = P.parse_adapter_spec("front", "TTAGGC;o=4...ACGT;e=0.2")
    assert (sp.params, sp.params2) == ({"min_overlap": 4}, {"max_error_rate": 0.2})
    p = P.build_trim_params(P.TrimConfig(adapters=[("back", "^TTAGGC...ACGTTGCA;e=0.2")]))
    assert [p.adapters[i].where for i in range(2)] == [abi.WHERE["prefix"], abi.WHERE["back"]]
    assert [p.adapters[i].link for i in range(2)] == [2 | abi.LINK_BACK_OPTIONAL, abi.LINK_BACK_HALF]
    assert (p.adapters[0].k, p.adapters[1].k) == (0, 1)
    for kind, spec in (("front", "TTAGGC...illumina"), ("front", "A...C...G"), ("front", "TTAGGC$...ACGT"), ("front", "TTAGGC...^ACGT"),
                       ("front", "TTAGGC;required;optional...ACGT")):
        with pytest.raises(P.UnsupportedAdapterSpec):
            P.parse_adapter_spec(kind, spec)
    with pytest.raises(P.UnsupportedAdapterSpec):
        P.build_trim_params(P.TrimConfig(adapters=[("front", "TTAGGC...AACTGTAGGCACCATCAAT")], qiagenumi=True, uniq_mol_ids="0,12"))


def test_parse_cutoffs_doctests():  # digest.py:19-35
    assert P.parse_cutoffs("5") == [0, 5] or tuple(P.parse_cutoffs("5")) == (0, 5)
    assert tuple(P.parse_cutoffs("6,7")) == (6, 7)
    with pytest.raises(Exception):
        P.parse_cutoffs("1,2,3")


def kinds(p):
    return [p.mod_kind[i] for i in range(p.n_mods)]


def test_modifier_order_and_parameters():
    cfg = P.TrimConfig(adapters=[("back", "illumina")], nextseq_trim=20, quality_cutoff="5,15", quality_base=64, trim_n=True, cut=[2, -3],
                       times=2, minimum_length=14, error_rate=0.12, overlap=3)
    p = P.build_trim_params(cfg)
    assert kinds(p) == [abi.MOD_NEXTSEQ, abi.MOD_QUALITY, abi.MOD_ADAPTER, abi.MOD_NEND, abi.MOD_CUT, abi.MOD_CUT]  # digest.py:87-99
    assert (p.mod_a[0], p.mod_b[0]) == (20, 64)
    assert (p.mod_a[1], p.mod_b[1], p.mod_c[1]) == (5, 15, 64)
    assert (p.mod_a[4], p.mod_a[5]) == (2, -3)
    assert p.times == 2 and p.min_len == 14 and p.n_adapters == 1
    assert P.trim_slots(p) == 6                                               # HEAD: one emission slot per modifier
    assert P.trim_slots(P.build_trim_params(P.TrimConfig(adapters=[("back", "illumina")], count_mode="release"))) == 1
    a = p.adapters[0]
    assert a.m == 29 and a.k == int(0.12 * 29) and a.min_overlap == 3 and a.indel_cost == 1 and a.wildcard_ref == 0
    # cutadapt compares cost <= length * rate in double: the integer table must be its floor for every length
    for rate in (0.0, 0.05, 0.1, 0.12, 0.2, 0.34, 0.5):
        ad = P.build_adapter(P.parse_adapter_spec("back", ILL_BACK), P.TrimConfig(adapters=[("back", ILL_BACK)], error_rate=rate))
        for L in range(abi.MAX_ADAPTER_LEN + 1):
            assert all((c <= L * rate) == (c <= ad.max_err[L]) for c in range(0, 40)), (rate, L)
    # a cut of zero adds no modifier (digest.py:51-53); no quality cut-off, no adapter: empty pipeline
    assert kinds(P.build_trim_params(P.TrimConfig(adapters=[], quality_cutoff=None, cut=[0]))) == []


def test_wildcard_adapters_and_rejections():
    cfg = P.TrimConfig(adapters=[("back", "ACGTNNACGR")])
    a = P.build_trim_params(cfg).adapters[0]
    assert a.wildcard_ref == 1 and a.effective_length == 8 and [a.n_counts[i] for i in range(11)] == [0, 0, 0, 0, 0, 1, 2, 2, 2, 2, 2]
    with pytest.raises(P.UnsupportedAdapterSpec):
        P.build_trim_params(P.TrimConfig(adapters=[("back", "NNNN")]))                      # cutadapt: only N wildcards
    with pytest.raises(P.UnsupportedAdapterSpec):
        P.build_trim_params(P.TrimConfig(adapters=[("back", "ACGTN")], match_adapter_wildcards=False))
    with pytest.raises(RuntimeError):
        P.build_trim_params(P.TrimConfig(adapters=[("back", "ACGT")], cut=[1, 2, 3]))          # digest.py:47-48
    with pytest.raises(RuntimeError):
        P.build_trim_params(P.TrimConfig(adapters=[("back", "ACGT")], cut=[1, 2]))             # digest.py:49-50
    with pytest.raises(RuntimeError):
        P.build_trim_params(P.TrimConfig(adapters=[("back", "ACGT")], qiagenumi=True))         # needs -umi
    with pytest.raises(RuntimeError):
        P.build_trim_params(P.TrimConfig(adapters=[("back", "ACGT")], action="mask"))
    q = P.build_trim_params(P.TrimConfig(adapters=[("back", "AACTGTAGGCACCATCAAT")], qiagenumi=True, uniq_mol_ids="0,12"))
    assert q.umi_mode == abi.UMI_QIAGEN and q.qia_adapter_len == 19 and (q.umi5, q.umi3) == (0, 12) and P.trim_slots(q) == 1


CHILD = textwrap.dedent(
    r"""
    import json, sys
    sys.path.insert(0, %(root)r)
    from tests.golden import make_reference_golden as G, standins
    standins.install(G.REFERENCE)
    from mirge.libs.digest import stipulate   # the reference's own code (third-party classes are the stand-ins)
    out = []
    for ov in json.loads(sys.argv[1]):
        if "adapters" in ov:
            ov["adapters"] = [tuple(a) for a in ov["adapters"]]
        mods = stipulate(G.reference_args(**ov))
        row = []
        for m in mods:
            n = type(m).__name__
            if n == "NextseqQualityTrimmer": row.append(["nextseq", m.cutoff, m.base])
            elif n == "QualityTrimmer": row.append(["quality", m.cf, m.cb, m.base])
            elif n == "AdapterCutter": row.append(["adapter", m.times, [[a.where, a.sequence] for a in m.adapters]])
            elif n == "NEndTrimmer": row.append(["nend"])
            elif n == "UnconditionalCutter": row.append(["cut", m.length])
            else: row.append([n])
        out.append(row)
    print(json.dumps(out))
    """
)


STIPULATE_GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "reference_stipulate.json")


def product_pipeline(ov):
    """The modifier rows of build_trim_params for one set of argument overrides, in the CHILD script's format."""
    ov = dict(ov)
    if "adapters" in ov:
        ov["adapters"] = [tuple(a) for a in ov["adapters"]]
    tp = P.build_trim_params(P.TrimConfig.from_args(G.reference_args(**ov)))
    names = {abi.MOD_NEXTSEQ: "nextseq", abi.MOD_QUALITY: "quality", abi.MOD_ADAPTER: "adapter", abi.MOD_NEND: "nend", abi.MOD_CUT: "cut"}
    rows = []
    for i in range(tp.n_mods):
        k = names[tp.mod_kind[i]]
        if k == "nextseq":
            rows.append([k, tp.mod_a[i], tp.mod_b[i]])
        elif k == "quality":
            rows.append([k, tp.mod_a[i], tp.mod_b[i], tp.mod_c[i]])
        elif k == "adapter":
            rows.append([k, tp.times, [["back" if tp.adapters[a].where == 0 else "front",
                                        bytes(tp.adapters[a].ascii[: tp.adapters[a].m]).decode()] for a in range(tp.n_adapters)]])
        elif k == "cut":
            rows.append([k, tp.mod_a[i]])
        else:
            rows.append([k])
    return rows


def test_pipeline_equals_the_reference_stipulate(tmp_path):
    """build_trim_params against the modifier list the reference's stipulate() builds for six argument sets, stored in
    tests/golden/reference_stipulate.json (recorded from the product at 78fb5a6, whose rows this comparison had found equal to
    the reference's own).  With a reference checkout at $MIRGE_REFERENCE the reference's stipulate() is run as well (in a
    child process: it needs the stand-ins of tests/golden/standins.py) and held against the stored rows."""
    import json

    with open(STIPULATE_GOLDEN) as f:
        golden = json.load(f)
    cases, ref = golden["cases"], golden["rows"]
    for ov, row in zip(cases, ref):
        assert product_pipeline(ov) == row, (ov, row)
    if G.REFERENCE.exists():
        script = tmp_path / "child.py"
        script.write_text(CHILD % {"root": os.path.dirname(os.path.dirname(os.path.abspath(__file__)))})
        p = subprocess.run([sys.executable, str(script), json.dumps(cases)], capture_output=True, text=True, timeout=300)
        assert p.returncode == 0, p.stderr[-2000:]
        assert json.loads(p.stdout.strip().splitlines()[-1]) == ref
