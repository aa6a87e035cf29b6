"""Scheme grammar / adapter table / CLI naming against pinned values and tests/golden/reference_common.json, written by
scripts/make_golden_common.py.  That file's "source" field says what it holds: the values of the original cutseq's
cutseq/common.py, or (as committed now, the original not having been available) a snapshot of cutseq_b200.common that
only catches changes of its own behaviour."""

import json
import os

import pytest

from cutseq_b200 import common, run
from tests.helpers import GOLD


def ref_common():
    with open(os.path.join(GOLD, "reference_common.json")) as f:
        return json.load(f)


def test_takarav3_parts():
    b = common.BarcodeConfig(common.BUILDIN_ADAPTERS["TAKARAV3"])
    assert b.p5.fw == "ACACGACGCTCTTCCGATCT" and b.p5.rc == "AGATCGGAAGAGCGTCGTGT"
    assert b.p7.fw == "AGATCGGAAGAGCACACGTC" and b.p7.rc == "GACGTGTGCTCTTCCGATCT"
    assert (b.mask5.len, b.mask3.len, b.umi5.len, b.umi3.len, b.inline5.len, b.inline3.len) == (3, 6, 0, 8, 0, 0)
    assert b.strand == "-"


def test_table_has_18_entries():
    assert len(common.BUILDIN_ADAPTERS) == 18
    assert list(common.BUILDIN_ADAPTERS)[0] == "SMALLRNA"


@pytest.mark.parametrize("scheme", ["ACGT>ACGTJUNK", "acgt(tt)NNXX<XN(gg)acgt", "A-C", "ACGT(AC)>(GT)TTTT"])
def test_grammar_accepts(scheme):
    b = common.BarcodeConfig(scheme)
    assert b.p5.len > 0 and b.p7.len > 0


@pytest.mark.parametrize("scheme", ["ACGTXN>ACGT", "ACGT()>ACGT", ">ACGT", "ACGT>", "ACGT>NXACGT", ""])
def test_grammar_rejects(scheme):
    with pytest.raises(SystemExit) as e:
        common.BarcodeConfig(scheme)
    assert e.value.code == 1


def test_remove_fq_suffix():
    assert common.remove_fq_suffix("x/y/input_R1.fq.gz") == "x/y/input"
    assert common.remove_fq_suffix("a_R2_001.fastq.gz") == "a"
    assert common.remove_fq_suffix("a.fastq") == "a"
    assert common.remove_fq_suffix("plain") == "plain"
    assert common.remove_fq_suffix("s_R1.fq") == "s"


def test_against_reference_common():
    ref = ref_common()
    assert list(common.BUILDIN_ADAPTERS.items()) == [tuple(kv) for kv in ref["adapters"]]
    assert len(ref["schemes"]) == len(ref["adapters"]) + 4
    for s, want in ref["schemes"].items():
        a = common.BarcodeConfig(s)
        assert a.to_dict() == want["to_dict"], s
        for part, (rc, text) in want["parts"].items():
            assert getattr(a, part).rc == rc and repr(getattr(a, part)) == text, (s, part)
    assert len(ref["remove_fq_suffix"]) == 7 and len(ref["reverse_complement"]) == 3
    for f, stem in ref["remove_fq_suffix"].items():
        assert common.remove_fq_suffix(f) == stem, f
    for s, rc in ref["reverse_complement"].items():
        assert common.reverse_complement(s) == rc, s


def test_list_adapters_output_matches_reference(capsys):
    common.print_builtin_adapters()
    assert capsys.readouterr().out == ref_common()["list_adapters"]


def test_cli_defaults_and_naming(capsys):
    p = run.build_parser()
    a = p.parse_args(["-A", "takarav3", "in_R1.fq.gz", "in_R2.fq.gz"])
    assert (a.min_quality, a.min_length, a.threads, a.force_trim_min_length, a.conditional_cutter) == (20, 20, 1, 50, True)
    assert run.resolve_scheme(a) == common.BUILDIN_ADAPTERS["TAKARAV3"]
    assert run._default_outputs(None, a.input_file, None, "trimmed") == ["in_trimmed_R1.fastq.gz", "in_trimmed_R2.fastq.gz"]
    assert run._default_outputs(None, a.input_file, "pre", "short") == ["pre_short_R1.fastq.gz", "pre_short_R2.fastq.gz"]
    with pytest.raises(SystemExit):
        run._default_outputs(["only_one"], a.input_file, None, "trimmed")
    b = p.parse_args(["-a", "acgt xx > acgt", "--no-conditional-cutter", "x.fq"])
    assert run.resolve_scheme(b) == "ACGTXX>ACGT" and b.conditional_cutter is False


def test_dry_run_lists_program(capsys):
    run.main(["-A", "TAKARAV3", "--trim-polyA", "-n", "x.fq"])
    out = capsys.readouterr().out
    assert "Step 1: SuffixRemover('.1')" in out and "NonInternalFrontAdapter" in out and "QualityTrimmer(cutoff_front=0, cutoff_back=20" in out


def test_every_builtin_scheme_compiles_to_a_program():
    """All 18 built-in schemes, single-end and paired, with and without the optional steps: the op program follows the
    fixed order of run.py:326-426 / 533-731 (strip, 5' adapter, 3' adapter, inline, UMI, rename, mask, polyA, qtrim)."""
    from cutseq_b200 import _abi as A
    from cutseq_b200 import program, run
    from cutseq_b200.common import BUILDIN_ADAPTERS, BarcodeConfig

    for name in BUILDIN_ADAPTERS:
        for extra in ([], ["--trim-polyA"], ["--trim-polyA-wo-direction", "--no-conditional-cutter", "--ensure-inline-barcode", "--auto-rc"]):
            args = run.build_parser().parse_args(["-A", name] + extra + ["a.fq", "b.fq"])
            bc = BarcodeConfig(run.resolve_scheme(args))
            settings = run.settings_from_args(args)
            for prog in (program.compile_single(bc, settings), program.compile_paired(bc, settings)):
                for ops in ([prog.ops_r1, prog.ops_r2] if prog.paired else [prog.ops_r1]):
                    kinds = [op.kind for op in ops]
                    assert kinds[0] == A.OP_STRIP_SUFFIX and kinds.count(A.OP_RENAME) == 1 and kinds.count(A.OP_QTRIM) == 1
                    assert len(ops) <= A.CSQ_MAX_OPS
                    # the two full-adapter searches come first among the alignments: 5' (rightmost front), then 3' (back)
                    aligns = [op for op in ops if op.kind == A.OP_ALIGN]
                    assert aligns[0].adapter_kind == A.AD_RIGHTMOST_FRONT and aligns[0].min_overlap == 10
                    assert aligns[1].adapter_kind in (A.AD_BACK, A.AD_BACK_ANYWHERE) and aligns[1].min_overlap == 3
                    # nothing but REVCOMP may follow the quality trimmer
                    q = kinds.index(A.OP_QTRIM)
                    assert all(k == A.OP_REVCOMP for k in kinds[q + 1:])
                    # the rename sits between the UMI cuts and the mask cuts: it is preceded by at most the UMI cuts
                    assert kinds.index(A.OP_RENAME) > kinds.index(A.OP_ALIGN)
                assert prog.describe()
