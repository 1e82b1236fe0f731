"""Pins the CPU restatement of pcr.Simulate (tests/pcr_util.py, Tm from oracle/) on the expectations of
the reference's own tests: primers/pcr/example_test.go:10-36,58-69 and pcr_test.go:13-101."""
import json
import os

import pytest

import pcr_util as P


def test_reference_expectations():
    for seqs, circular, primers, ok in P.reference_cases():
        fr, err = P.simulate(seqs, 55.0, circular, primers)
        assert ok(fr, err), primers


def test_constants_equal_the_reference_test_files():
    """The strings of the reference's example_test.go / pcr_test.go, as tests/golden/make_pcr_goldens.py stored them."""
    g = json.load(open(os.path.join(os.path.dirname(__file__), "golden", "pcr_goldens.json")))
    assert P.FULL_AMPLICON == g["example_simulate_output"]
    assert P.GENE.decode() == g["example_gene"]
    assert P.BAD_FRAGMENT.decode() == g["example_bad_fragment"]
    assert P.CIRCULAR_TARGET == g["circular_target_fragment"]
    assert P.FULL_AMPLICON == g["issue279_want"]


def test_minimal_length_quirks():
    # the loop keeps the last length that FAILED the test: Tm(minimal primer) < target <= Tm(one base more)
    import oracle_ffi as o
    ml = P.minimal_length(P.FWD, 55.0)
    assert 7 <= ml < len(P.FWD)
    assert o.melting_temp(P.FWD[len(P.FWD) - ml:]) < 55.0 <= o.melting_temp(P.FWD[len(P.FWD) - ml - 1:])
    assert P.minimal_length(b"CTGCAGGTCGACTCTAG", 55.0) == 17           # whole primer below target: ignored (pcr.go:103)
    assert P.minimal_length(b"G" * 15 + b"C" * 15, 15.0) == 0            # the 7-mer (Tm 19.6) already reaches the target
    assert P.minimal_length(b"G" * 15 + b"C" * 15, 20.0) == 7            # ... and just misses this one
    # ADVICE r1: a GC-rich primer whose 15-nt suffix is already above the target still has a minimal part of 7..14 nt
    gc = b"GCGGCCGCGGGCCCGCGGCCGC"
    assert o.melting_temp(gc[-15:]) >= 55.0 and 7 <= P.minimal_length(gc, 55.0) < 15
    assert P.minimal_length(b"ACGTACG", 55.0) == 7                       # 7 nt is legal (pcr.go:35), whole primer below target
    with pytest.raises(IndexError):
        P.minimal_length(b"ACGT", 55.0)
