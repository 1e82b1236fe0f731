"""GPU parity: libpolyb200 (through the C ABI) vs the CPU oracle, bit-exact.

Mirrors the reference's own tests for the path (search/mash/mash_test.go:9-62,
example_test.go:9-22) and adds seeded batches at sizes the oracle finishes in seconds,
the committed goldens, and size-independent properties at BASELINE scale.
"""
import json
import os

import numpy as np
import pytest

from poly_b200 import mash, synth

pytestmark = pytest.mark.gpu

A = "ATGCGATCGATCGATCGATCGATCGATCGATCGATCGATCGATCGATCGATCGATCGATCGA"
B = "ATCGATCGATCGATCGATCGATCGATCGATCGATCGAATGCGATCGATCGATCGATCGATCG"
GOLD = json.load(open(os.path.join(os.path.dirname(__file__), "golden", "survey_goldens.json")))


def test_reference_TestMash(gpu):
    """search/mash/mash_test.go:9-62, statement for statement."""
    f1 = mash.New(17, 10); f1.Sketch(A)
    f2 = mash.New(17, 9); f2.Sketch(A)
    assert f1.Distance(f2) == 0
    assert f2.Distance(f1) == 0
    spoof = mash.New(17, 10); spoof.Sketches[0] = 0
    assert f1.Distance(spoof) == 1
    spoof = mash.New(17, 9)
    assert f1.Distance(spoof) == 1
    f1 = mash.New(17, 10); f1.Sketch(A)
    f2 = mash.New(17, 5); f2.Sketch(B)
    d = f1.Distance(f2)
    assert 0.19 < d < 0.21 and d == 0.19999999999999996
    f1 = mash.New(17, 10); f1.Sketch(B)
    f2 = mash.New(17, 5); f2.Sketch(A)
    assert f1.Distance(f2) == 0


def test_reference_ExampleMash(gpu):
    f1 = mash.New(17, 10); f1.Sketch(A)
    f2 = mash.New(17, 9); f2.Sketch(A)
    assert repr(f1.Distance(f2)) in ("0.0",)  # Go prints 0


def test_survey_golden_sketches(gpu):
    g = GOLD["mash"]
    m = mash.New(17, 10); m.Sketch(A)
    assert [int(x) for x in m.Sketches] == [int(x, 16) for x in g["A_k17_s10"]]
    m = mash.New(17, 5); m.Sketch(B)
    assert [int(x) for x in m.Sketches] == [int(x, 16) for x in g["B_k17_s5"]]
    m = mash.New(17, 10); m.Sketch(B)
    assert [int(x) for x in m.Sketches] == [int(x, 16) for x in g["B_k17_s10"]]


def test_cfg1_bit_exact_and_checksums(gpu, oracle):
    """BASELINE configs[0]: 1k x 150 bp, k=21, s=1000 (fill regime, fast TMA path)."""
    n, L, k, s = 1000, 150, 21, 1000
    reads = synth.independent_reads(n, L)
    got = mash.sketch_uniform(reads, n, L, k, s)
    rc, want = oracle.sketch_batch(reads, synth.uniform_offsets(n, L), k, s, variant=0)
    assert rc == 0
    assert got.shape == (n, L - k)
    assert np.array_equal(got, want[:, : L - k])
    assert not want[:, L - k:].any()
    c = GOLD["cfg1"]
    assert synth.fnv1a64(got) == int(c["fnv_compact"], 16)
    padded = np.zeros((n, s), np.uint32); padded[:, : L - k] = got
    assert synth.fnv1a64(padded) == int(c["fnv_padded"], 16)
    assert int(got.astype(np.uint64).sum()) == int(c["sum"], 16)


@pytest.mark.parametrize("k", [11, 13, 15, 16, 17, 19, 21, 23, 24, 25, 27, 29, 31, 32])
@pytest.mark.parametrize("L", [64, 150, 151, 100])
def test_uniform_fast_path_all_instantiated_k(gpu, oracle, k, L):
    n, s = 32 * 9 + 5, 4096  # tiles + a ragged remainder that takes the generic kernel
    reads = synth.independent_reads(n, L, first_read=7)
    got = mash.sketch_uniform(reads, n, L, k, s)
    rc, want = oracle.sketch_batch(reads, synth.uniform_offsets(n, L), k, s, variant=1)
    assert np.array_equal(got, want[:, : max(L - k, 0)])


@pytest.mark.parametrize("k", [0, 1, 2, 3, 4, 5, 7, 11, 13, 20, 22, 33, 40, 64])
def test_generic_k(gpu, oracle, k):
    n, L, s = 77, 97, 500
    rng = np.random.default_rng(k)
    reads = rng.integers(0, 256, n * L, dtype=np.uint8)  # arbitrary bytes are legal (mash.go:74-76)
    got = mash.sketch_uniform(reads, n, L, k, s)
    rc, want = oracle.sketch_batch(reads, synth.uniform_offsets(n, L), k, s, variant=1)
    assert np.array_equal(got, want[:, : got.shape[1]])


def test_ragged_batch_mixed_regimes(gpu, oracle):
    """Empty reads, reads shorter than k, fill regime and select regime in one batch."""
    rng = np.random.default_rng(1)
    k, s = 21, 64
    lens = [0, 1, 20, 21, 22, 23, 50, 84, 85, 86, 150, 300, 1000, 2500, 64 + 21, 63 + 21] + list(rng.integers(0, 400, 100))
    seqs = [bytes(rng.choice(list(b"ACGTNacgt"), size=int(l)).astype(np.uint8)) for l in lens]
    bases, offsets = mash.flatten(seqs)
    out, count, status = mash.sketch_arrays(bases, offsets, k, s, pad_zero=True)
    rc, want = oracle.sketch_batch(bases, offsets, k, s, variant=0)
    assert rc == 0 and not status.any()
    assert np.array_equal(out, want)
    assert np.array_equal(count, np.minimum(np.maximum(np.array(lens) - k, 0), s))
    # and through the object API
    ms = mash.SketchBatch(seqs, k, s)
    for m, w in zip(ms, want):
        assert np.array_equal(m.Sketches, w)


def test_select_regime_duplicates_and_ties(gpu, oracle):
    """Bottom-s is a MULTISET (duplicates kept, SURVEY 8a a3): low-complexity reads."""
    rng = np.random.default_rng(2)
    for k, s, L in [(17, 10, 62), (4, 50, 4000), (31, 2000, 10000), (8, 1000, 3000), (21, 1, 60), (5, 300, 20000)]:
        seqs = [bytes(rng.choice(list(b"AC"), size=L).astype(np.uint8)) for _ in range(5)]
        seqs.append(b"A" * L)
        bases, offsets = mash.flatten(seqs)
        out, count, status = mash.sketch_arrays(bases, offsets, k, s)
        for i, q in enumerate(seqs):
            o = oracle.OracleMash(k, s)
            rc = o.Sketch(q, faithful=(L <= 4000))
            if rc != 0:
                assert status[i] == 1
                continue
            assert status[i] == 0 and count[i] == min(max(L - k, 0), s)
            assert np.array_equal(out[i, : count[i]], o.Sketches[: count[i]]), (k, s, L, i)


def test_select_regime_long_reads_with_pruning(gpu, oracle):
    """Reads far longer than the candidate buffer: chunked streaming, admission limit, repeated exact
    prunes; ragged lengths at arbitrary byte alignment; low-complexity reads for ties."""
    rng = np.random.default_rng(31)
    for k, s in [(21, 1000), (31, 2000), (16, 64), (32, 3), (13, 1), (24, 5000), (20, 300)]:
        lens = [int(x) for x in rng.integers(30_000, 120_000, 4)] + [4224 + k, 4225 + k, 2 * 4224 + k + 1, s + k, s + k + 1]
        seqs = [bytes(rng.choice(list(b"ACGT"), size=l).astype(np.uint8)) for l in lens]
        seqs.append(bytes(rng.choice(list(b"AC"), size=70_001).astype(np.uint8)))
        seqs.append(b"ACG" * 20_000)
        if s == 1000:  # a genome-sized sequence: one row spread over many work items of the threshold walk
            seqs.append(bytes(rng.choice(list(b"ACGT"), size=2_500_003).astype(np.uint8)))
            seqs += [bytes(rng.choice(list(b"ACGT"), size=int(l)).astype(np.uint8)) for l in rng.integers(0, 3000, 40)]
        bases, offsets = mash.flatten(seqs)
        out, count, status = mash.sketch_arrays(bases, offsets, k, s)
        for i, q in enumerate(seqs):
            o = oracle.OracleMash(k, s)
            rc = o.Sketch(q, faithful=False)
            if rc != 0:
                assert status[i] == 1, (k, s, i)
                continue
            cnt = min(max(len(q) - k, 0), s)
            assert status[i] == 0 and count[i] == cnt, (k, s, i)
            assert np.array_equal(out[i, :cnt], o.Sketches[:cnt]), (k, s, i, len(q))


def test_cfg3_shape_sample_golden(gpu, oracle):
    """8 family reads of the cfg3 shape (10 kbp, k=31, s=2000, R=4): SURVEY 8d goldens."""
    n, L, k, s = 8, 10000, 31, 2000
    reads = synth.family_reads(n, L, family=4)
    got = mash.sketch_uniform(reads, n, L, k, s)
    c = GOLD["cfg3_sample"]
    assert [hex(int(x)) for x in got[0, :3]] == c["first3"]
    assert hex(int(got[0, 1999])) == c["last"]
    assert (np.diff(got.astype(np.int64), axis=1) >= 0).all()
    assert synth.fnv1a64(got) == int(c["fnv"], 16)
    same, dist = mash.distance_block(got)
    assert [int(x) for x in same[0]] == c["row0"]
    rc, want = oracle.sketch_batch(reads, synth.uniform_offsets(n, L), k, s, variant=1)
    assert np.array_equal(got, want)


def test_sketch_on_non_fresh_mash_keeps_tail(gpu, oracle):
    """mash.go:81-84 only overwrites the first L-k slots when L-k < s."""
    m = mash.New(21, 1000); o = oracle.OracleMash(21, 1000)
    long = bytes(synth.independent_reads(1, 1500))
    short = bytes(synth.independent_reads(1, 150, first_read=3))
    for q in (long, short):
        m.Sketch(q); o.Sketch(q)
        assert np.array_equal(m.Sketches, o.Sketches)
    assert m.Sketches[500] != 0  # tail of the previous (sorted) sketch survives


def test_panics_small_sketch_sizes(gpu, oracle):
    """sketchSize in {0,1}: mash.go:96-98 indexes Sketches[-1]."""
    seq = bytes(synth.independent_reads(1, 100))
    for s in (0, 1):
        o = oracle.OracleMash(21, s)
        rc = o.Sketch(seq)
        m = mash.New(21, s)
        if rc != 0:
            with pytest.raises(IndexError):
                m.Sketch(seq)
        else:
            m.Sketch(seq)
            assert np.array_equal(m.Sketches, o.Sketches)
    # s == 1 without panic: first hash is the minimum -> craft by trying reads
    found = False
    for r in range(400):
        q = bytes(synth.independent_reads(1, 24, first_read=r))
        o = oracle.OracleMash(21, 1)
        if o.Sketch(q) == 0:
            m = mash.New(21, 1); m.Sketch(q)
            assert np.array_equal(m.Sketches, o.Sketches)
            found = True
            break
    assert found
    with pytest.raises(IndexError):
        mash.New(17, 0).Distance(mash.New(17, 5))
    with pytest.raises(IndexError):
        mash.New(17, -1)


def test_pairs_literal_semantics_unsorted_and_mixed_sizes(gpu, oracle):
    """Similarity on unsorted (n < s) sketches follows the literal walk + early-out."""
    rng = np.random.default_rng(3)
    ms, os_ = [], []
    specs = [(21, 1000, 150), (21, 100, 150), (21, 129, 150), (21, 130, 151), (17, 10, 62), (17, 9, 62), (17, 5, 62), (21, 50, 5000), (21, 64, 5000)]
    for (k, s, L) in specs:
        for rep in range(2):
            q = bytes(synth.independent_reads(1, L, first_read=rep))
            m = mash.New(k, s); m.Sketch(q); ms.append(m)
            o = oracle.OracleMash(k, s); o.Sketch(q); os_.append(o)
            assert np.array_equal(m.Sketches, o.Sketches)
    # hand-made arrays: random unsorted, with zeros, equal values
    for s in (1, 2, 7, 40):
        for rep in range(3):
            m = mash.New(5, s); m.Sketches[:] = rng.integers(0, 12, s); ms.append(m)
            o = oracle.OracleMash(5, s); o.Sketches[:] = m.Sketches; os_.append(o)
    n = len(ms)
    pairs = np.array([(i, j) for i in range(n) for j in range(n)], dtype=np.uint32)
    same, sim, dist = mash.similarity_pairs(ms, pairs)
    for p, (i, j) in enumerate(pairs):
        w_same, w_sim = os_[i].SimilarityCount(os_[j])
        assert same[p] == w_same and sim[p] == w_sim and dist[p] == os_[i].Distance(os_[j]), (i, j)
    # identical 150-bp reads have reference Distance 1.0 at k=21, s=1000 (SURVEY "READ THIS FIRST")
    assert ms[0].Distance(ms[0]) == 1.0


def test_distance_block_matches_pairs_and_oracle(gpu, oracle):
    n, L, k, s = 24, 3000, 21, 256
    reads = synth.family_reads(n, L, family=6)
    sk = mash.sketch_uniform(reads, n, L, k, s)
    same, dist = mash.distance_block(sk)
    for i in range(n):
        for j in range(n):
            oi = oracle.OracleMash(k, s); oi.Sketches[:] = sk[i]
            oj = oracle.OracleMash(k, s); oj.Sketches[:] = sk[j]
            c, _ = oi.SimilarityCount(oj)
            assert same[i, j] == c and dist[i, j] == oi.Distance(oj)
    assert same.max() == s and (same == same.T).all()
    # unsorted (fill-regime, zero padded) sketches through the same block kernel
    reads = synth.independent_reads(16, 150)
    out, _, _ = mash.sketch_arrays(reads, synth.uniform_offsets(16, 150), 21, 200, pad_zero=True)
    out[3] = out[2]
    same, dist = mash.distance_block(out)
    for i in range(16):
        for j in range(16):
            oi = oracle.OracleMash(21, 200); oi.Sketches[:] = out[i]
            oj = oracle.OracleMash(21, 200); oj.Sketches[:] = out[j]
            assert same[i, j] == oi.SimilarityCount(oj)[0] and dist[i, j] == oi.Distance(oj)
    # row block
    s2, d2 = mash.distance_block(out, 5, 11)
    assert np.array_equal(s2, same[5:11]) and np.array_equal(d2, dist[5:11])


def test_full_size_properties_cfg2_slice(gpu, oracle):
    """BASELINE cfg2 shape at 2M reads (device path via host API): spot-check rows against
    the oracle, and a checksum-of-checksums that is independent of chunking."""
    n, L, k, s = 2_000_000, 150, 21, 1000
    reads = synth.independent_reads(n, L)
    got = mash.sketch_uniform(reads, n, L, k, s)
    idx = np.r_[0:64, n // 2 - 32: n // 2 + 32, n - 64: n, np.random.default_rng(5).integers(0, n, 512)]
    sub = np.concatenate([reads[i * L:(i + 1) * L] for i in idx])
    rc, want = oracle.sketch_batch(sub, synth.uniform_offsets(len(idx), L), k, s, variant=1)
    assert np.array_equal(got[idx], want[:, : L - k])
    # chunk-independence: the same reads sketched in two halves
    h1 = mash.sketch_uniform(reads[: (n // 2) * L], n // 2, L, k, s)
    assert np.array_equal(h1, got[: n // 2])
    # shift property: read i+1 of a sliding set shares k-mer hashes with read i
    one = reads[: L + 1]
    a = mash.sketch_uniform(np.ascontiguousarray(one[:L]), 1, L, k, s)[0]
    b = mash.sketch_uniform(np.ascontiguousarray(one[1:]), 1, L, k, s)[0]
    assert np.array_equal(a[1:], b[:-1])


def _oracle_same_matrix(oracle, sk, rows):
    n, s = sk.shape
    out = np.zeros((len(rows), n), np.uint32)
    for a, i in enumerate(rows):
        oi = oracle.OracleMash(0, s); oi.Sketches[:] = sk[i]
        for j in range(n):
            oj = oracle.OracleMash(0, s); oj.Sketches[:] = sk[j]
            out[a, j] = oi.SimilarityCount(oj)[0]
    return out


def test_distance_join_multiset_and_skew(gpu, oracle):
    """All-ascending inputs take the inverted-index join (distance_join.cu): duplicates inside a
    sketch (multiset min-count), identical sketches, values piled into one bucket, row blocks;
    and the same sets with one non-ascending row appended take the pairwise kernel, which must
    agree with the oracle on the ascending rows as well."""
    rng = np.random.default_rng(21)
    cases = []
    # (a) low-complexity reads: many repeated k-mers -> duplicate hashes inside each sketch
    seqs = [bytes(rng.choice(list(b"AC"), size=600).astype(np.uint8)) for _ in range(20)] + [b"A" * 600, b"AC" * 300]
    bases, off = mash.flatten(seqs)
    out, cnt, st = mash.sketch_arrays(bases, off, 6, 128)
    assert (cnt == 128).all()
    cases.append(out)
    # (b) hand-made ascending multisets over a tiny value range (heavy ties, one hot bucket)
    cases.append(np.sort(rng.integers(0, 9, (40, 33)), axis=1).astype(np.uint32))
    # (c) identical sketches + values at both ends of the 32-bit range
    x = np.sort(rng.integers(0, 2 ** 32, (1, 64), dtype=np.uint64), axis=1).astype(np.uint32)
    y = np.concatenate([np.repeat(x, 30, 0), np.sort(rng.integers(0, 2 ** 32, (10, 64), dtype=np.uint64), axis=1).astype(np.uint32)])
    y[5, 0] = 0; y[6, -1] = 0xFFFFFFFF
    cases.append(np.sort(y, axis=1))
    for sk in cases:
        n = len(sk)
        want = _oracle_same_matrix(oracle, sk, range(n))
        same, dist = mash.distance_block(sk)
        assert np.array_equal(same, want)
        assert np.array_equal(dist, 1 - want / float(sk.shape[1]))
        s2, _ = mash.distance_block(sk, 3, n - 2)
        assert np.array_equal(s2, want[3:n - 2])
    for sk in cases:
        sk = np.concatenate([sk, sk[1:2, ::-1]])  # a descending copy of row 1
        assert (sk[-1, 1:] < sk[-1, :-1]).any()
        same, _ = mash.distance_block(sk)
        assert np.array_equal(same, _oracle_same_matrix(oracle, sk, range(len(sk))))


def test_distance_join_larger_family_set(gpu, oracle):
    """2k sketches of the cfg3 family shape at reduced size: spot-check rows against the oracle and
    check the structural properties of the full matrix (symmetry, diagonal, family blocks)."""
    n, L, k, s, fam = 2000, 2500, 31, 256, 20
    reads = synth.family_reads(n, L, family=fam)
    sk = mash.sketch_uniform(reads, n, L, k, s)
    same, _ = mash.distance_block(sk, want_distance=False)
    assert (np.diag(same) == s).all() and (same == same.T).all()
    rows = [0, 1, 19, 20, 777, 1999]
    assert np.array_equal(same[rows], _oracle_same_matrix(oracle, sk, rows))
    blocks = same.reshape(n // fam, fam, n // fam, fam)
    off_family = blocks.copy()
    for f in range(n // fam):
        off_family[f, :, f, :] = 0
    assert off_family.max() <= 2 and blocks[3, :, 3, :].min() > 20


def test_cfg3_full_size_properties(gpu, oracle):
    """BASELINE configs[2] sketching at full size (100k x 10 kbp, k=31, s=2000): every row
    ascending, spot rows bit-exact vs the oracle, and an all-pairs row block whose structure
    matches the family construction."""
    import torch
    from poly_b200 import _lib

    n, L, k, s = 100_000, 10_000, 31, 2000
    L_ = _lib.lib()
    dev = torch.device("cuda", int(os.environ.get("LOCAL_RANK", "0")))
    torch.cuda.set_device(dev)
    st = torch.cuda.current_stream().cuda_stream
    d_reads = torch.empty(n * L, dtype=torch.uint8, device=dev)
    _lib.check(L_.pg_synth_reads_dev(d_reads.data_ptr(), 0, n, L, synth.SEED_READS, 1, 100, st))
    d_sk = torch.empty((n, s), dtype=torch.int32, device=dev)
    _lib.check(L_.pg_mash_sketch_uniform_dev(d_reads.data_ptr(), n, L, k, s, 0, d_sk.data_ptr(), s, None, st))
    sk64 = d_sk.to(torch.int64) & 0xFFFFFFFF
    assert bool((sk64[:, 1:] >= sk64[:, :-1]).all())                          # sortedness of all 100k rows
    idx = [0, 1, 99, 100, 54_321, n - 1]
    got = d_sk[idx].cpu().numpy().view(np.uint32)
    host_reads = np.concatenate([synth.family_reads(1, L, family=100, first_read=i) for i in idx])
    dev_reads = np.concatenate([d_reads[i * L:(i + 1) * L].cpu().numpy() for i in idx])
    assert np.array_equal(host_reads, dev_reads)                               # device generator == numpy generator
    rc, want = oracle.sketch_batch(host_reads, synth.uniform_offsets(len(idx), L), k, s, variant=1)
    assert rc == 0 and np.array_equal(got, want)
    rows = 512
    d_same = torch.empty((rows, n), dtype=torch.int32, device=dev)
    _lib.check(L_.pg_mash_distance_block_dev(d_sk.data_ptr(), n, s, 0, rows, d_same.data_ptr(), None, st))
    same = d_same.cpu().numpy()
    assert (np.diag(same[:, :rows]) == s).all() and (same[:, :rows] == same[:, :rows].T).all()
    fam = same[:100, :100]
    assert fam[~np.eye(100, dtype=bool)].min() > 500 and same[:100, 100:].max() <= 3
    a = oracle.OracleMash(k, s); a.Sketches[:] = got[0]
    b = oracle.OracleMash(k, s); b.Sketches[:] = got[1]
    assert same[0, 1] == a.SimilarityCount(b)[0]


def test_randomized_differential_sketch(gpu, oracle):
    """120 random (k, s, L, n) combinations over all dispatch paths (TMA tiles, generic fill,
    select with bucket sort-select / radix fallback, odd sketch sizes, reads shorter than k)."""
    rng = np.random.default_rng(2026)
    ks = [0, 1, 3, 4, 7, 11, 13, 15, 16, 17, 19, 20, 21, 23, 24, 25, 27, 29, 31, 32, 33, 40]
    for trial in range(120):
        k = int(rng.choice(ks))
        L = int(rng.choice([0, 1, k, k + 1, 36, 64, 100, 150, 151, 152, 301, 1000, 2500]))
        s = int(rng.choice([2, 3, 5, 9, 10, 64, 127, 128, 129, 1000, 1001, 2000]))
        n = int(rng.choice([1, 31, 32, 33, 64, 97]))
        alpha = [b"ACGT", b"AC", bytes(range(256)), b"A"][trial % 4]
        reads = rng.choice(list(alpha), size=n * L).astype(np.uint8) if L else np.zeros(0, np.uint8)
        got = mash.sketch_uniform(reads, n, L, k, s)
        rc, want = oracle.sketch_batch(reads, synth.uniform_offsets(n, L), k, s, variant=1)
        assert rc == 0
        cnt = min(max(L - k, 0), s)
        assert np.array_equal(got, want[:, :cnt]), (k, s, L, n, trial)
    # ragged batches through the offsets entry point
    for trial in range(20):
        k = int(rng.choice([4, 13, 21, 31])); s = int(rng.choice([7, 64, 1000]))
        lens = rng.integers(0, 400, int(rng.integers(1, 80)))
        seqs = [bytes(rng.choice(list(b"ACGTN"), size=int(l)).astype(np.uint8)) for l in lens]
        bases, offsets = mash.flatten(seqs)
        out, count, status = mash.sketch_arrays(bases, offsets, k, s, pad_zero=True)
        rc, want = oracle.sketch_batch(bases, offsets, k, s, variant=1)
        assert rc == 0 and not status.any() and np.array_equal(out, want), (k, s, trial)


@pytest.mark.parametrize("k", [11, 16, 21, 24, 31])
def test_ragged_fast_path(gpu, oracle, k):
    """K1r (sketch_fill_ragged_kernel): ragged reads all in the fill regime -- TMA-staged tiles of 32
    reads with per-thread lengths; includes reads shorter than k, empty reads, a tail < 32 reads and
    arbitrary bytes."""
    rng = np.random.default_rng(k)
    s = 1000
    lens = np.concatenate([rng.integers(0, 220, 32 * 30 + 11), [0, 1, k - 1, k, k + 1, 219]])
    rng.shuffle(lens)
    seqs = [bytes(rng.integers(0, 256, int(l), dtype=np.uint8)) if i % 7 == 0 else bytes(rng.choice(list(b"ACGT"), size=int(l)).astype(np.uint8))
            for i, l in enumerate(lens)]
    bases, offsets = mash.flatten(seqs)
    for pad in (False, True):
        out, count, status = mash.sketch_arrays(bases, offsets, k, s if not pad else 256, pad_zero=pad)
        rc, want = oracle.sketch_batch(bases, offsets, k, s if not pad else 256, variant=1)
        assert rc == 0 and not status.any()
        assert np.array_equal(count, np.minimum(np.maximum(lens - k, 0), s if not pad else 256))
        assert np.array_equal(out, want[:, : out.shape[1]]), (k, pad)


def test_select_threshold_path(gpu, oracle, monkeypatch):
    """K2t (value-threshold walk + exact select): rows of one and of several work items, several launch
    groups, and rows on which the estimate must fail -- homopolymers / short repeats (fewer than s
    distinct hashes below the threshold, or far more than the buffer holds) -- which the device-side
    retry list hands to the exact streaming kernel.  Everything bit-exact against the oracle."""
    rng = np.random.default_rng(77)
    monkeypatch.setenv("PG_K2T_GROUP_ROWS", "7")
    # Between them the cases (and the ragged batch below) run every select-stage variant, (batch width U, bucket
    # function) as launch_select_thresh picks them from k, s and L:
    #   (3, shift) k = 32          (3, mul) k = 16, k = 11       (4, shift) s = 517, L = 539   (4, mul) s = 517, L = 1055
    #   (5, shift) k = 31          (5, mul) s = 733              (6, shift) k = 21, s = 1000   (6, mul) the ragged batch
    #   (8, shift) s = 1185        (8, mul) k = 24
    # and the walk with rare admissions (fewer than 1 in 512 hashes, the last case) next to the common one.
    cases = [(21, 1000, 40_000, 20), (31, 2000, 10_000, 40), (16, 64, 5_000, 33), (21, 1000, 1021 + 21, 9), (21, 1000, 1300, 9),
             (24, 5000, 30_000, 5), (32, 3, 9_000, 12), (11, 500, 2176 * 8 + 11 + 1, 6), (28, 300, 7_013, 8),
             (21, 517, 539, 9), (21, 517, 1055, 9), (21, 733, 1487, 9), (21, 1185, 1207, 9), (21, 1746, 1_047_621, 5)]
    for k, s, L, n in cases:
        reads = rng.choice(list(b"ACGT"), size=n * L).astype(np.uint8).reshape(n, L)
        reads[1] = ord("A")                                                   # homopolymer: one distinct hash
        reads[2] = np.frombuffer((b"ACG" * (L // 3 + 1))[:L], dtype=np.uint8)  # period 3: three distinct hashes
        reads[3] = rng.choice(list(b"AC"), size=L).astype(np.uint8)           # low complexity
        reads[4, : L // 2] = reads[4, L // 2: 2 * (L // 2)]                    # every k-mer of one half twice
        got = mash.sketch_uniform(reads.reshape(-1), n, L, k, s)
        rc, want = oracle.sketch_batch(reads.reshape(-1), synth.uniform_offsets(n, L), k, s, variant=1)
        assert rc == 0
        cnt = min(L - k, s)
        assert np.array_equal(got, want[:, :cnt]), (k, s, L, n, [i for i in range(n) if not np.array_equal(got[i], want[i, :cnt])])
    # ragged batch whose longest read spans several items: row x item mapping with empty items
    lens = [int(x) for x in rng.integers(1200, 50_000, 30)] + [0, 5, 1021, 1022, 1023]
    seqs = [bytes(rng.choice(list(b"ACGT"), size=l).astype(np.uint8)) for l in lens] + [b"T" * 30_000]
    bases, offsets = mash.flatten(seqs)
    out, count, status = mash.sketch_arrays(bases, offsets, 21, 1000, pad_zero=True)
    rc, want = oracle.sketch_batch(bases, offsets, 21, 1000, variant=1)
    assert rc == 0 and not status.any() and np.array_equal(out, want)


def test_select_beyond_shared_memory_limits(gpu, oracle):
    """Sketch sizes above 16384 and k above 1024 in the select regime (sketch_select_large.cu: hashes through
    global memory, radix select, bitonic sort in tiles and across tiles): the reference has no limit there
    (mash.go:68-104).  Uniform and ragged batches, ties, fill-regime rows in between, the s = 1 panic rule."""
    rng = np.random.default_rng(2026)
    for k, s, L, n in [(21, 20_000, 50_000, 5), (31, 16_385, 16_385 + 31 + 7, 3), (1500, 64, 6_000, 4), (17, 70_000, 300_000, 2),
                       (1025, 3, 4_000, 3), (24, 16_385, 16_385 + 24, 2)]:
        reads = rng.choice(list(b"ACGT"), size=n * L).astype(np.uint8).reshape(n, L)
        reads[1] = rng.choice(list(b"AC"), size=L).astype(np.uint8)            # low complexity: many tied hashes
        if n > 2:
            reads[2, : L // 2] = reads[2, L // 2: 2 * (L // 2)]                 # every k-mer of one half twice
        got = mash.sketch_uniform(reads.reshape(-1), n, L, k, s)
        rc, want = oracle.sketch_batch(reads.reshape(-1), synth.uniform_offsets(n, L), k, s, variant=1)
        assert rc == 0
        cnt = min(L - k, s)
        assert np.array_equal(got, want[:, :cnt]), (k, s, L, n, [i for i in range(n) if not np.array_equal(got[i], want[i, :cnt])])
    # ragged: select-regime rows (n >= s) between fill-regime and empty rows, rows wider than s
    s, k = 17_000, 21
    lens = [40_000, 100, 17_021, 17_020, 0, 90_001, 17_022, 5]
    seqs = [bytes(rng.choice(list(b"ACGT"), size=l).astype(np.uint8)) for l in lens] + [b"G" * 30_000]
    bases, offsets = mash.flatten(seqs)
    out, count, status = mash.sketch_arrays(bases, offsets, k, s, pad_zero=True)
    rc, want = oracle.sketch_batch(bases, offsets, k, s, variant=1)
    assert rc == 0 and not status.any() and np.array_equal(out, want)
    assert list(count) == [min(max(l - k, 0), s) for l in lens] + [s]
    # s = 1 beyond k = 1024: Sketches[0] is the minimum; the reference panics iff a later hash is below the first
    L, k = 3_000, 1100
    reads = rng.choice(list(b"ACGT"), size=6 * L).astype(np.uint8)
    out, count, status = mash.sketch_arrays(reads, synth.uniform_offsets(6, L), k, 1, pad_zero=True)
    saw = set()
    for i in range(6):
        o = oracle.OracleMash(k, 1)
        rc = o.Sketch(bytes(reads[i * L:(i + 1) * L]))
        saw.add(rc != 0)
        assert (status[i] != 0) == (rc != 0)
        if rc == 0:
            assert out[i, 0] == o.Sketches[0]
    assert saw  # the six reads ran


def test_sketch_into_leaves_the_tail_alone(gpu, oracle):
    """PG_SKETCH_TAIL_KEEP: only count[i] words of a row are written, like (*Mash).Sketch on an existing Mash
    (mash.go:73-80 never touches Sketches[n:s]).  Pageable and pinned output, ragged and fixed-length reads."""
    import torch
    from poly_b200 import _lib

    rng = np.random.default_rng(5)
    k, s = 21, 200
    lens = [150, 21, 0, 400, 22, 150, 221, 220, 5000, 90]
    seqs = [bytes(rng.choice(list(b"ACGT"), size=l).astype(np.uint8)) for l in lens]
    uniform = [bytes(rng.choice(list(b"ACGT"), size=150).astype(np.uint8)) for _ in range(70)]
    for batch in (seqs, uniform):
        bases, offsets = mash.flatten(batch)
        rc, want = oracle.sketch_batch(bases, offsets, k, s, variant=1)
        assert rc == 0
        n = len(batch)
        pinned = torch.empty((n, s), dtype=torch.int32, pin_memory=True).numpy().view(np.uint32)
        for out in (np.empty((n, s), dtype=np.uint32), pinned):
            out[:] = 0xDEADBEEF
            count, status = mash.sketch_into(bases, offsets, k, s, out)
            assert not status.any()
            for i, seq in enumerate(batch):
                c = min(max(len(seq) - k, 0), s)
                assert count[i] == c
                assert np.array_equal(out[i, :c], want[i, :c]) and (out[i, c:] == 0xDEADBEEF).all(), i
    # the device-pointer entry points refuse the flag (their kernels define the whole row)
    d = torch.zeros(64, dtype=torch.uint8, device="cuda")
    o = torch.zeros(64, dtype=torch.int32, device="cuda")
    assert gpu.lib().pg_mash_sketch_uniform_dev(d.data_ptr(), 1, 64, 21, 10, 2, o.data_ptr(), 10, None, 0) == _lib.PG_ERR_ARG


def test_select_rows_wider_than_s_are_zero_filled(gpu, oracle):
    """include/poly_b200.h: words [count, row_stride) of every row are zeros -- also in the select regime
    and for device-pointer callers that hand in a dirty buffer."""
    import torch

    n, L, k, s, stride = 40, 3000, 21, 100, 131
    reads = synth.independent_reads(n, L)
    dev = torch.device("cuda", 0)
    d_in = torch.from_numpy(reads).to(dev)
    d_out = torch.full((n, stride), -1, dtype=torch.int32, device=dev)
    st = torch.cuda.current_stream().cuda_stream
    gpu.check(gpu.lib().pg_mash_sketch_uniform_dev(d_in.data_ptr(), n, L, k, s, 0, d_out.data_ptr(), stride, None, st))
    got = d_out.cpu().numpy().view(np.uint32)
    rc, want = oracle.sketch_batch(reads, synth.uniform_offsets(n, L), k, s, variant=1)
    assert rc == 0 and np.array_equal(got[:, :s], want) and not got[:, s:].any()


def test_distance_sparse_equals_dense(gpu, oracle):
    """pg_mash_distance_sparse: exactly the non-zero off-diagonal entries of the dense row block, for ascending
    sketches (inverted-index join) and for unsorted zero-padded ones (pairwise kernel), full and upper."""
    n, L, k, s = 96, 3000, 21, 128
    reads = synth.family_reads(n, L, family=6)
    sk = mash.sketch_uniform(reads, n, L, k, s)
    sk[7] = sk[6]                                      # identical sketches
    fill, _, _ = mash.sketch_arrays(synth.independent_reads(33, 150), synth.uniform_offsets(33, 150), 21, 200, pad_zero=True)
    fill[3] = fill[2]
    for sketches in (sk, fill):
        dense, _ = mash.distance_block(sketches, want_distance=False)
        for (rb, re) in [(0, len(sketches)), (5, min(41, len(sketches)))]:
            for upper in (True, False):
                pi, pj, ps = mash.distance_sparse(sketches, rb, re, upper=upper)
                want = [(i, j, int(dense[i, j])) for i in range(rb, re) for j in range(len(sketches))
                        if dense[i, j] and i != j and (j > i or not upper)]
                assert list(zip(pi.tolist(), pj.tolist(), ps.tolist())) == want
    assert len(mash.distance_sparse(sk)[0]) > 100
