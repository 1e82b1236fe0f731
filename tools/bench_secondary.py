#!/usr/bin/env python
"""Timings of the non-headline kernels on their BASELINE configs (device-resident, CUDA events):
cfg3 (100k x 10 kbp, k=31, s=2000: K2 sketch + K3 all-pairs on a row block) and cfg5
(1M x 25 bp primers vs a 10 kb template: K4 SW score, K5 Tm).  Prints one JSON line per kernel;
copy into profiles/.  Not the driver's bench (that is bench.py)."""
import argparse
import json
import os
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from poly_b200 import _lib, align, synth  # noqa: E402

ap = argparse.ArgumentParser()
ap.add_argument("--reads", type=int, default=100_000)
ap.add_argument("--rows", type=int, default=512, help="row block of the all-pairs matrix to time")
ap.add_argument("--primers", type=int, default=1_000_000)
ap.add_argument("--iters", type=int, default=3)
ap.add_argument("--only-k2", action="store_true", help="stop after the K2 legs")
args = ap.parse_args()

L = _lib.lib()
_lib.check(L.pg_init(0))
dev = torch.device("cuda", 0)
st = torch.cuda.current_stream().cuda_stream


def timed(fn, iters=args.iters, warm=1):
    for _ in range(warm):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(iters):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / iters


# ---- cfg3: K2 + K3 ---------------------------------------------------------------------
n, RL, k, s = args.reads, 10_000, 31, 2000
d_reads = torch.empty(n * RL, dtype=torch.uint8, device=dev)
_lib.check(L.pg_synth_reads_dev(d_reads.data_ptr(), 0, n, RL, synth.SEED_READS, 1, 100, st))
d_sk = torch.empty((n, s), dtype=torch.int32, device=dev)
ms = timed(lambda: _lib.check(L.pg_mash_sketch_uniform_dev(d_reads.data_ptr(), n, RL, k, s, 0, d_sk.data_ptr(), s, None, st)))
alg = n * (RL + 4 * s)
print(json.dumps({"kernel": "K2 sketch_select (cfg3)", "reads": n, "read_len": RL, "k": k, "s": s, "ms": ms,
                  "gbases_per_s": n * RL / ms / 1e6, "algorithmic_GBps": alg / ms / 1e6, "kernel_name": L.pg_last_kernel().decode()}))
# genome-scale select regime: 256 sequences x 4 Mbp, k=21, s=1000 (n/s = 4000: the admission limit does the work)
gn, gL, gk, gs = 256, 4_000_000, 21, 1000
d_gen = torch.empty(gn * gL, dtype=torch.uint8, device=dev)
_lib.check(L.pg_synth_reads_dev(d_gen.data_ptr(), 0, gn, gL, synth.SEED_READS + 7, 0, 1, st))
d_gsk = torch.empty((gn, gs), dtype=torch.int32, device=dev)
ms_g = timed(lambda: _lib.check(L.pg_mash_sketch_uniform_dev(d_gen.data_ptr(), gn, gL, gk, gs, 0, d_gsk.data_ptr(), gs, None, st)))
g = d_gsk.cpu().numpy().view(np.uint32)
print(json.dumps({"kernel": "K2 sketch_select (256 x 4 Mbp genomes)", "k": gk, "s": gs, "ms": ms_g, "gbases_per_s": gn * gL / ms_g / 1e6,
                  "ascending": bool((np.diff(g.astype(np.int64), axis=1) >= 0).all()), "fnv": hex(synth.fnv1a64(g)),
                  "kernel_name": L.pg_last_kernel().decode()}))
ms_1 = timed(lambda: _lib.check(L.pg_mash_sketch_uniform_dev(d_gen.data_ptr(), 1, gL, gk, gs, 0, d_gsk.data_ptr(), gs, None, st)))
print(json.dumps({"kernel": "K2 sketch_select (ONE 4 Mbp sequence = mash.Sketch(genome))", "ms": ms_1, "gbases_per_s": gL / ms_1 / 1e6,
                  "same_as_batch_row0": bool((d_gsk[0].cpu().numpy().view(np.uint32) == g[0]).all()), "kernel_name": L.pg_last_kernel().decode()}))
# beyond the shared-memory kernels (sketch_select_large.cu): 64 of the genomes at s = 100000
xs, xn = 100_000, 64
d_xsk = torch.empty((xn, xs), dtype=torch.int32, device=dev)
ms_x = timed(lambda: _lib.check(L.pg_mash_sketch_uniform_dev(d_gen.data_ptr(), xn, gL, gk, xs, 0, d_xsk.data_ptr(), xs, None, st)), iters=2)
gx = d_xsk.cpu().numpy().view(np.uint32)
print(json.dumps({"kernel": "K2x large sketch (64 x 4 Mbp genomes, s = 100000)", "k": gk, "s": xs, "ms": ms_x, "gbases_per_s": xn * gL / ms_x / 1e6,
                  "ascending": bool((np.diff(gx.astype(np.int64), axis=1) >= 0).all()),
                  "head_equals_s1000_sketch": bool((gx[:, :gs] == g[:xn]).all()), "kernel_name": L.pg_last_kernel().decode()}))
del d_gen, d_xsk
if args.only_k2:
    sys.exit(0)
rows = min(args.rows, n)
d_same = torch.empty((rows, n), dtype=torch.int32, device=dev)
ms = timed(lambda: _lib.check(L.pg_mash_distance_block_dev(d_sk.data_ptr(), n, s, 0, rows, d_same.data_ptr(), None, st)), iters=1, warm=1)
pairs = rows * n
same = d_same.cpu().numpy()
print(json.dumps({"kernel": "K3 distance_block (cfg3 row block)", "rows": rows, "cols": n, "pairs": pairs, "ms": ms,
                  "gpairs_per_s": pairs / ms / 1e6, "full_allpairs_estimate_s": (n * (n - 1) / 2) / (pairs / ms * 1e3),
                  "diag_ok": bool((np.diag(same[:, :rows]) == s).all()), "row0_family_mean": float(same[0, 1:100].mean()),
                  "row0_other_max": int(same[0, 100:].max()), "kernel_name": L.pg_last_kernel().decode()}))
del d_same, d_sk, d_reads

# ---- cfg5: K4 + K5 ---------------------------------------------------------------------
m, PL, TL = args.primers, 25, 10_000
pr = torch.from_numpy(synth.primers(m)).to(dev)
off = torch.arange(m + 1, dtype=torch.int64, device=dev) * PL
tpl = torch.from_numpy(synth.template(TL)).to(dev)
alpha = align.NewAlphabet(["-", "A", "C", "G", "T"])
mat = np.array([[0, 0, 0, 0, 0], [0, 3, -3, -3, -3], [0, -3, 3, -3, -3], [0, -3, -3, 3, -3], [0, -3, -3, -3, 3]], dtype=np.int64)
lut = alpha.byte_lut()
score = torch.empty(m, dtype=torch.int64, device=dev)
ec = torch.empty(m, dtype=torch.int32, device=dev)
ep = torch.empty(m, dtype=torch.int64, device=dev)
ms = timed(lambda: _lib.check(L.pg_sw_score_batch_dev(pr.data_ptr(), off.data_ptr(), m, PL, tpl.data_ptr(), TL, 1, lut.ctypes.data, lut.ctypes.data,
                                                     mat.ctypes.data, 5, 5, -2, score.data_ptr(), ec.data_ptr(), ep.data_ptr(), st)), iters=2)
cells = m * PL * TL
print(json.dumps({"kernel": "K4 sw_score (cfg5)", "queries": m, "qlen": PL, "tlen": TL, "ms": ms, "gcups": cells / ms / 1e6,
                  "first6": score[:6].cpu().tolist(), "kernel_name": L.pg_last_kernel().decode()}))
tm = torch.empty(m, dtype=torch.float64, device=dev)
ms = timed(lambda: _lib.check(L.pg_tm_batch_dev(pr.data_ptr(), off.data_ptr(), m, 500e-9, 50e-3, 0.0, tm.data_ptr(), None, None, None, st)), iters=10)
print(json.dumps({"kernel": "K5 tm (cfg5)", "primers": m, "ms": ms, "mprimers_per_s": m / ms / 1e3, "first3": tm[:3].cpu().tolist()}))

# ---- ragged short reads (K1r): 2M reads, lengths uniform in [100, 150], k=21, s=1000 ------------
rng = np.random.default_rng(0)
nrag = 2_000_000
lens = rng.integers(100, 151, nrag)
offs = np.zeros(nrag + 1, dtype=np.int64); offs[1:] = np.cumsum(lens)
rag = torch.from_numpy(synth.independent_reads(int(offs[-1] // 150 + 1), 150)[: offs[-1]]).to(dev)
d_offs = torch.from_numpy(offs).to(dev)
d_rout = torch.empty((nrag, 129), dtype=torch.int32, device=dev)
d_cnt = torch.empty(nrag, dtype=torch.int32, device=dev)
ms = timed(lambda: _lib.check(L.pg_mash_sketch_batch_dev(rag.data_ptr(), d_offs.data_ptr(), nrag, 150, 21, 1000, 0, d_rout.data_ptr(), 129,
                                                         d_cnt.data_ptr(), None, st)), iters=5)
print(json.dumps({"kernel": "K1r ragged fill (2M reads, len 100..150)", "ms": ms, "gbases_per_s": float(offs[-1]) / ms / 1e6,
                  "kernel_name": L.pg_last_kernel().decode(), "count_ok": bool((d_cnt.cpu().numpy() == lens - 21).all())}))
del rag, d_rout

# ---- widened rows: FASTQ ingest (8f.2) and batched DesignPrimers (8f.3) ------------------------
import ctypes as C
from poly_b200 import pcr  # noqa: E402

nrec = 2_000_000
reads = synth.independent_reads(nrec, 150).reshape(nrec, 150)
rec = np.empty((nrec, 16 + 151 + 2 + 151), dtype=np.uint8)
rec[:, :16] = np.frombuffer(b"@r runid=0 ch=1\n", dtype=np.uint8)
rec[:, 16:166] = reads
rec[:, 166] = 10
rec[:, 167:169] = np.frombuffer(b"+\n", dtype=np.uint8)
rec[:, 169:319] = 73
rec[:, 319] = 10
text = torch.from_numpy(rec.reshape(-1)).to(dev)
d_bases = torch.empty(nrec * 150 + 64, dtype=torch.uint8, device=dev)
d_off = torch.empty(nrec + 1, dtype=torch.int64, device=dev)
nr, tot, ec, el = C.c_uint64(0), C.c_uint64(0), C.c_int32(0), C.c_uint64(0)


def ingest():
    _lib.check(L.pg_fastq_ingest_dev(text.data_ptr(), text.numel(), d_bases.data_ptr(), d_bases.numel(), d_off.data_ptr(), nrec,
                                     C.byref(nr), C.byref(tot), C.byref(ec), C.byref(el), st))


ms = timed(ingest, iters=3)
ok = nr.value == nrec and ec.value == 0 and bool(torch.equal(d_bases[: nrec * 150].cpu(), torch.from_numpy(reads.reshape(-1))))
print(json.dumps({"kernel": "FASTQ ingest (8f.2)", "records": nrec, "text_GB": text.numel() / 1e9, "ms": ms,
                  "text_GBps": text.numel() / ms / 1e6, "matches_generator": ok}))
del text, d_bases, d_off
# FASTA ingest (8f.2): 200k records x 50 lines of 60 residues, both reader models
nfa, nl_per, width = 200_000, 50, 60
body = synth.independent_reads(nfa * nl_per, width).reshape(nfa, nl_per, width)
fa = np.empty((nfa, 12 + nl_per * (width + 1)), dtype=np.uint8)
fa[:, :12] = np.frombuffer(b">seq0000000\n", dtype=np.uint8)
blk = fa[:, 12:].reshape(nfa, nl_per, width + 1)
blk[:, :, :width] = body
blk[:, :, width] = 10
ftext = torch.from_numpy(fa.reshape(-1)).to(dev)
f_bases = torch.empty(nfa * nl_per * width + 64, dtype=torch.uint8, device=dev)
f_names = torch.empty(nfa * 16, dtype=torch.uint8, device=dev)
f_off = torch.empty(nfa + 1, dtype=torch.int64, device=dev)
f_noff = torch.empty(nfa + 1, dtype=torch.int64, device=dev)
ntot = C.c_uint64(0)
for alias in (0, 1):
    def fasta_ingest():
        _lib.check(L.pg_fasta_ingest_dev(ftext.data_ptr(), ftext.numel(), 65536, alias, f_bases.data_ptr(), f_bases.numel(), f_off.data_ptr(),
                                         f_names.data_ptr(), f_names.numel(), f_noff.data_ptr(), nfa, C.byref(nr), C.byref(tot), C.byref(ntot),
                                         C.byref(ec), C.byref(el), st))
    ms = timed(fasta_ingest, iters=3)
    same = bool(torch.equal(f_bases[: nfa * nl_per * width].cpu(), torch.from_numpy(body.reshape(-1))))
    print(json.dumps({"kernel": "FASTA ingest (8f.2)", "bufio_alias": alias, "records": nr.value, "text_GB": ftext.numel() / 1e9, "ms": ms,
                      "text_GBps": ftext.numel() / ms / 1e6, "err_code": ec.value, "sequences_equal_generator": same}))
del ftext, f_bases
genes = [bytes(r) for r in synth.independent_reads(100_000, 300).reshape(100_000, 300)]
import time as _t
t0 = _t.perf_counter(); fl, rl, stt = pcr.design_primer_lengths(genes, 55.0); dt = _t.perf_counter() - t0
print(json.dumps({"kernel": "DesignPrimers batch (8f.3, host API incl. copies)", "genes": len(genes), "ms": dt * 1e3,
                  "mean_fwd_len": float(fl.mean()), "mean_rev_len": float(rl.mean()), "panics": int((stt != 0).sum())}))
