"""GPU parity suite (-m gpu): the CUDA path through the C ABI against the CPU oracle and the
reference's golden matrices.  Integer/byte work: every comparison is bit-exact."""
import os

import numpy as np
import pytest

from conftest import (GOLDEN, assert_same_triplets, golden_dict, same_entries, to_oracle_batch, to_staged,
                      triplet_dict)

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def vb():
    import vartrix_b200
    return vartrix_b200


def _run_engine(vb, sb, bcs, mode, umi, **kw):
    with vb.Engine(mode, umi=umi, **kw) as eng:
        eng.set_barcodes(bcs)
        return eng.run(sb)


def _oracle_run(oracle, sb, bcs, mode, umi, threads=8):
    return oracle.run_batch(to_oracle_batch(oracle, sb), oracle.Barcodes(bcs.keys), oracle.MODES[mode], umi, n_threads=threads)


# ------------------------------------------------------------------------------------------------
# reference goldens (BASELINE.json configs[0] and the other six regression tests, main.rs:1207-1466)
# ------------------------------------------------------------------------------------------------
def test_reference_goldens_through_the_cuda_path(vb, oracle, goldens, golden_batches):
    for case in goldens["cases"]:
        sb = to_staged(golden_batches[case["batch"]])
        bcs = vb.Barcodes([k.encode() for k in goldens["barcodes"][case["barcodes"]]])
        got = _run_engine(vb, sb, bcs, case["scoring_method"], case["umi"])
        g = goldens["matrices"][case["out"]]
        assert same_entries(triplet_dict(got.row, got.col, got.val), golden_dict(g)), case["name"]
        if case["ref"]:
            assert same_entries(triplet_dict(got.row, got.col, got.val2), golden_dict(goldens["matrices"][case["ref"]])), case["name"]
        exp = _oracle_run(oracle, sb, bcs, case["scoring_method"], case["umi"])
        assert_same_triplets(got, exp)
        assert got.metrics == exp.metrics, case["name"]


def test_fixture_raw_scores_bit_exact(vb, oracle, golden_batches):
    """Scores.ref_score / alt_score (main.rs:926-927) of every fetched fixture record (2 123 pairs)."""
    with vb.Engine("coverage") as eng:
        for name, ob in golden_batches.items():
            sb = to_staged(ob)
            cs = sb.cand_start.astype(np.int64)
            pair_locus = np.repeat(np.arange(sb.n_loci), np.diff(cs)).astype(np.uint32)
            rs, as_ = eng.score_pairs(sb, sb.cand_read, pair_locus)
            ors, oas = oracle.score_pairs(ob, sb.cand_read, pair_locus, n_threads=8)
            assert np.array_equal(rs.astype(np.int32), ors), name
            assert np.array_equal(as_.astype(np.int32), oas), name


# ------------------------------------------------------------------------------------------------
# randomized pairs: every tile class, ragged lengths, exotic alphabets
# ------------------------------------------------------------------------------------------------
def _random_pairs_batch(vb, rng, n_loci, reads_per_locus, m_lo, m_hi, n_lo, n_hi, alphabet=b"ACGT", read_codes=(1, 2, 4, 8),
                        related=True):
    haps, ref_off, ref_len, alt_off, alt_len = bytearray(), [], [], [], []
    nibs, read_off, read_len = bytearray(), [], []
    cand = []
    alpha = np.frombuffer(alphabet, np.uint8)
    dec = np.frombuffer(b"=ACMGRSVTWYHKDBN", np.uint8)
    enc = {int(dec[i]): i for i in range(16)}
    for l in range(n_loci):
        nr = int(rng.integers(n_lo, n_hi + 1)); na = int(rng.integers(n_lo, n_hi + 1))
        ref = alpha[rng.integers(0, len(alpha), nr)]
        alt = ref.copy()[:na] if na <= nr else np.concatenate([ref, alpha[rng.integers(0, len(alpha), na - nr)]])
        if len(alt):
            k = int(rng.integers(0, len(alt))); alt[k] = alpha[rng.integers(0, len(alpha))]
        for h, offs, lens in ((ref, ref_off, ref_len), (alt, alt_off, alt_len)):
            while len(haps) % 16: haps.append(0)
            offs.append(len(haps)); lens.append(len(h)); haps.extend(h.tobytes())
        for _ in range(reads_per_locus):
            m = int(rng.integers(m_lo, m_hi + 1))
            if related and nr > 0 and rng.random() < 0.8:       # mostly substrings of a haplotype with a few edits
                src = ref if rng.random() < 0.5 else alt
                if len(src) == 0: src = ref
                s = int(rng.integers(0, max(1, len(src))))
                seq = np.resize(src[s:s + m], m) if len(src[s:s + m]) else alpha[rng.integers(0, len(alpha), m)]
                seq = seq.copy()
                for _e in range(int(rng.integers(0, 4))):
                    if m: seq[int(rng.integers(0, m))] = alpha[rng.integers(0, len(alpha))]
                codes = np.array([enc.get(int(c), 15) for c in np.char.upper(seq.view("S1")).view(np.uint8)], np.uint8)
            else:
                codes = np.array(read_codes, np.uint8)[rng.integers(0, len(read_codes), m)]
            if m & 1: codes = np.concatenate([codes, np.zeros(1, np.uint8)])
            while len(nibs) % 16: nibs.append(0)
            read_off.append(len(nibs)); read_len.append(m)
            nibs.extend(((codes[0::2] << 4) | codes[1::2]).astype(np.uint8).tobytes())
            cand.append((len(read_len) - 1, l))
    while len(nibs) % 16: nibs.append(0)
    n_reads = len(read_len)
    cand_start = np.arange(n_loci + 1, dtype=np.uint64) * reads_per_locus
    sb = vb.StagedBatch(
        locus_row=np.arange(n_loci), hap_bytes=np.frombuffer(bytes(haps), np.uint8), ref_off=ref_off, ref_len=ref_len,
        alt_off=alt_off, alt_len=alt_len, cand_start=cand_start, read_nib=np.frombuffer(bytes(nibs), np.uint8),
        read_off=read_off, read_len=read_len, cb_bytes=np.zeros(0, np.uint8), read_cb_off=np.full(n_reads, vb.engine.NO_CB),
        read_cb_len=np.zeros(n_reads), read_umi_key=np.full(n_reads, vb.engine.NO_UMI, np.uint64),
        cand_read=np.arange(n_reads), n_rows=n_loci)
    pr = np.array([c[0] for c in cand], np.uint32); pl = np.array([c[1] for c in cand], np.uint32)
    return sb, pr, pl


@pytest.mark.parametrize("name,kw", [
    ("class0_snv_shape", dict(n_loci=40, reads_per_locus=9, m_lo=100, m_hi=151, n_lo=190, n_hi=208)),
    ("split_shapes_mixed_reads", dict(n_loci=60, reads_per_locus=13, m_lo=60, m_hi=256, n_lo=150, n_hi=232)),
    ("class1_indel_shape", dict(n_loci=30, reads_per_locus=7, m_lo=120, m_hi=150, n_lo=209, n_hi=232)),
    ("class2", dict(n_loci=20, reads_per_locus=6, m_lo=90, m_hi=160, n_lo=233, n_hi=256)),
    ("class3", dict(n_loci=20, reads_per_locus=6, m_lo=90, m_hi=250, n_lo=257, n_hi=320)),
    ("generic_wide_haps", dict(n_loci=8, reads_per_locus=5, m_lo=50, m_hi=200, n_lo=321, n_hi=700)),
    ("tiny_and_empty", dict(n_loci=60, reads_per_locus=5, m_lo=0, m_hi=12, n_lo=0, n_hi=14)),
    ("ragged_everything", dict(n_loci=80, reads_per_locus=11, m_lo=1, m_hi=300, n_lo=1, n_hi=330)),
    ("lowercase_alt_bytes", dict(n_loci=20, reads_per_locus=8, m_lo=80, m_hi=150, n_lo=150, n_hi=208, alphabet=b"ACGTacgt")),
    ("iupac_haplotypes_generic", dict(n_loci=20, reads_per_locus=8, m_lo=80, m_hi=150, n_lo=150, n_hi=208,
                                      alphabet=b"ACGTNRYKM=", read_codes=tuple(range(16)), related=False)),
    ("reads_with_N_and_iupac", dict(n_loci=20, reads_per_locus=8, m_lo=80, m_hi=150, n_lo=150, n_hi=208,
                                    read_codes=(1, 2, 4, 8, 15, 15, 3, 0), related=False)),
    ("long_reads_row_blocks", dict(n_loci=3, reads_per_locus=3, m_lo=1025, m_hi=1400, n_lo=180, n_hi=208)),
    ("very_long_reads_row_blocks", dict(n_loci=2, reads_per_locus=5, m_lo=2000, m_hi=6000, n_lo=150, n_hi=320)),
    ("long_reads_wide_windows_generic", dict(n_loci=2, reads_per_locus=3, m_lo=300, m_hi=900, n_lo=330, n_hi=500)),
])
def test_random_pairs_bit_exact(vb, oracle, name, kw):
    rng = np.random.default_rng(sum(map(ord, name)))
    sb, pr, pl = _random_pairs_batch(vb, rng, **kw)
    perm = rng.permutation(len(pr))                 # arbitrary pair order is allowed
    ors, oas = oracle.score_pairs(to_oracle_batch(oracle, sb), pr[perm], pl[perm], n_threads=8)
    # folded + shared-prefix kernels where the windows allow, shared-prefix only, single-phase classes only
    for kw_eng in (dict(), dict(no_fold=True), dict(no_split=True)):
        with vb.Engine("coverage", **kw_eng) as eng:
            rs, as_ = eng.score_pairs(sb, pr[perm], pl[perm])
        bad = np.nonzero((rs.astype(np.int32) != ors) | (as_.astype(np.int32) != oas))[0]
        assert bad.size == 0, (name, kw_eng, bad[:5], rs[bad[:5]], ors[bad[:5]], as_[bad[:5]], oas[bad[:5]])


# ------------------------------------------------------------------------------------------------
# windows the folded kernel takes: both flanks (>= 96 columns) common to ref and alt, 1..40 allele columns
# ------------------------------------------------------------------------------------------------
def _edited(rng, src, alpha, sub, indel):
    out = []
    for b in src:
        u = rng.random()
        if u < sub:
            out.append(alpha[rng.integers(0, len(alpha))])
        elif u < sub + indel:
            continue
        elif u < sub + 2 * indel:
            out.append(b); out.extend(alpha[rng.integers(0, len(alpha), int(rng.integers(1, 6)))])
        else:
            out.append(b)
    return np.array(out, np.uint8)


def _fold_pairs_batch(vb, rng, n_loci, reads_per_locus, m_lo, m_hi, mid_lo, mid_hi, flank_lo=96, flank_hi=96, alphabet=b"ACGT",
                      same_mid_len=False, sub=0.01, indel=0.004, related_mid=True, long_loci=0):
    haps, ref_off, ref_len, alt_off, alt_len = bytearray(), [], [], [], []
    nibs, read_off, read_len = bytearray(), [], []
    alpha = np.frombuffer(alphabet, np.uint8)
    enc = {ord("A"): 1, ord("C"): 2, ord("G"): 4, ord("T"): 8, ord("N"): 15}
    for l in range(n_loci):
        left = alpha[rng.integers(0, len(alpha), int(rng.integers(flank_lo, flank_hi + 1)))]
        right = alpha[rng.integers(0, len(alpha), int(rng.integers(flank_lo, flank_hi + 1)))]
        lr = int(rng.integers(mid_lo, mid_hi + 1)); la = lr if same_mid_len else int(rng.integers(mid_lo, mid_hi + 1))
        mr = alpha[rng.integers(0, len(alpha), lr)]
        if related_mid:                                  # SNV / indel like: the alt allele is an edit of the ref allele
            ma = np.resize(mr, la).copy()
            ma[int(rng.integers(0, la))] = alpha[rng.integers(0, len(alpha))]
        else:
            ma = alpha[rng.integers(0, len(alpha), la)]
        ref = np.concatenate([left, mr, right]); alt = np.concatenate([left, ma, right])
        for h, offs, lens in ((ref, ref_off, ref_len), (alt, alt_off, alt_len)):
            while len(haps) % 16: haps.append(0)
            offs.append(len(haps)); lens.append(len(h)); haps.extend(h.tobytes())
        for ri in range(reads_per_locus):
            m = int(rng.integers(m_lo, m_hi + 1))
            if l < long_loci and ri == 1:
                m = int(rng.integers(153, 257))            # one read of this locus is too long for the folded kernel
            src = ref if rng.random() < 0.5 else alt
            u = rng.random()
            if u < 0.1:
                seq = alpha[rng.integers(0, len(alpha), m)]
            else:                                        # a stretch of a haplotype (possibly hanging over an end) with edits
                s0 = int(rng.integers(-20, len(src) - 10))
                seq = np.array([src[j] if 0 <= j < len(src) else alpha[rng.integers(0, len(alpha))] for j in range(s0, s0 + m + 8)], np.uint8)
                seq = _edited(rng, seq, alpha, sub, indel)[:m]
            if u > 0.97 and len(seq):
                seq = seq.copy(); seq[int(rng.integers(0, len(seq)))] = ord("N")
            m = len(seq)
            codes = np.array([enc[int(c)] for c in seq], np.uint8)
            if m & 1: codes = np.concatenate([codes, np.zeros(1, np.uint8)])
            while len(nibs) % 16: nibs.append(0)
            read_off.append(len(nibs)); read_len.append(m)
            nibs.extend(((codes[0::2] << 4) | codes[1::2]).astype(np.uint8).tobytes())
    while len(nibs) % 16: nibs.append(0)
    n_reads = len(read_len)
    sb = vb.StagedBatch(
        locus_row=np.arange(n_loci), hap_bytes=np.frombuffer(bytes(haps), np.uint8), ref_off=ref_off, ref_len=ref_len,
        alt_off=alt_off, alt_len=alt_len, cand_start=np.arange(n_loci + 1, dtype=np.uint64) * reads_per_locus,
        read_nib=np.frombuffer(bytes(nibs), np.uint8), read_off=read_off, read_len=read_len, cb_bytes=np.zeros(0, np.uint8),
        read_cb_off=np.full(n_reads, vb.engine.NO_CB), read_cb_len=np.zeros(n_reads),
        read_umi_key=np.full(n_reads, vb.engine.NO_UMI, np.uint64), cand_read=np.arange(n_reads), n_rows=n_loci)
    pr = np.arange(n_reads, dtype=np.uint32); pl = np.repeat(np.arange(n_loci), reads_per_locus).astype(np.uint32)
    return sb, pr, pl


@pytest.mark.parametrize("name,kw,all_fold", [
    ("snv_pad100", dict(n_loci=60, reads_per_locus=13, m_lo=140, m_hi=151, mid_lo=9, mid_hi=9, same_mid_len=True), True),
    ("indel_pad100", dict(n_loci=60, reads_per_locus=9, m_lo=100, m_hi=152, mid_lo=9, mid_hi=40), True),
    ("complex_alleles", dict(n_loci=60, reads_per_locus=7, m_lo=30, m_hi=152, mid_lo=1, mid_hi=40, related_mid=False), True),
    ("shortest_middle", dict(n_loci=40, reads_per_locus=6, m_lo=1, m_hi=152, mid_lo=1, mid_hi=2), True),
    ("noisy_reads_gaps_across_the_junctions", dict(n_loci=50, reads_per_locus=9, m_lo=80, m_hi=152, mid_lo=1, mid_hi=40,
                                                   sub=0.03, indel=0.03), True),
    ("low_complexity", dict(n_loci=40, reads_per_locus=9, m_lo=60, m_hi=152, mid_lo=1, mid_hi=30, alphabet=b"AC",
                            sub=0.02, indel=0.02), True),
    ("homopolymer", dict(n_loci=20, reads_per_locus=6, m_lo=60, m_hi=152, mid_lo=1, mid_hi=30, alphabet=b"A"), True),
    ("wider_flanks_and_too_wide", dict(n_loci=60, reads_per_locus=6, m_lo=100, m_hi=152, mid_lo=1, mid_hi=30, flank_lo=96,
                                       flank_hi=110), False),
])
def test_fold_windows_bit_exact(vb, oracle, name, kw, all_fold):
    rng = np.random.default_rng(sum(map(ord, name)) + 7)
    sb, pr, pl = _fold_pairs_batch(vb, rng, **kw)
    perm = rng.permutation(len(pr))
    ors, oas = oracle.score_pairs(to_oracle_batch(oracle, sb), pr[perm], pl[perm], n_threads=8)
    for kw_eng in (dict(), dict(no_fold=True)):
        with vb.Engine("coverage", **kw_eng) as eng:
            rs, as_ = eng.score_pairs(sb, pr[perm], pl[perm])
            tiles = eng.tile_counts()
        bad = np.nonzero((rs.astype(np.int32) != ors) | (as_.astype(np.int32) != oas))[0]
        assert bad.size == 0, (name, kw_eng, bad[:5], rs[bad[:5]], ors[bad[:5]], as_[bad[:5]], oas[bad[:5]])
        if kw_eng:
            assert tiles[7] == 0 and sum(tiles) > 0
        elif all_fold:                                  # every locus of these families must take the folded kernel
            assert tiles[7] > 0 and sum(tiles) == tiles[7], tiles
        else:
            assert tiles[7] > 0 and sum(tiles) > tiles[7], tiles


def test_fold_is_decided_per_locus_by_its_longest_read(vb, oracle):
    rng = np.random.default_rng(99)
    sb, pr, pl = _fold_pairs_batch(vb, rng, n_loci=12, reads_per_locus=5, m_lo=120, m_hi=152, mid_lo=9, mid_hi=9, same_mid_len=True,
                                   long_loci=4)
    lens = sb.read_len.reshape(12, 5)
    assert (lens[:4].max(axis=1) > 152).all() and (lens[4:] <= 152).all()
    ors, oas = oracle.score_pairs(to_oracle_batch(oracle, sb), pr, pl, n_threads=8)
    with vb.Engine("coverage") as eng:
        rs, as_ = eng.score_pairs(sb, pr, pl)
        tiles = eng.tile_counts()
    assert tiles[7] == 8 * 2 and tiles[5] == 4        # 8 loci x ceil(5/4) folded tiles; 4 loci x ceil(5/8) two-phase tiles
    assert np.array_equal(rs.astype(np.int32), ors) and np.array_equal(as_.astype(np.int32), oas)


# ------------------------------------------------------------------------------------------------
# whole path on synthetic shards of the BASELINE.json shapes (scaled to oracle-in-seconds sizes)
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("mode", ["consensus", "coverage", "alt_frac"])
@pytest.mark.parametrize("kind,umi", [("snv", False), ("indel", True), ("snv", True), ("indel", False)])
def test_synthetic_shard_matches_oracle(vb, oracle, mode, kind, umi):
    sb, bcs, info = vb.synth.make_shard(300, 120, depth=50, seed=11, kind=kind, umi=umi, reads_per_umi=3)
    got = _run_engine(vb, sb, bcs, mode, umi)
    exp = _oracle_run(oracle, sb, bcs, mode, umi)
    assert_same_triplets(got, exp)
    assert_same_triplets(_run_engine(vb, sb, bcs, mode, umi, no_split=True), exp)
    assert_same_triplets(_run_engine(vb, sb, bcs, mode, umi, no_fold=True), exp)
    assert got.metrics == exp.metrics and got.metrics["num_scored"] == info["n_pairs"]
    # text output is byte-identical to the oracle's writer as well
    assert vb.mtx.mtx_text(sb.n_rows, len(bcs), got.row, got.col, got.val) == oracle.mtx_text(sb.n_rows, len(bcs), exp.row, exp.col, exp.val)


def test_device_resident_submit_equals_host_submit(vb):
    """vtx_submit_device_ex (what bench.py's `value` times): same triplets as the host-buffer path, for SNV and indel shards."""
    import torch
    for kind, umi in (("snv", False), ("indel", True)):
        sb, bcs, info = vb.synth.make_shard(400, 150, depth=40, seed=21, kind=kind, umi=umi)
        exp = _run_engine(vb, sb, bcs, "coverage", umi)
        keep, db = [], sb.to_c()
        for f in vb.StagedBatch.FIELDS:
            a = getattr(sb, f)
            t = torch.from_numpy(a.view(np.uint8).reshape(-1) if a.dtype.itemsize > 1 else a.reshape(-1)).cuda()
            keep.append(t)
            setattr(db, f, t.data_ptr() if t.numel() else None)
        with vb.Engine("coverage", umi=umi) as eng:
            eng.set_barcodes(bcs)
            for _ in range(2):                         # resubmitting the same resident shard gives the same answer
                eng.submit_device(db, int(sb.read_len.max()), int(max(sb.ref_len.max(), sb.alt_len.max())))
                dev = eng.finish_device()
                got = eng.fetch(dev)
                assert_same_triplets(got, exp)
                assert got.metrics == exp.metrics


def test_bench_dump_outputs_are_the_oracle_triplets(vb, oracle, tmp_path):
    """bench.py --dump-outputs writes what its timed `value` steps returned: the oracle's triplets of the same seeded shard."""
    import json
    import subprocess
    import sys
    from conftest import ROOT
    from vartrix_b200 import dist as vdist
    d = tmp_path / "dump"
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--workload", "config2", "--loci", "400", "--steps", "2",
                        "--warmup", "1", "--no-cpu-baseline", "--dump-outputs", str(d)], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr[-3000:]
    assert json.loads(r.stdout.strip().splitlines()[-1])["steps"] == 2
    sb, bcs, _ = vb.synth.make_shard(**vdist.rank_workload(dict(vb.synth.CONFIGS["config2"], n_loci=400), 0))
    exp = _oracle_run(oracle, sb, bcs, "coverage", False)
    for f in ("row", "col", "val", "val2"):
        assert np.array_equal(np.load(d / f"{f}.npy"), getattr(exp, f).astype(np.float64), equal_nan=True), f
    m = exp.metrics
    assert np.array_equal(np.load(d / "metrics.npy"), [len(exp.row), m["num_scored"], m["num_not_cell_bc"], m["num_non_umi"]])


def test_edge_cases(vb, oracle):
    sb, bcs, info = vb.synth.make_shard(40, 10, depth=30, seed=3, umi=True, unlisted_frac=0.3)
    # reads without CB / without UB, loci without candidates
    sb.read_cb_off[::7] = vb.engine.NO_CB
    sb.read_umi_key[::5] = vb.engine.NO_UMI
    cs = sb.cand_start.copy(); cs[5:9] = cs[5]; cs[20] = cs[21]
    sb.cand_start = np.maximum.accumulate(cs)
    for mode in ("coverage", "alt_frac", "consensus"):
        for umi in (False, True):
            assert_same_triplets(_run_engine(vb, sb, bcs, mode, umi), _oracle_run(oracle, sb, bcs, mode, umi))
    # nothing listed at all -> empty result, all candidates counted as CB misses
    none = vb.Barcodes([b"NOT-A-BARCODE-1"])
    got = _run_engine(vb, sb, none, "coverage", False)
    assert len(got.row) == 0 and got.metrics["num_scored"] == 0 and got.metrics["num_not_cell_bc"] == sb.n_cand
    # empty shard
    empty = sb.shard(0, 0)
    got = _run_engine(vb, empty, bcs, "coverage", False)
    assert len(got.row) == 0


@pytest.mark.parametrize("umi", [False, True])
def test_deep_loci_use_the_hash_sort_slot_kernel(vb, oracle, umi):
    """Loci deeper than 2 048 pairs (a variant in a highly expressed gene) leave the O(d^2) slot kernel."""
    sb, bcs, info = vb.synth.make_shard(5, 700, depth=5000, seed=17, kind="snv", umi=umi, reads_per_umi=4, chunk_loci=1)
    cs = sb.cand_start.copy(); cs[2] = cs[1] + 900          # mix: one shallow locus between deep ones
    keep = np.concatenate([np.arange(int(cs[0]), int(cs[2])), np.arange(int(sb.cand_start[2]), sb.n_cand)])
    sb.cand_read = sb.cand_read[keep]
    cs[2:] = sb.cand_start[2:] - (sb.cand_start[2] - cs[2]); sb.cand_start = cs
    for mode in ("coverage", "consensus"):
        assert_same_triplets(_run_engine(vb, sb, bcs, mode, umi), _oracle_run(oracle, sb, bcs, mode, umi))


def test_min_score_boundary_and_ties(vb, oracle):
    """evaluate_scores: strict '<' on MIN_SCORE 25 (main.rs:1020) and ties -> UNKNOWN."""
    hap = b"ACGTTGCAAGGCTTAACCGGATCGATCGTAGCTAGCTAGGATCCATTGGCA" * 4
    reads = [hap[10:34], hap[10:35], hap[10:36], b"T" * 30]       # scores 24, 25, 26, ~1
    nibs, off = bytearray(), []
    enc = {65: 1, 67: 2, 71: 4, 84: 8}
    for r in reads:
        c = [enc[x] for x in r] + ([0] if len(r) & 1 else [])
        while len(nibs) % 16: nibs.append(0)
        off.append(len(nibs)); nibs.extend(bytes((c[i] << 4) | c[i + 1] for i in range(0, len(c), 2)))
    while len(nibs) % 16: nibs.append(0)
    hb = np.zeros(((len(hap) + 15) // 16 * 16) * 2, np.uint8); hb[:len(hap)] = np.frombuffer(hap, np.uint8)
    ao = (len(hap) + 15) // 16 * 16; hb[ao:ao + len(hap)] = np.frombuffer(hap, np.uint8)    # ref == alt -> ties
    tags = np.frombuffer(b"AAAA-1CCCC-1GGGG-1TTTT-1", np.uint8)
    sb = vb.StagedBatch(locus_row=[0], hap_bytes=hb, ref_off=[0], ref_len=[len(hap)], alt_off=[ao], alt_len=[len(hap)],
                        cand_start=[0, 4], read_nib=np.frombuffer(bytes(nibs), np.uint8), read_off=off,
                        read_len=[len(r) for r in reads], cb_bytes=tags, read_cb_off=[0, 6, 12, 18], read_cb_len=[6] * 4,
                        read_umi_key=[1, 2, 3, 4], cand_read=[0, 1, 2, 3], n_rows=1)
    bcs = vb.Barcodes([b"AAAA-1", b"CCCC-1", b"GGGG-1", b"TTTT-1"])
    got = _run_engine(vb, sb, bcs, "coverage", False)
    assert_same_triplets(got, _oracle_run(oracle, sb, bcs, "coverage", False))
    assert list(got.unk_cnt) == [0, 1, 1, 0] and list(got.col) == [0, 1, 2, 3]     # 24/24 -> None, 25/25 and 26/26 -> UNKNOWN


def test_multiple_submits_accumulate_in_row_order(vb, oracle):
    sb, bcs, _ = vb.synth.make_shard(90, 40, depth=20, seed=21)
    whole = _oracle_run(oracle, sb, bcs, "alt_frac", False)
    with vb.Engine("alt_frac") as eng:
        eng.set_barcodes(bcs)
        for lo, hi in vb.shard_bounds(sb.cand_start, 4):
            eng.submit(sb.shard(lo, hi))
        got = eng.finish()
        assert_same_triplets(got, whole)
        again = eng.run(sb)                       # the context is reusable after finish
        assert_same_triplets(again, whole)
        t = eng.timing()
        assert t["n_pairs"] == whole.metrics["num_scored"] and t["sw_launches"] >= 1 and t["sw_ms"] > 0


# ------------------------------------------------------------------------------------------------
# full BASELINE size (config 2: 10k SNV loci x 5k barcodes, 475k pairs): size-independent properties
# ------------------------------------------------------------------------------------------------
def test_full_size_config2_properties(vb, oracle):
    cfg = vb.synth.CONFIGS["config2"]
    sb, bcs, info = vb.synth.make_shard(**cfg)
    with vb.Engine("coverage") as eng:
        eng.set_barcodes(bcs)
        a = eng.run(sb)
        b = eng.run(sb)
        parts = []
        for lo, hi in vb.shard_bounds(sb.cand_start, 3):
            parts.append(eng.run(sb.shard(lo, hi)))
    assert_same_triplets(a, b)                                             # run-to-run determinism
    key = a.row.astype(np.int64) * len(bcs) + a.col
    assert (np.diff(key) > 0).all()                                        # row-major sorted, no duplicate cells
    assert a.metrics["num_scored"] == info["n_pairs"]
    assert a.metrics["num_scored"] + a.metrics["num_not_cell_bc"] == sb.n_cand
    assert int(a.ref_cnt.sum() + a.alt_cnt.sum() + a.unk_cnt.sum()) <= info["n_pairs"]
    for f in ("row", "col", "ref_cnt", "alt_cnt", "unk_cnt"):              # locus sharding is invisible in the result
        assert np.array_equal(np.concatenate([getattr(p, f) for p in parts]), getattr(a, f)), f
    # checksum of checksums against the oracle on a 400-locus window of the same shard
    win = sb.shard(5000, 5400)
    exp = _oracle_run(oracle, win, bcs, "coverage", False)
    sel = (a.row >= 5000) & (a.row < 5400)
    assert np.array_equal(a.col[sel], exp.col) and np.array_equal(a.alt_cnt[sel], exp.alt_cnt) and np.array_equal(a.ref_cnt[sel], exp.ref_cnt)


def test_api_rejects_malformed_input_with_messages(vb):
    """Error behaviour across the boundary: negative code + message, never a crash or a silent wrong answer."""
    import ctypes as C
    from vartrix_b200 import _capi
    sb, bcs, _ = vb.synth.make_shard(6, 5, depth=4, seed=1)
    with vb.Engine("coverage") as eng:
        with pytest.raises(vb.VtxError, match="vtx_set_barcodes must be called"):
            eng.submit(sb)
        with pytest.raises(vb.VtxError, match="duplicate barcode"):
            eng.set_barcodes(vb.Barcodes([b"AAA-1", b"CCC-1", b"AAA-1"]))
        eng.set_barcodes(bcs)
        bad = sb.shard(0, 6); bad.cand_read[3] = 10_000
        with pytest.raises(vb.VtxError, match="cand_read out of range"):
            eng.submit(bad)
        bad = sb.shard(0, 6); bad.ref_off[2] += 4
        with pytest.raises(vb.VtxError, match="multiples of 16"):
            eng.submit(bad)
        bad = sb.shard(0, 6); bad.locus_row[3] = bad.locus_row[2]
        with pytest.raises(vb.VtxError, match="strictly ascending"):
            eng.submit(bad)
        bad = sb.shard(0, 6); bad.read_umi_key[0] = 1 << 63
        with pytest.raises(vb.VtxError, match="UMI key"):
            eng.submit(bad)
        bad = sb.shard(0, 6); bad.cand_start[-1] += 1
        with pytest.raises(vb.VtxError, match="cand_start"):
            eng.submit(bad)
        assert len(eng.run(sb).row) > 0                      # the context survives rejected submits
    cfg = _capi.Config(device=0, mode=0, use_umi=0, match=2, mismatch=-5, gap_open=-5, gap_extend=-1, min_score=25, stream=None, flags=0)
    h = C.c_void_p()
    L = _capi.load()
    assert L.vtx_create(C.byref(cfg), C.byref(h)) == -4 and b"compiled in" in L.vtx_last_error(None)
    cfg.match = 1; cfg.device = 99
    assert L.vtx_create(C.byref(cfg), C.byref(h)) == -1 and b"out of range" in L.vtx_last_error(None)


def test_values_only_fetch_and_raw_score_side_channel(vb, oracle):
    sb, bcs, info = vb.synth.make_shard(40, 20, depth=10, seed=4)
    exp = _oracle_run(oracle, sb, bcs, "coverage", False)
    with vb.Engine("coverage", values_only=True) as eng:
        eng.set_barcodes(bcs)
        got = eng.run(sb)
    assert np.array_equal(got.row, exp.row) and np.array_equal(got.col, exp.col)
    assert np.array_equal(got.val, exp.val) and np.array_equal(got.val2, exp.val2) and got.ref_cnt.size == 0


def test_fuzz_whole_path_against_oracle(vb, oracle):
    """Differential fuzz of the whole path: irregular shards (reads shared between loci, repeated candidates, missing
    tags, tiny barcode lists so that cells collide, interned-style UMI keys, every mode) against the oracle."""
    rng = np.random.default_rng(20240924)
    for it in range(24):
        n_loci = int(rng.integers(1, 30))
        sb, pr, pl = _random_pairs_batch(vb, rng, n_loci=n_loci, reads_per_locus=int(rng.integers(1, 12)), m_lo=int(rng.integers(1, 60)),
                                         m_hi=int(rng.integers(60, 200)), n_lo=int(rng.integers(40, 150)), n_hi=int(rng.integers(150, 260)))
        n_reads = sb.n_reads
        # candidates: every locus draws a random multiset of reads (reads are shared between loci, some repeated)
        per = rng.integers(0, 40, size=n_loci)
        cand_start = np.concatenate([[0], np.cumsum(per)]).astype(np.uint64)
        cand_read = rng.integers(0, n_reads, size=int(per.sum())).astype(np.uint32)
        n_bc = int(rng.integers(1, 7))
        keys = [f"BC{k:02d}-1".encode() for k in range(n_bc)]
        tags = keys + [b"UNLISTED-1", b"BC00-2"]
        pick = rng.integers(0, len(tags), size=n_reads)
        cb_bytes = np.frombuffer(b"".join(tags), np.uint8)
        offs = np.concatenate([[0], np.cumsum([len(t) for t in tags])])
        read_cb_off = offs[pick].astype(np.uint32); read_cb_len = np.array([len(tags[i]) for i in pick], np.uint16)
        read_cb_off[rng.random(n_reads) < 0.1] = vb.engine.NO_CB
        umi = rng.integers(0, 4, size=n_reads).astype(np.uint64) | (np.uint64(1) << np.uint64(61)) * (rng.random(n_reads) < 0.5).astype(np.uint64)
        umi[rng.random(n_reads) < 0.1] = vb.engine.NO_UMI
        shard = vb.StagedBatch(locus_row=np.cumsum(rng.integers(1, 4, size=n_loci)), hap_bytes=sb.hap_bytes, ref_off=sb.ref_off, ref_len=sb.ref_len,
                               alt_off=sb.alt_off, alt_len=sb.alt_len, cand_start=cand_start, read_nib=sb.read_nib, read_off=sb.read_off,
                               read_len=sb.read_len, cb_bytes=cb_bytes, read_cb_off=read_cb_off, read_cb_len=read_cb_len, read_umi_key=umi,
                               cand_read=cand_read, n_rows=int(3 * n_loci + 4))
        bcs = vb.Barcodes(keys)
        mode = ("consensus", "coverage", "alt_frac")[it % 3]
        use_umi = bool(it & 1)
        got = _run_engine(vb, shard, bcs, mode, use_umi, no_split=bool(it & 2), no_fold=bool(it & 4))
        exp = _oracle_run(oracle, shard, bcs, mode, use_umi, threads=4)
        assert_same_triplets(got, exp)
        assert got.metrics == exp.metrics, it
