"""Folded kernel (vtx_k_sw_fold) with the profile pre-merged over (forward, reverse) read-base pairs.

Tiles whose reads are all ACGT read one merged profile row per step; a tile with an N or IUPAC read base runs the
mixed main pass.  These tests place such bases where the forward and the reverse half of a row disagree (first / last
base, the self-mirrored middle row, rows whose mirror is also N, a whole read), cover every read length the kernel
takes, and size the allele table from max_hap_len on both sides of the 9- / 8-warp CTA switch.  Raw scores are
bit-exact against the CPU oracle, and the folded class must have taken every tile."""
import numpy as np
import pytest

from conftest import assert_same_triplets, to_oracle_batch

pytestmark = pytest.mark.gpu

FOLD = 7                                   # tile class of the folded kernel (vtx_last_tile_counts)
FLANK = 96                                 # both flanks common to ref and alt, the narrowest the folded kernel takes
NIB = {ord("="): 0, ord("A"): 1, ord("C"): 2, ord("R"): 5, ord("G"): 4, ord("T"): 8, ord("N"): 15}
ACGT = np.frombuffer(b"ACGT", np.uint8)


@pytest.fixture(scope="module")
def vb():
    import vartrix_b200
    return vartrix_b200


def _rand(rng, n):
    return ACGT[rng.integers(0, 4, n)]


def _locus(rng, mid_ref, mid_alt):
    left, right = _rand(rng, FLANK), _rand(rng, FLANK)
    mr = _rand(rng, mid_ref)
    ma = np.resize(mr, mid_alt).copy()
    ma[int(rng.integers(0, mid_alt))] = ACGT[rng.integers(0, 4)]
    return np.concatenate([left, mr, right]), np.concatenate([left, ma, right])


def _read(rng, ref, alt, m):
    """m bases of a haplotype (hanging over an end at times) with a few substitutions."""
    src = ref if rng.random() < 0.5 else alt
    s0 = int(rng.integers(-10, len(src) - max(1, m // 2)))
    seq = np.array([src[j] if 0 <= j < len(src) else ACGT[rng.integers(0, 4)] for j in range(s0, s0 + m)], np.uint8)
    for _ in range(int(rng.integers(0, 3))):
        seq[int(rng.integers(0, m))] = ACGT[rng.integers(0, 4)]
    return seq


def _batch(vb, loci):
    """loci: [(ref, alt, [read, ...])] as uint8 arrays -> (StagedBatch, pair_read, pair_locus)."""
    haps, ref_off, ref_len, alt_off, alt_len = bytearray(), [], [], [], []
    nibs, read_off, read_len, pair_locus = bytearray(), [], [], []
    for l, (ref, alt, reads) in enumerate(loci):
        for h, offs, lens in ((ref, ref_off, ref_len), (alt, alt_off, alt_len)):
            while len(haps) % 16: haps.append(0)
            offs.append(len(haps)); lens.append(len(h)); haps.extend(bytes(h))
        for seq in reads:
            codes = np.array([NIB[int(c)] for c in seq], np.uint8)
            if len(codes) & 1: codes = np.concatenate([codes, np.zeros(1, np.uint8)])
            while len(nibs) % 16: nibs.append(0)
            read_off.append(len(nibs)); read_len.append(len(seq)); pair_locus.append(l)
            nibs.extend(((codes[0::2] << 4) | codes[1::2]).astype(np.uint8).tobytes())
    while len(nibs) % 16: nibs.append(0)
    n_reads, n_loci = len(read_len), len(loci)
    cand_start = np.concatenate([[0], np.cumsum([len(r) for _, _, r in loci])]).astype(np.uint64)
    sb = vb.StagedBatch(
        locus_row=np.arange(n_loci), hap_bytes=np.frombuffer(bytes(haps), np.uint8), ref_off=ref_off, ref_len=ref_len,
        alt_off=alt_off, alt_len=alt_len, cand_start=cand_start, read_nib=np.frombuffer(bytes(nibs), np.uint8),
        read_off=read_off, read_len=read_len, cb_bytes=np.zeros(0, np.uint8), read_cb_off=np.full(n_reads, vb.engine.NO_CB),
        read_cb_len=np.zeros(n_reads), read_umi_key=np.full(n_reads, vb.engine.NO_UMI, np.uint64),
        cand_read=np.arange(n_reads), n_rows=n_loci)
    return sb, np.arange(n_reads, dtype=np.uint32), np.array(pair_locus, np.uint32)


def _check_raw_scores(vb, oracle, loci):
    sb, pr, pl = _batch(vb, loci)
    ors, oas = oracle.score_pairs(to_oracle_batch(oracle, sb), pr, pl, n_threads=8)
    with vb.Engine("coverage") as eng:
        rs, as_ = eng.score_pairs(sb, pr, pl)
        tiles = eng.tile_counts()
    assert tiles[FOLD] > 0 and sum(tiles) == tiles[FOLD], tiles
    bad = np.nonzero((rs.astype(np.int32) != ors) | (as_.astype(np.int32) != oas))[0]
    assert bad.size == 0, (bad[:5], rs[bad[:5]], ors[bad[:5]], as_[bad[:5]], oas[bad[:5]])


def _with_n(seq, rows, base=ord("N")):
    seq = seq.copy()
    seq[list(rows)] = base
    return seq


def _n_placements(m):
    """Rows to overwrite with N in a read of m bases: each placement stresses another half of the mixed row word."""
    out = [[0], [m - 1], [0, m - 1]]                                  # first / last base (and the mirror of each other)
    if m & 1:
        out.append([(m - 1) // 2])                                   # the self-mirrored middle row
    if m >= 6:
        out.append([1, m - 2, 3, m - 4])                             # rows whose mirror is also N
        out.append([2])                                              # mirror is an ordinary base
    out.append(list(range(m)))                                       # the whole read
    return out


@pytest.mark.parametrize("base", ["N", "R", "="])
def test_one_read_of_four_with_a_non_acgt_base(vb, oracle, base):
    rng = np.random.default_rng(1000 + ord(base))
    loci = []
    for m in (1, 2, 3, 7, 8, 75, 150, 151, 152):
        for rows in _n_placements(m):
            ref, alt = _locus(rng, 9, 9)
            reads = [_read(rng, ref, alt, int(rng.integers(max(1, m - 20), 153))) for _ in range(4)]
            k = int(rng.integers(0, 4))
            reads[k] = _with_n(_read(rng, ref, alt, m), rows, ord(base))
            loci.append((ref, alt, reads))
            if rng.random() < 0.5:                                   # an all-ACGT tile of the same kind next to it
                loci.append((ref, alt, [_read(rng, ref, alt, int(rng.integers(1, 153))) for _ in range(4)]))
    _check_raw_scores(vb, oracle, loci)


def test_every_read_length_the_folded_kernel_takes(vb, oracle):
    rng = np.random.default_rng(7)
    lengths = rng.permutation(np.arange(1, 153))
    loci = []
    for i in range(0, len(lengths), 4):
        ref, alt = _locus(rng, 9, 9)
        reads = [_read(rng, ref, alt, int(m)) for m in lengths[i:i + 4]]
        if i % 12 == 4:                                              # some of them in mixed tiles
            reads[0] = _with_n(reads[0], [int(rng.integers(0, len(reads[0])))])
        loci.append((ref, alt, reads))
    _check_raw_scores(vb, oracle, loci)


@pytest.mark.parametrize("width", [1, 19, 20, 40])
def test_allele_table_sized_from_the_widest_window(vb, oracle, width):
    """The widest allele (ref or alt) of the batch has `width` columns: the per-warp table holds exactly that many."""
    rng = np.random.default_rng(width)
    loci = []
    for l in range(48):
        wr = width if l % 3 == 0 else int(rng.integers(1, width + 1))
        wa = width if l % 3 == 1 else int(rng.integers(1, width + 1))
        ref, alt = _locus(rng, wr, wa)
        reads = [_read(rng, ref, alt, int(rng.integers(60, 153))) for _ in range(4 + l % 5)]
        if l % 7 == 0:
            reads[1] = _with_n(reads[1], [0, len(reads[1]) - 1])
        loci.append((ref, alt, reads))
    _check_raw_scores(vb, oracle, loci)


@pytest.mark.parametrize("promised_hap", [211, 212, 232])
def test_device_submit_with_a_wider_promised_window(vb, oracle, promised_hap):
    """A resident SNV shard (201-column windows) submitted with a larger max_hap_len: the allele table and the CTA shape
    follow the promise (mid_cap 19, 20 and 40 columns), the triplets stay the oracle's."""
    import torch
    sb, bcs, info = vb.synth.make_shard(300, 120, depth=30, seed=33, kind="snv")
    assert int(max(sb.ref_len.max(), sb.alt_len.max())) == 201
    exp = oracle.run_batch(to_oracle_batch(oracle, sb), oracle.Barcodes(bcs.keys), oracle.MODES["coverage"], False, n_threads=8)
    keep, db = [], sb.to_c()
    for f in vb.StagedBatch.FIELDS:
        a = getattr(sb, f)
        t = torch.from_numpy(a.view(np.uint8).reshape(-1) if a.dtype.itemsize > 1 else a.reshape(-1)).cuda()
        keep.append(t)
        setattr(db, f, t.data_ptr() if t.numel() else None)
    with vb.Engine("coverage") as eng:
        eng.set_barcodes(bcs)
        eng.submit_device(db, int(sb.read_len.max()), promised_hap)
        got = eng.fetch(eng.finish_device())
        tiles = eng.tile_counts()
    assert tiles[FOLD] > 0 and sum(tiles) == tiles[FOLD], tiles
    assert_same_triplets(got, exp)
    assert got.metrics == exp.metrics and got.metrics["num_scored"] == info["n_pairs"]
