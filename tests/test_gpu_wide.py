"""GPU parity tests for the multi-lane band kernels (bands 32..256, packed s16x2 and 32-bit lanes), the int-score mode,
reads the 16-bit lanes cannot take (large quality sums, long reads, 'N' at wide bands), long candidate lists and the
BASELINE shapes round 1 never checked against the oracle (H = 1024, C4's band 32 mix)."""
import numpy as np
import pytest

from helpers import ACGT, random_positions, random_region
from test_gpu_parity import _close, _oracle_scores, _tasks_for

pytestmark = pytest.mark.gpu


@pytest.mark.parametrize("band", [32, 64, 128, 256])
def test_align_scores_wide_bands_match_oracle(engine, coracle, band):
    rng = np.random.default_rng(500 + band)
    hap_len = 2 * band + 420
    haps, reads = random_region(rng, band, n_haps=5, n_reads=60, hap_len=hap_len, read_len_choices=[1, 7, 40, 76, 150, 151, 300],
                                read_n_rate=0.1, edge_reads=False)
    tasks = _tasks_for(rng, haps, reads, band, 500)
    want = _oracle_scores(coracle, haps, reads, band, tasks, 2)
    for bits in (16, 32):
        got = engine.align_scores(band, haps, reads, tasks, nuc_prior=2, precision_bits=bits)
        assert np.array_equal(got, want), (band, bits, np.nonzero(got != want)[0][:10], got[got != want][:10], want[got != want][:10])


def test_align_scores_long_and_high_quality_reads(engine, coracle):
    """Reads beyond the packed path: longer than its 1023-base bins, or a quality sum that does not fit a 16-bit lane."""
    from octopus_b200.batch import pack_haplotypes, pack_reads
    rng = np.random.default_rng(77)
    band = 64
    hap_len = 2600
    base = ACGT[rng.integers(0, 4, hap_len)]
    seqs = []
    for h in range(3):
        s = base.copy()
        s[rng.integers(0, hap_len, 20)] = ACGT[rng.integers(0, 4, 20)]
        seqs.append(s)
    haps = pack_haplotypes(seqs, [np.roll(s, 1) for s in seqs], [rng.integers(1, 126, hap_len).astype(np.int8) for _ in seqs],
                           [np.roll(s, -1) for s in seqs], [rng.integers(1, 126, hap_len).astype(np.int8) for _ in seqs],
                           [rng.integers(3, 46, hap_len).astype(np.int8) for _ in seqs], [rng.integers(1, 11, hap_len).astype(np.int8) for _ in seqs])
    bases, quals = [], []
    for L, q in ((800, 41), (1023, 20), (1024, 20), (1500, 30), (2300, 93), (900, 60)):
        p = int(rng.integers(0, hap_len - L))
        b = base[p:p + L].copy()
        b[rng.integers(0, L, L // 25)] = ACGT[rng.integers(0, 4, L // 25)]
        bases.append(b)
        quals.append(np.full(L, q, np.uint8))
    reads = pack_reads(bases, quals)
    tasks = _tasks_for(rng, haps, reads, band, 40)
    want = _oracle_scores(coracle, haps, reads, band, tasks, 2)
    for bits in (16, 32):
        got = engine.align_scores(band, haps, reads, tasks, nuc_prior=2, precision_bits=bits)
        assert np.array_equal(got, want), (bits, got, want)


@pytest.mark.parametrize("band_req", [33, 64, 100, 200])
def test_populate_wide_bands_match_oracle(engine, coracle, band_req):
    from octopus_b200 import HaplotypeLikelihoodModel
    rng = np.random.default_rng(600 + band_req)
    band = HaplotypeLikelihoodModel(HaplotypeLikelihoodModel.Config(max_indel_error=band_req)).pad_requirement()
    for trial in range(4):
        hap_len = 2 * band + int(rng.choice([200, 330]))
        haps, reads = random_region(rng, band, n_haps=int(rng.integers(1, 24)), n_reads=int(rng.integers(1, 50)), hap_len=hap_len,
                                    read_len_choices=[40, 76, 100, 150], read_n_rate=0.08, edge_reads=(trial % 2 == 0))
        positions = random_positions(rng, haps, reads) if trial % 2 else None
        flanks = (int(rng.integers(0, 90)), int(rng.integers(0, 90))) if trial == 3 else None
        for dp_only in (False, True):
            for int_scores in (False, True):
                cfg = HaplotypeLikelihoodModel.Config(max_indel_error=band_req, disable_naive_shortcut=dp_only, map_positions=False,
                                                      use_int_scores=int_scores)
                rc, want, wst = coracle.populate(band, haps, reads, positions, flanks, dp_only=dp_only, map_positions=False)
                got, st = engine.populate(cfg, haps, reads, positions, flanks, want_status=True)
                ok_pairs = wst == 0
                assert np.array_equal(st[~ok_pairs], wst[~ok_pairs])
                ok, worst = _close(got[ok_pairs], want[ok_pairs])
                assert ok, (band_req, trial, dp_only, int_scores, worst)


def test_populate_int_scores_and_unsafe_reads_equal_the_default(engine, coracle):
    """use_int_scores routes every read through the 32-bit lanes; reads whose quality sum overflows 16 bits go there on their
    own. Both must give the oracle's values (band 16 and 32, flank state and device mapper included)."""
    from octopus_b200 import HaplotypeLikelihoodModel
    rng = np.random.default_rng(31)
    for band in (16, 32):
        haps, reads = random_region(rng, band, n_haps=9, n_reads=80, hap_len=1000, read_len_choices=[76, 150, 700, 760], read_n_rate=0.05)
        reads.quals[:] = np.where(rng.random(len(reads.quals)) < 0.9, 41, reads.quals)      # long reads: quality sum ~ 30 000 > 16-bit budget
        for flanks in (None, (120, 150)):
            for mapit in (False, True):
                rc, want, wst = coracle.populate(band, haps, reads, None, flanks, map_positions=mapit)
                for int_scores in (False, True):
                    cfg = HaplotypeLikelihoodModel.Config(max_indel_error=band, use_int_scores=int_scores, map_positions=mapit)
                    got, st = engine.populate(cfg, haps, reads, None, flanks, want_status=True)
                    ok_pairs = wst == 0
                    assert np.array_equal(st[~ok_pairs], wst[~ok_pairs])
                    ok, worst = _close(got[ok_pairs], want[ok_pairs])
                    assert ok, (band, flanks, mapit, int_scores, worst)


def test_populate_long_candidate_lists(engine, coracle):
    """The reference takes mapping-position lists of any length (haplotype_likelihood_model.cpp:211-237): more than the k-mer mapper's
    10 per pair must neither be truncated nor overflow the task lists."""
    from octopus_b200 import HaplotypeLikelihoodModel
    from octopus_b200.batch import pack_positions
    rng = np.random.default_rng(41)
    band = 16
    haps, reads = random_region(rng, band, n_haps=6, n_reads=25, hap_len=400, read_len_choices=[60, 100], edge_reads=False)
    lists = [[sorted(set(int(x) for x in rng.integers(0, 400 - reads.length(r), int(rng.integers(0, 40))))) for r in range(reads.n)] for h in range(haps.n)]
    positions = pack_positions(lists, haps.n, reads.n)
    for flanks in (None, (50, 60)):
        for dp_only in (True, False):
            cfg = HaplotypeLikelihoodModel.Config(max_indel_error=band, disable_naive_shortcut=dp_only)
            rc, want, wst = coracle.populate(band, haps, reads, positions, flanks, dp_only=dp_only)
            got, st = engine.populate(cfg, haps, reads, positions, flanks, want_status=True)
            ok_pairs = wst == 0
            ok, worst = _close(got[ok_pairs], want[ok_pairs])
            assert ok, (flanks, dp_only, worst)


def test_populate_h1024_shape(engine, coracle):
    """C5's shape: 1024 haplotypes (the 16-bit haplotype field of the DP task word, per-read task lists of 1024 entries)."""
    from octopus_b200 import HaplotypeLikelihoodModel, synth
    haps, reads, band = synth.make_batch("C5", n_reads=48)
    assert haps.n == 1024
    cfg = HaplotypeLikelihoodModel.Config(max_indel_error=band, disable_naive_shortcut=True, map_positions=False)
    got = engine.populate(cfg, haps, reads)
    rc, want, _ = coracle.populate(band, haps, reads, dp_only=True, map_positions=False)
    assert rc == 0
    ok, worst = _close(got, want)
    assert ok, worst


def test_populate_c4_shape_vs_oracle(engine, coracle):
    """C4: band 32 (two lanes per alignment pair), mixed 76 / 150 / 250 bp reads, 500 bp haplotypes — against the oracle."""
    from octopus_b200 import HaplotypeLikelihoodModel, synth
    haps, reads, band = synth.make_batch("C4", n_reads=300, n_haps=40)
    assert band == 32
    for dp_only in (True, False):
        cfg = HaplotypeLikelihoodModel.Config(max_indel_error=band, disable_naive_shortcut=dp_only, map_positions=False)
        got = engine.populate(cfg, haps, reads)
        rc, want, _ = coracle.populate(band, haps, reads, dp_only=dp_only, map_positions=False)
        ok, worst = _close(got, want)
        assert ok, (dp_only, worst)


def test_populate_with_error_model_penalties(engine, coracle):
    """A region whose penalty arrays come from the reference's error models (reset()), haplotypes with tandem repeats: long constant
    runs and low penalties inside repeats, unlike the i.i.d. synthetic arrays."""
    from octopus_b200 import ErrorModel, HaplotypeLikelihoodModel
    from octopus_b200.batch import pack_reads
    rng = np.random.default_rng(53)
    hap_len, band = 420, 16
    base = ACGT[rng.integers(0, 4, hap_len)].copy()
    for motif, k, at in ((b"A", 18, 60), (b"CA", 12, 150), (b"GAT", 9, 230), (b"T", 9, 330)):
        rep = np.tile(np.frombuffer(motif, np.uint8), k)
        base[at:at + len(rep)] = rep
    seqs = []
    for h in range(12):
        s = base.copy()
        if h % 3 == 1:
            s = np.concatenate([s[:70], s[71:], ACGT[rng.integers(0, 4, 1)]])          # one A fewer in the homopolymer
        if h % 3 == 2:
            s = np.concatenate([s[:160], np.frombuffer(b"CA", np.uint8), s[160:-2]])   # one CA more
        s[rng.integers(0, hap_len, 2)] = ACGT[rng.integers(0, 4, 2)]
        seqs.append(s)
    haps = ErrorModel("PCR-free.HiSeq-2500").reset(seqs, begin=np.zeros(len(seqs), np.int64))
    bases, quals, begin = [], [], []
    for r in range(120):
        L = int(rng.choice([76, 100, 150]))
        p = int(rng.integers(0, hap_len - L))
        b = seqs[int(rng.integers(0, len(seqs)))][p:p + L].copy()
        for _ in range(int(rng.choice([0, 0, 1, 2]))):
            b[rng.integers(0, L)] = ACGT[rng.integers(0, 4)]
        bases.append(b); quals.append(rng.integers(2, 42, L).astype(np.uint8)); begin.append(p)
    reads = pack_reads(bases, quals, reverse=(rng.random(120) < 0.5).astype(np.uint8), begin=np.asarray(begin, np.int64))
    for flanks in (None, (40, 60)):
        for mapit in (False, True):
            cfg = HaplotypeLikelihoodModel.Config(max_indel_error=band, map_positions=mapit)
            got, st = engine.populate(cfg, haps, reads, None, flanks, want_status=True)
            rc, want, wst = coracle.populate(band, haps, reads, None, flanks, map_positions=mapit)
            ok_pairs = wst == 0
            assert np.array_equal(st[~ok_pairs], wst[~ok_pairs])
            ok, worst = _close(got[ok_pairs], want[ok_pairs])
            assert ok, (flanks, mapit, worst)


def test_device_mapper_takes_long_haplotypes(engine, coracle):
    """Round 1's mapper refused haplotypes above 2053 bp (per-thread vote arrays); the reference has no such limit. Now the votes
    live in shared-memory tiles of 2048 diagonals: several tiles, ties across tiles, long reads (16-bit counters)."""
    from octopus_b200 import HaplotypeLikelihoodModel
    from octopus_b200.batch import pack_haplotypes, pack_reads
    rng = np.random.default_rng(61)
    band = 16
    for hap_len, read_lens in ((5200, [100, 150]), (4500, [150, 300, 420])):
        base = ACGT[rng.integers(0, 4, hap_len)].copy()
        base[3000:3400] = base[600:1000]                 # a 400-base duplication: equal vote counts 2400 diagonals apart
        seqs = []
        for h in range(5):
            s = base.copy()
            s[rng.integers(0, hap_len, 12)] = ACGT[rng.integers(0, 4, 12)]
            seqs.append(s)
        haps = pack_haplotypes(seqs, [np.roll(s, 1) for s in seqs], [rng.integers(1, 126, hap_len).astype(np.int8) for _ in seqs],
                               [np.roll(s, -1) for s in seqs], [rng.integers(1, 126, hap_len).astype(np.int8) for _ in seqs],
                               [rng.integers(3, 46, hap_len).astype(np.int8) for _ in seqs], [rng.integers(1, 11, hap_len).astype(np.int8) for _ in seqs],
                               begin=np.zeros(5, np.int64))
        bases, quals, begin = [], [], []
        for r in range(40):
            L = int(rng.choice(read_lens))
            p = int(rng.choice([rng.integers(0, hap_len - L), rng.integers(600, 1000 - min(L, 399))]))
            b = base[p:p + L].copy()
            for _ in range(int(rng.integers(0, 3))):
                b[rng.integers(0, L)] = ACGT[rng.integers(0, 4)]
            bases.append(b); quals.append(rng.integers(10, 42, L).astype(np.uint8)); begin.append(p)
        reads = pack_reads(bases, quals, begin=np.asarray(begin, np.int64))
        for flanks in (None, (500, 700)):
            cfg = HaplotypeLikelihoodModel.Config(max_indel_error=band, map_positions=True)
            got, st = engine.populate(cfg, haps, reads, None, flanks, want_status=True)
            rc, want, wst = coracle.populate(band, haps, reads, None, flanks, map_positions=True)
            ok_pairs = wst == 0
            assert np.array_equal(st[~ok_pairs], wst[~ok_pairs])
            ok, worst = _close(got[ok_pairs], want[ok_pairs])
            assert ok, (hap_len, flanks, worst)


def test_lean_flank_kernel_geometries(engine, coracle):
    """Flank states from none to overlapping, short and long reads, qualities down to 0: the lean flank kernel, the crossing-cell
    kernel (narrow non-flank windows, reads with 'N'), the plain DP (flanks covering the window) and the traceback queue all meet
    the oracle."""
    from octopus_b200 import HaplotypeLikelihoodModel
    rng = np.random.default_rng(71)
    for band in (8, 16, 32):
        for trial in range(5):
            hap_len = int(rng.choice([300, 420]))
            haps, reads = random_region(rng, band, n_haps=int(rng.integers(2, 30)), n_reads=int(rng.integers(5, 60)), hap_len=hap_len,
                                        read_len_choices=[25, 40, 76, 100, 150], read_n_rate=0.1, edge_reads=(trial % 2 == 0))
            if trial == 4:
                reads.quals[rng.random(len(reads.quals)) < 0.1] = 0
            for flanks in ((0, 0), (30, 40), (int(hap_len * 0.45), int(hap_len * 0.45)), (hap_len // 2, hap_len // 2 + 5), (hap_len - 10, 0), (0, hap_len - 20)):
                for mapit in (False, True):
                    cfg = HaplotypeLikelihoodModel.Config(max_indel_error=band, map_positions=mapit)
                    got, st = engine.populate(cfg, haps, reads, None, flanks, want_status=True)
                    rc, want, wst = coracle.populate(band, haps, reads, None, flanks, map_positions=mapit)
                    ok_pairs = wst == 0
                    assert np.array_equal(st[~ok_pairs], wst[~ok_pairs])
                    ok, worst = _close(got[ok_pairs], want[ok_pairs])
                    assert ok, (band, trial, flanks, mapit, worst)


def test_reserved_sms_leave_results_unchanged(coracle):
    """phmm_reserve_sms: the DP blocks that land on reserved SMs exit and the others take their work; every mode's result is what it
    is without the reservation (and the oracle's)."""
    from octopus_b200 import HaplotypeLikelihoodModel, PairHMMEngine
    rng = np.random.default_rng(97)
    eng = PairHMMEngine(0)
    for band, flanks, mapit in ((16, None, False), (16, (30, 40), True), (32, None, True), (64, None, False)):
        haps, reads = random_region(rng, band, n_haps=40, n_reads=3000, hap_len=2 * band + 300, read_len_choices=[76, 100, 150], read_n_rate=0.02)
        cfg = HaplotypeLikelihoodModel.Config(max_indel_error=band, disable_naive_shortcut=not mapit, map_positions=mapit)
        eng.reserve_sms(0)
        base = eng.populate(cfg, haps, reads, None, flanks)
        for n in (8, 100, 147, 10**6):
            eng.reserve_sms(n)
            assert np.array_equal(eng.populate(cfg, haps, reads, None, flanks), base), (band, n)
        rc, want, wst = coracle.populate(band, haps, reads, None, flanks, dp_only=not mapit, map_positions=mapit)
        ok, worst = _close(base[wst == 0], want[wst == 0])
        assert ok, (band, worst)
    eng.close()


def test_two_engines_share_the_kernels_shared_memory_limit(engine):
    """The dynamic shared-memory limit of a kernel is per process: a second engine that needs LESS than the first must not lower it
    (the first engine's next launch would fail with 'invalid argument'). Regression test of the engine's high-water bookkeeping."""
    from octopus_b200 import HaplotypeLikelihoodModel, PairHMMEngine
    rng = np.random.default_rng(131)
    other = PairHMMEngine(0)
    for band in (16, 32):
        cfg = HaplotypeLikelihoodModel.Config(max_indel_error=band, disable_naive_shortcut=True, map_positions=False)
        long_h, long_r = random_region(rng, band, n_haps=24, n_reads=400, hap_len=2 * band + 420, read_len_choices=[250], read_n_rate=0.0)
        short_h, short_r = random_region(rng, band, n_haps=24, n_reads=400, hap_len=2 * band + 120, read_len_choices=[40], read_n_rate=0.0)
        first = engine.populate(cfg, long_h, long_r)
        other.populate(cfg, short_h, short_r)
        assert np.array_equal(engine.populate(cfg, long_h, long_r), first), band
        assert np.array_equal(other.populate(cfg, long_h, long_r), first), band
    other.close()


def test_populate_regions_equals_one_call_per_region(engine, coracle):
    """phmm_populate_regions: many small regions (ragged haplotype and read counts, own flank states) in one kernel chain give, region
    by region, what phmm_populate gives for the region alone — and the oracle's values."""
    from octopus_b200 import HaplotypeLikelihoodModel
    from octopus_b200.batch import concat_blocks
    rng = np.random.default_rng(83)
    for band, mapit, dp_only in ((8, False, True), (16, True, False), (16, False, False), (32, True, False), (64, False, True)):
        hap_blocks, read_blocks, flanks = [], [], []
        for g in range(int(rng.integers(3, 9))):
            hap_len = 2 * band + int(rng.choice([200, 260, 330]))
            h, r = random_region(rng, band, n_haps=int(rng.integers(1, 45)), n_reads=int(rng.integers(1, 70)), hap_len=hap_len,
                                 read_len_choices=[40, 76, 100, 150], read_n_rate=0.05, edge_reads=(g % 2 == 0))
            hap_blocks.append(h); read_blocks.append(r)
            flanks.append((int(rng.integers(0, 80)), int(rng.integers(0, 80))) if g % 3 else None)
        haps, reads, hf, rf = concat_blocks(hap_blocks, read_blocks)
        cfg = HaplotypeLikelihoodModel.Config(max_indel_error=band, disable_naive_shortcut=dp_only, map_positions=mapit)
        flat, off, st = engine.populate_regions(cfg, haps, reads, hf, rf, flank_states=flanks, want_status=True)
        mats = engine.split_regions(flat, off, hf, rf)
        sts = engine.split_regions(st, off, hf, rf)
        for g, (h, r) in enumerate(zip(hap_blocks, read_blocks)):
            rc, want, wst = coracle.populate(band, h, r, None, flanks[g], dp_only=dp_only, map_positions=mapit)
            ok_pairs = wst == 0
            assert np.array_equal(sts[g][~ok_pairs], wst[~ok_pairs]), (band, g)
            ok, worst = _close(mats[g][ok_pairs], want[ok_pairs])
            assert ok, (band, mapit, g, worst)
            one, _ = engine.populate(cfg, h, r, None, flanks[g], want_status=True)
            assert np.array_equal(one[ok_pairs], mats[g][ok_pairs]), (band, g)


def test_align_reads_register_traceback_and_fallbacks(engine, coracle):
    """phmm_align_reads with the register traceback kernel (bands <= 32) and the generic kernel side by side: long reads beyond the
    register kernel's shared-memory budget, reads with 'N', wide bands — each pair against HaplotypeLikelihoodModel::align (oracle)."""
    from octopus_b200 import HaplotypeLikelihoodModel
    from test_gpu_parity import REL_TOL
    rng = np.random.default_rng(97)
    for band_req, lens, hap_len in ((8, [30, 76], 300), (16, [76, 150, 900], 1200), (32, [100, 250], 600), (64, [100, 150], 500)):
        band = HaplotypeLikelihoodModel(HaplotypeLikelihoodModel.Config(max_indel_error=band_req)).pad_requirement()
        haps, reads = random_region(rng, band, n_haps=5, n_reads=50, hap_len=hap_len, read_len_choices=lens, read_n_rate=0.15, edge_reads=True)
        pairs = np.array([(int(rng.integers(0, reads.n)), int(rng.integers(0, haps.n))) for _ in range(250)], dtype=np.int32)
        lists, off = [], [0]
        for r, h in pairs:
            p0 = int(reads.begin[r])
            ps = sorted({int(np.clip(p0 + rng.integers(-10, 11), 0, haps.length(h))) for _ in range(int(rng.integers(0, 4)))})
            lists.extend(ps); off.append(len(lists))
        positions = (np.asarray(off, np.int64), np.asarray(lists if lists else [0], np.int32))
        flanks = (int(rng.integers(0, 80)), int(rng.integers(0, 80))) if band_req != 16 else None
        cfg = HaplotypeLikelihoodModel.Config(max_indel_error=band_req)
        mp, lk, cig, st = engine.align_reads(cfg, haps, reads, pairs, positions, flanks)
        for j, (r, h) in enumerate(pairs):
            hp = haps.hap(int(h)); b, q = reads.read(int(r)); rev = bool(reads.reverse[r])
            wst, wmp, wlk, wcig, wext = coracle.model_align(band, hp["seq"].tobytes(), b.tobytes(), q, hp["gap_open"], hp["gap_extend"],
                                                            hp["snv_mask_rev" if rev else "snv_mask_fwd"].tobytes(), hp["snv_prior_rev" if rev else "snv_prior_fwd"],
                                                            positions[1][off[j]:off[j + 1]], int(reads.begin[r]), mapping_quality=int(reads.mapq[r]), flanks=flanks)
            if wst == 1:
                assert (st[j] & 0xFFFF) == 2 and (st[j] >> 16) == wext
                continue
            assert wst == 0 and st[j] == 0, (band_req, j, wst, st[j])
            assert mp[j] == wmp and cig[j] == wcig, (band_req, j, mp[j], wmp, cig[j], wcig)
            assert abs(lk[j] - wlk) <= REL_TOL * max(abs(wlk), 1e-300)


def test_align_pairs_equals_the_mutation_model_hmm(engine, refhmm):
    """N4: phmm_align_pairs on (target haplotype, padded given haplotype) pairs == hmm::PairHMM<VariableGapExtendMutationModel, 32, int>::align,
    the call DeNovoModel makes (denovo_model.cpp:249-262): no SNV mask, scalar mismatch penalty, band 32, offset = band."""
    from octopus_b200 import HaplotypeLikelihoodModel
    from octopus_b200.batch import pack_haplotypes, pack_reads
    rng = np.random.default_rng(101)
    band, mismatch = 32, 40
    truths, targets, pairs = [], [], []
    base = ACGT[rng.integers(0, 4, 260)]
    for h in range(12):
        s = base.copy()
        for _ in range(int(rng.integers(0, 4))):
            s[rng.integers(0, len(s))] = ACGT[rng.integers(0, 4)]
        if h % 3 == 1:
            i = int(rng.integers(20, 200)); s = np.concatenate([s[:i], s[i + int(rng.integers(1, 8)):]])
        if h % 3 == 2:
            i = int(rng.integers(20, 200)); s = np.concatenate([s[:i], ACGT[rng.integers(0, 4, int(rng.integers(1, 8)))], s[i:]])
        targets.append(s)
        truths.append(np.concatenate([np.full(band, ord("N"), np.uint8), s, np.full(band, ord("N"), np.uint8)]))     # pad_given (denovo_model.cpp:206-220)
    go = [rng.integers(20, 60, len(t)).astype(np.int8) for t in truths]
    ge = [rng.integers(1, 11, len(t)).astype(np.int8) for t in truths]
    tb = pack_haplotypes(truths, [np.zeros(len(t), np.uint8) for t in truths], [np.full(len(t), 100, np.int8) for t in truths],
                         [np.zeros(len(t), np.uint8) for t in truths], [np.full(len(t), 100, np.int8) for t in truths], go, ge)
    rb = pack_reads(targets, [np.full(len(t), mismatch, np.uint8) for t in targets])
    for a in range(12):
        for b in range(12):
            if abs(len(targets[a]) - (len(truths[b]) - 2 * band)) < band:              # can_try_align_with_hmm (:244-247)
                pairs.append((a, b))
    pairs = np.asarray(pairs, np.int32)
    cfg = HaplotypeLikelihoodModel.Config(max_indel_error=band, use_mapping_quality=False, use_int_scores=True)
    off, lk, cig, st = engine.align_pairs(cfg, tb, rb, pairs, np.full(len(pairs), band, np.int32))
    for j, (a, b) in enumerate(pairs):
        rc, woff, wlk, wcig = refhmm.align_mutation_model(truths[b].tobytes(), targets[a].tobytes(), mismatch, go[b], ge[b])
        if rc == 2:
            assert st[j] == 4
            continue
        assert rc == 0 and st[j] == 0, (j, rc, st[j])
        assert (off[j], cig[j]) == (woff, wcig) and lk[j] == wlk, (j, off[j], woff, cig[j], wcig, lk[j], wlk)
