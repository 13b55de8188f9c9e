"""GPU parity tests: the CUDA engine (through the C ABI) against the oracle on the same seeded inputs.
Integer scores must be bit-exact; final ln-likelihoods must agree to 1e-4 relative (BASELINE.json's bar) — in fact the
only floating-point work is the double-precision epilogue, so the observed difference is a few ulp."""
import numpy as np
import pytest

from helpers import random_positions, random_region

pytestmark = pytest.mark.gpu

REL_TOL = 1e-4


def _tasks_for(rng, haps, reads, band, n):
    t = np.zeros((n, 4), dtype=np.int32)
    k = 0
    while k < n:
        r, h = int(rng.integers(0, reads.n)), int(rng.integers(0, haps.n))
        room = haps.length(h) - (reads.length(r) + 2 * band - 1)
        if room < 0:
            continue
        t[k] = (r, h, int(rng.integers(0, room + 1)), int(rng.integers(0, 2)))
        k += 1
    return t


def _oracle_scores(coracle, haps, reads, band, tasks, nuc):
    out = np.empty(len(tasks), dtype=np.int32)
    for j, (r, h, a, rev) in enumerate(tasks):
        hp = haps.hap(int(h))
        b, q = reads.read(int(r))
        W = len(b) + 2 * band - 1
        m = hp["snv_mask_rev" if rev else "snv_mask_fwd"][a:a + W]
        p = hp["snv_prior_rev" if rev else "snv_prior_fwd"][a:a + W]
        out[j] = coracle.align(band, hp["seq"][a:a + W].tobytes(), b.tobytes(), q.astype(np.int8), hp["gap_open"][a:a + W],
                               hp["gap_extend"][a:a + W], nuc, m.tobytes(), p)
    return out


def test_align_scores_reference_kats(engine, kats):
    from octopus_b200.batch import pack_haplotypes, pack_reads
    for bits in (16, 32):
        for c in kats:
            W = len(c["truth"])
            haps = pack_haplotypes([c["truth"]], [np.zeros(W, np.uint8)], [np.full(W, 100, np.int8)], [np.zeros(W, np.uint8)],
                                   [np.full(W, 100, np.int8)], [np.asarray(c["gap_open"], np.int8)], [np.full(W, c["gap_extend"], np.int8)])
            reads = pack_reads([c["read"]], [np.asarray(c["quals"], np.uint8)])
            s = engine.align_scores(c["band"], haps, reads, np.array([[0, 0, 0, 0]], np.int32), nuc_prior=c["nuc_prior"], precision_bits=bits)
            assert int(s[0]) == c["score"], (c["suite"], c["index"], bits)


@pytest.mark.parametrize("band", [8, 16, 32, 64])
def test_align_scores_match_oracle(engine, coracle, band):
    rng = np.random.default_rng(100 + band)
    haps, reads = random_region(rng, band, n_haps=7, n_reads=90, hap_len=330, read_len_choices=[1, 5, 33, 76, 100, 150, 151],
                                read_n_rate=0.1, edge_reads=False)
    tasks = _tasks_for(rng, haps, reads, band, 1500)
    for nuc in (2, 4):
        want = _oracle_scores(coracle, haps, reads, band, tasks, nuc)
        for bits in (16, 32):
            got = engine.align_scores(band, haps, reads, tasks, nuc_prior=nuc, precision_bits=bits)
            assert np.array_equal(got, want), (band, nuc, bits, np.nonzero(got != want)[0][:10])
    assert engine.launch_count() >= 3


def test_align_scores_match_reference_kernel(engine, refkernels):
    from octopus_b200 import synth
    haps, reads, band = synth.make_batch("C2", n_reads=600, n_haps=16)
    rng = np.random.default_rng(9)
    tasks = _tasks_for(rng, haps, reads, band, 6000)
    got = engine.align_scores(band, haps, reads, tasks, nuc_prior=2)
    k = next(iter(refkernels.values()))
    batch = dict(read_bases=reads.bases, read_quals=reads.quals, read_off=reads.off, hap_seq=haps.seq,
                 hap_mask_fwd=haps.snv_mask_fwd, hap_prior_fwd=haps.snv_prior_fwd, hap_mask_rev=haps.snv_mask_rev,
                 hap_prior_rev=haps.snv_prior_rev, hap_gap_open=haps.gap_open, hap_gap_extend=haps.gap_extend, hap_off=haps.off)
    for rev in (0, 1):
        sel = tasks[:, 3] == rev
        want = k.align_batch(band, batch, tasks[sel, 0], tasks[sel, 1], tasks[sel, 2], nuc_prior=2, nthreads=2, strand_rev=bool(rev))
        assert np.array_equal(got[sel], want)


def _close(got, want):
    got, want = np.asarray(got), np.asarray(want)
    denom = np.maximum(np.abs(want), 1e-300)
    bad = np.abs(got - want) > REL_TOL * denom
    return not bad.any(), float(np.max(np.abs(got - want) / denom))


@pytest.mark.parametrize("band_req", [8, 12, 16, 32, 40])
def test_populate_matches_oracle(engine, coracle, band_req):
    from octopus_b200 import HaplotypeLikelihoodModel
    rng = np.random.default_rng(200 + band_req)
    band = HaplotypeLikelihoodModel(HaplotypeLikelihoodModel.Config(max_indel_error=band_req)).pad_requirement()
    for trial in range(6):
        hap_len = int(rng.choice([260, 300, 420]))
        haps, reads = random_region(rng, band, n_haps=int(rng.integers(1, 40)), n_reads=int(rng.integers(1, 70)), hap_len=hap_len,
                                    read_len_choices=[40, 76, 100, 150], read_n_rate=0.05, edge_reads=(trial % 2 == 0))
        positions = random_positions(rng, haps, reads) if trial % 3 else None
        flanks = (int(rng.integers(0, 90)), int(rng.integers(0, 90))) if trial % 2 else None
        for dp_only in (False, True):
            for use_mq in (True, False):
                mapit = (trial % 3 == 0) and (trial % 2 == 0 or dp_only)      # positions=None: k-mer mapped on the device, or original only
                # trial 5: a trigger at or above the cap is ignored (haplotype_likelihood_model.cpp:49-51); trial 3: a low cap that bites
                trig, cap = {1: (40, 120), 3: (40, 50), 5: (200, 50)}.get(trial, (None, 120))
                cfg = HaplotypeLikelihoodModel.Config(max_indel_error=band_req, use_mapping_quality=use_mq, mapping_quality_cap=cap,
                                                      mapping_quality_cap_trigger=trig, disable_naive_shortcut=dp_only,
                                                      map_positions=mapit)
                rc, want, wst = coracle.populate(band, haps, reads, positions, flanks, use_mapping_quality=use_mq, mapq_cap=cap,
                                                 mapq_cap_trigger=-1 if trig is None else trig, dp_only=dp_only, map_positions=mapit)
                got, st = engine.populate(cfg, haps, reads, positions, flanks, want_status=True)
                ok_pairs = wst == 0
                assert np.array_equal((st & 0xFFFF) == 2, (wst & 0xFFFF) == 2)
                assert np.array_equal(st[~ok_pairs], wst[~ok_pairs])
                if not use_mq:
                    assert np.array_equal(got[ok_pairs], want[ok_pairs]), (band_req, trial, dp_only)   # -ln10/10 * integer: exact
                ok, worst = _close(got[ok_pairs], want[ok_pairs])
                assert ok, (band_req, trial, dp_only, use_mq, worst)


def test_populate_raises_short_haplotype_error(engine):
    from octopus_b200 import HaplotypeLikelihoodModel, ShortHaplotypeError
    from octopus_b200.batch import pack_haplotypes, pack_reads
    rng = np.random.default_rng(3)
    s = np.frombuffer(b"ACGT", np.uint8)[rng.integers(0, 4, 60)]
    haps = pack_haplotypes([s], [s], [np.full(60, 50, np.int8)], [s], [np.full(60, 50, np.int8)], [np.full(60, 30, np.int8)], [np.full(60, 3, np.int8)])
    reads = pack_reads([s[5:55]], [np.full(50, 30, np.uint8)], begin=np.array([5]))
    with pytest.raises(ShortHaplotypeError):
        engine.populate(HaplotypeLikelihoodModel.Config(max_indel_error=16, map_positions=False), haps, reads)


def test_populate_device_resident_inputs_equal_host_inputs(engine):
    import torch
    from octopus_b200 import HaplotypeLikelihoodModel, synth
    haps, reads, band = synth.make_batch("C2", n_reads=3000, n_haps=32)
    cfg = HaplotypeLikelihoodModel.Config(max_indel_error=band)
    host = engine.populate(cfg, haps, reads)
    dev = engine.populate(cfg, haps.to_device("cuda:0"), reads.to_device("cuda:0"))
    assert isinstance(dev, torch.Tensor) and dev.is_cuda
    assert np.array_equal(dev.cpu().numpy(), host)


def test_packed_16bit_path_equals_int32_path_at_scale(engine):
    """Two independent GPU implementations (packed s16x2 register kernel vs the int32 generic kernel, selected by
    use_int_scores) must produce the same matrix — a size-independent check run well beyond oracle-sized inputs."""
    from octopus_b200 import HaplotypeLikelihoodModel, synth
    for name, nr, nh in (("C2", 20000, 64), ("C4", 6000, 24)):
        haps, reads, band = synth.make_batch(name, n_reads=nr, n_haps=nh)
        a = engine.populate(HaplotypeLikelihoodModel.Config(max_indel_error=band, disable_naive_shortcut=True, map_positions=False), haps, reads)
        b = engine.populate(HaplotypeLikelihoodModel.Config(max_indel_error=band, disable_naive_shortcut=True, use_int_scores=True, map_positions=False), haps, reads)
        assert np.array_equal(a, b), name


def test_traceback_seam_reproduces_reference_kats(engine, kats, coracle):
    """phmm_align_traceback == the reference's traceback overload: score, first_pos and both alignment strings of every KAT,
    and the oracle's traceback on random SNV-mask inputs."""
    for c in kats:
        got = engine.align(c["band"], c["truth"], c["read"], c["quals"], c["gap_open"], c["gap_extend"], c["nuc_prior"])
        assert got == (c["score"], c["first_pos"], c["align_truth"], c["align_read"]), (c["suite"], c["index"])
    from helpers import random_alignment_case
    rng = np.random.default_rng(77)
    for _ in range(60):
        band = int(rng.choice([8, 16, 32, 64]))
        c = random_alignment_case(rng, band, int(rng.integers(1, 120)))
        q8 = c["quals"].astype(np.int8)
        got = engine.align(band, c["truth"].tobytes(), c["read"].tobytes(), q8, c["gap_open"], c["gap_extend"], 3, c["snv_mask"].tobytes(), c["snv_prior"])
        want = coracle.align_tb(band, c["truth"].tobytes(), c["read"].tobytes(), q8, c["gap_open"], c["gap_extend"], 3, c["snv_mask"].tobytes(), c["snv_prior"])
        assert got == want


def test_populate_with_device_kmer_mapper_matches_reference_loop(engine, coracle):
    """positions = None and map_positions = 1: the engine maps every (haplotype, read) pair with the reference's K=6 k-mer
    mapper on the device, exactly as HaplotypeLikelihoodArray::populate does inline (haplotype_likelihood_array.cpp:89-92)."""
    from octopus_b200 import HaplotypeLikelihoodModel, synth
    haps, reads, band = synth.make_batch("C2", n_reads=700, n_haps=24)
    for flanks in (None, (40, 30)):
        cfg = HaplotypeLikelihoodModel.Config(max_indel_error=band)
        got = engine.populate(cfg, haps, reads, flank_state=flanks)
        rc, want, _ = coracle.populate(band, haps, reads, None, flanks, map_positions=True)
        assert rc == 0
        ok, worst = _close(got, want)
        assert ok, worst
    # repetitive haplotypes: many equally good mapping positions (exercises the <= 10 cap and the tie order)
    rng = np.random.default_rng(4)
    unit = np.frombuffer(b"ACGTTGCAAG", dtype=np.uint8)
    rep = np.tile(unit, 40)[:360]
    from octopus_b200.batch import pack_haplotypes, pack_reads
    seqs = []
    for h in range(5):
        s = rep.copy(); s[rng.integers(0, 360, 3)] = np.frombuffer(b"ACGT", np.uint8)[rng.integers(0, 4, 3)]; seqs.append(s)
    n = 360
    haps2 = pack_haplotypes(seqs, [np.roll(s, 1) for s in seqs], [np.full(n, 60, np.int8)] * 5, [np.roll(s, -1) for s in seqs], [np.full(n, 60, np.int8)] * 5,
                            [rng.integers(3, 46, n).astype(np.int8) for _ in range(5)], [rng.integers(1, 11, n).astype(np.int8) for _ in range(5)])
    rb, rq, rbeg = [], [], []
    for r in range(40):
        p = int(rng.integers(20, 200)); L = int(rng.choice([50, 100]))
        b = seqs[int(rng.integers(0, 5))][p:p + L].copy()
        if r % 2: b[rng.integers(0, L)] = ord("A")
        rb.append(b); rq.append(rng.integers(10, 41, L).astype(np.uint8)); rbeg.append(p)
    reads2 = pack_reads(rb, rq, begin=np.asarray(rbeg))
    got = engine.populate(HaplotypeLikelihoodModel.Config(max_indel_error=16), haps2, reads2)
    rc, want, _ = coracle.populate(16, haps2, reads2, None, None, map_positions=True)
    ok, worst = _close(got, want)
    assert rc == 0 and ok, worst


def test_align_reads_matches_reference_align(engine, coracle):
    """phmm_align_reads == HaplotypeLikelihoodModel::align: mapping position, likelihood and CIGAR of the best alignment."""
    from octopus_b200 import HaplotypeLikelihoodModel
    rng = np.random.default_rng(31)
    for trial in range(4):
        band_req = [8, 16, 30, 16][trial]
        band = HaplotypeLikelihoodModel(HaplotypeLikelihoodModel.Config(max_indel_error=band_req)).pad_requirement()
        haps, reads = random_region(rng, band, n_haps=6, n_reads=40, hap_len=300, read_len_choices=[40, 76, 120], read_n_rate=0.1,
                                    edge_reads=(trial % 2 == 0))
        pairs = np.array([(int(rng.integers(0, reads.n)), int(rng.integers(0, haps.n))) for _ in range(300)], dtype=np.int32)
        lists, off = [], [0]
        for r, h in pairs:
            p0 = int(reads.begin[r])
            ps = sorted({int(np.clip(p0 + rng.integers(-10, 11), 0, haps.length(h))) for _ in range(int(rng.integers(0, 4)))})
            lists.extend(ps); off.append(len(lists))
        positions = (np.asarray(off, np.int64), np.asarray(lists if lists else [0], np.int32))
        flanks = (int(rng.integers(0, 80)), int(rng.integers(0, 80))) if trial % 2 else None
        cfg = HaplotypeLikelihoodModel.Config(max_indel_error=band_req, mapping_quality_cap_trigger=40 if trial == 3 else None)
        mp, lk, cig, st = engine.align_reads(cfg, haps, reads, pairs, positions, flanks)
        for j, (r, h) in enumerate(pairs):
            hp = haps.hap(int(h)); b, q = reads.read(int(r)); rev = bool(reads.reverse[r])
            wst, wmp, wlk, wcig, wext = coracle.model_align(band, hp["seq"].tobytes(), b.tobytes(), q, hp["gap_open"], hp["gap_extend"],
                                                            hp["snv_mask_rev" if rev else "snv_mask_fwd"].tobytes(), hp["snv_prior_rev" if rev else "snv_prior_fwd"],
                                                            positions[1][off[j]:off[j + 1]], int(reads.begin[r]), mapping_quality=int(reads.mapq[r]),
                                                            flanks=flanks, mapq_cap_trigger=40 if trial == 3 else -1)
            if wst == 1:
                assert (st[j] & 0xFFFF) == 2 and (st[j] >> 16) == wext
                continue
            assert wst == 0 and st[j] == 0, (trial, j, wst, st[j])
            assert mp[j] == wmp and cig[j] == wcig, (trial, j, mp[j], wmp, cig[j], wcig)
            assert abs(lk[j] - wlk) <= REL_TOL * max(abs(wlk), 1e-300)


def test_genotype_likelihood_reduction_on_the_resident_matrix(engine, coracle):
    """N1: ConstantMixtureGenotypeLikelihoodModel::evaluate over the matrix populate left on the device."""
    import itertools
    import torch
    from octopus_b200 import HaplotypeLikelihoodModel, synth
    haps, reads, band = synth.make_batch("C2", n_reads=4000, n_haps=12)
    m_dev = engine.populate(HaplotypeLikelihoodModel.Config(max_indel_error=band), haps.to_device("cuda:0"), reads.to_device("cuda:0"))
    m = m_dev.cpu().numpy()
    for ploidy in (1, 2, 3, 4):
        gts = np.array(list(itertools.combinations_with_replacement(range(12), ploidy))[:400], dtype=np.int32)
        want = coracle.genotype_likelihoods(m, gts)
        got_dev = engine.genotype_likelihoods(m_dev, gts)
        got_host = engine.genotype_likelihoods(m, gts)
        assert isinstance(got_dev, torch.Tensor)
        for got in (got_dev.cpu().numpy(), got_host):
            assert np.all(np.abs(got - want) <= 1e-9 * np.maximum(np.abs(want), 1.0)), ploidy


def test_populate_edge_cases(engine, coracle):
    """Single pair; qualities above 127 (the reference reinterprets them as int8, pair_hmm.hpp:372); reads longer than the
    fast path's row budget; wide bands (generic int32 kernels); int32 scores requested."""
    from octopus_b200 import HaplotypeLikelihoodModel
    from octopus_b200.batch import pack_haplotypes, pack_reads
    rng = np.random.default_rng(99)
    acgt = np.frombuffer(b"ACGT", np.uint8)

    def region(hap_len, read_lens, n_haps, qmax):
        seqs = [acgt[rng.integers(0, 4, hap_len)] for _ in range(n_haps)]
        haps = pack_haplotypes(seqs, [np.roll(s, 1) for s in seqs], [rng.integers(1, 126, hap_len).astype(np.int8) for _ in seqs],
                               [np.roll(s, -1) for s in seqs], [rng.integers(1, 126, hap_len).astype(np.int8) for _ in seqs],
                               [rng.integers(3, 46, hap_len).astype(np.int8) for _ in seqs], [rng.integers(1, 11, hap_len).astype(np.int8) for _ in seqs])
        bases, quals, begin = [], [], []
        for L in read_lens:
            p = int(rng.integers(0, hap_len - L + 1))
            b = seqs[int(rng.integers(0, n_haps))][p:p + L].copy()
            for _ in range(3):
                b[rng.integers(0, L)] = acgt[rng.integers(0, 4)]
            bases.append(b); quals.append(rng.integers(2, qmax + 1, L).astype(np.uint8)); begin.append(p)
        return haps, pack_reads(bases, quals, begin=np.asarray(begin))

    cases = [
        (dict(hap_len=120, read_lens=[40], n_haps=1, qmax=41), dict(max_indel_error=8)),
        (dict(hap_len=300, read_lens=[100, 100, 60, 151], n_haps=3, qmax=255), dict(max_indel_error=16)),
        (dict(hap_len=2600, read_lens=[1500, 1200, 150], n_haps=2, qmax=41), dict(max_indel_error=16)),
        (dict(hap_len=700, read_lens=[150, 100, 250], n_haps=3, qmax=41), dict(max_indel_error=64)),
        (dict(hap_len=900, read_lens=[150, 100], n_haps=2, qmax=41), dict(max_indel_error=100)),
        (dict(hap_len=300, read_lens=[100, 150, 150], n_haps=4, qmax=41), dict(max_indel_error=16, use_int_scores=True)),
    ]
    for rk, ck in cases:
        haps, reads = region(**rk)
        cfg = HaplotypeLikelihoodModel.Config(map_positions=False, **ck)
        band = HaplotypeLikelihoodModel(cfg).pad_requirement()
        for flanks in (None, (30, 25)):
            rc, want, wst = coracle.populate(band, haps, reads, None, flanks)
            got, st = engine.populate(cfg, haps, reads, flank_state=flanks, want_status=True)
            ok = wst == 0
            assert np.array_equal((st & 0xFFFF) == 2, (wst & 0xFFFF) == 2), (rk, ck)
            good, worst = _close(got[ok], want[ok])
            assert good, (rk, ck, flanks, worst)
    with pytest.raises(Exception) as ei:
        engine.populate(HaplotypeLikelihoodModel.Config(max_indel_error=300), *region(hap_len=120, read_lens=[40], n_haps=1, qmax=41))
    assert "256" in str(ei.value)


def test_populate_templates_sums_the_reads_of_each_template(engine, coracle):
    """populate(TemplateMap): the value of a template is the sum of its reads' values, in read order."""
    from octopus_b200 import HaplotypeLikelihoodModel, synth
    haps, reads, band = synth.make_batch("C2", n_reads=900, n_haps=10)
    rng = np.random.default_rng(8)
    sizes = []
    while sum(sizes) < reads.n:
        sizes.append(min(int(rng.choice([1, 2, 2, 2, 3])), reads.n - sum(sizes)))
    toff = np.concatenate([[0], np.cumsum(sizes)]).astype(np.int64)
    cfg = HaplotypeLikelihoodModel.Config(max_indel_error=band)
    got = engine.populate_templates(cfg, haps, reads, toff, flank_state=(50, 40))
    rc, per_read, _ = coracle.populate(band, haps, reads, None, (50, 40), map_positions=True)
    want = np.zeros((haps.n, len(sizes)))
    for t in range(len(sizes)):
        for r in range(toff[t], toff[t + 1]):
            want[:, t] = want[:, t] + per_read[:, r]
    ok, worst = _close(got, want)
    assert rc == 0 and ok, worst


def test_multi_sample_array_is_one_batch_with_per_sample_views(engine, coracle):
    """HaplotypeLikelihoodArray::populate(ReadMap) over several samples: one engine call on the concatenated reads; each
    sample's likelihoods_[h][sample] equals the oracle's values for that sample's reads; prime / merge_samples follow
    haplotype_likelihood_array.cpp:200-409."""
    from octopus_b200 import HaplotypeLikelihoodArray, HaplotypeLikelihoodModel, synth, shard
    haps, reads, band = synth.make_batch("C2", n_reads=700, n_haps=9)
    parts = {"NA1": shard.shard_reads(reads, 3, 0)[0], "NA2": shard.shard_reads(reads, 3, 1)[0], "NA3": shard.shard_reads(reads, 3, 2)[0]}
    model = HaplotypeLikelihoodModel(HaplotypeLikelihoodModel.Config(max_indel_error=band))
    before = engine.launch_count(total=True)
    arr = HaplotypeLikelihoodArray(model, engine).populate(parts, haps, flank_state=(40, 40))
    one_call = engine.launch_count(total=True) - before
    rc, want, _ = coracle.populate(band, haps, reads, None, (40, 40), map_positions=True)
    assert rc == 0 and arr.samples() == ["NA1", "NA2", "NA3"]
    lo = 0
    for name, block in parts.items():
        ok, worst = _close(arr.extract_sample(name), want[:, lo:lo + block.n])
        assert ok, (name, worst)
        lo += block.n
    merged = arr.merge_samples()
    assert merged.is_primed() and merged.num_likelihoods() == reads.n and _close(np.stack([merged[h] for h in range(haps.n)]), want)[0]
    engine.populate(model.config, haps, reads, flank_state=(40, 40))
    assert one_call == engine.launch_count()          # the three samples cost exactly one populate call's launches


def test_populate_matches_the_compiled_reference_populate(engine, refhmm):
    """The CUDA engine against the reference's OWN HaplotypeLikelihoodArray::populate (haplotype_likelihood_array.cpp compiled from
    /root/reference in the authoring container, oracle/_ref/libref_hmm.so) — no restatement in between: same haplotypes, reads,
    flank state and configuration in, the same [H][R] ln-likelihoods out (integer penalties identical; the double epilogue to 1e-4
    relative, in practice a few ulp)."""
    from octopus_b200 import HaplotypeLikelihoodModel, synth
    rng = np.random.default_rng(8086)
    for trial in range(8):
        band_req = int(rng.choice([6, 8, 16, 20]))
        band = next(b for b in (8, 16, 32) if band_req <= b)
        if trial < 6:
            haps, reads = random_region(rng, band, n_haps=int(rng.integers(1, 12)), n_reads=int(rng.integers(2, 50)), hap_len=int(rng.choice([200, 300])),
                                        read_len_choices=[40, 76, 100], read_n_rate=0.05, edge_reads=(trial % 2 == 0))
        else:
            haps, reads, band_req = synth.make_batch("C2", n_reads=300, n_haps=12, seed=trial)
        flanks = (int(rng.integers(0, 80)), int(rng.integers(0, 80))) if trial % 2 else None
        trig, cap = {1: (40, 120), 3: (40, 50), 5: (200, 50)}.get(trial, (None, 120))
        cfg = HaplotypeLikelihoodModel.Config(max_indel_error=band_req, mapping_quality_cap=cap, mapping_quality_cap_trigger=trig)
        st, want, _ = refhmm.array_populate(band_req, haps, reads, flanks=flanks, mapq_cap=cap, mapq_cap_trigger=-1 if trig is None else trig)
        if st == 1:
            from octopus_b200.api import ShortHaplotypeError
            with pytest.raises(ShortHaplotypeError):
                engine.populate(cfg, haps, reads, None, flanks)
            continue
        got = engine.populate(cfg, haps, reads, None, flanks)
        ok, worst = _close(got, want)
        assert ok and np.array_equal(got == 0.0, want == 0.0), (trial, worst)


def test_flank_discount_with_n_columns_matchable_below_two(engine, coracle, refhmm):
    """The reference's flank replay charges a mismatch against a truth 'N' exactly 2 although its DP charged min(q', 2)
    (simd_pair_hmm.hpp:388-392 vs :121-142). Haplotypes with several 'N's inside the flanks, reads with qualities 0 / 1 and SNV
    priors 0 / 1: every near-flank candidate must still equal the reference (such candidates take the exact traceback kernel)."""
    from octopus_b200 import HaplotypeLikelihoodModel
    from helpers import n_rich_flank_region
    rng = np.random.default_rng(1234)
    for trial in range(4):
        band = [8, 16, 16, 32][trial]
        haps, reads, flanks = n_rich_flank_region(rng)
        cfg = HaplotypeLikelihoodModel.Config(max_indel_error=band, use_mapping_quality=False)
        rc, want, wst = coracle.populate(band, haps, reads, None, flanks, use_mapping_quality=False, map_positions=True)
        got, st = engine.populate(cfg, haps, reads, None, flanks, want_status=True)
        ok = wst == 0
        assert np.array_equal(st[~ok], wst[~ok]) and np.array_equal(got[ok], want[ok]), (trial, np.abs(got[ok] - want[ok]).max())   # -ln10/10 * integer: exact
        if refhmm is not None and rc == 0:
            st_r, want_r, _ = refhmm.array_populate(band, haps, reads, flanks=flanks, use_mapping_quality=False)
            assert st_r == 0 and np.allclose(got, want_r, rtol=1e-12, atol=0)
