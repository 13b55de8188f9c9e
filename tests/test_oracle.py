"""The oracle is pinned here: against the reference's own known-answer tests (tests/golden/pair_hmm_kats.json,
extracted from test/unit/core/models/pair_hmm_tests.cpp) and against the reference's SIMD kernel compiled into
oracle/_ref (its answers replayed from tests/golden/reference_calls.json.xz)."""
import numpy as np

from helpers import ACGT, random_alignment_case

C_LN10_DIV_10 = 0.230258509299404568401799145468436420760110148862877297603


def test_c_restatement_reproduces_reference_kats(coracle, kats):
    assert len(kats) == 22
    for c in kats:
        s = coracle.align(c["band"], c["truth"], c["read"], c["quals"], c["gap_open"], c["gap_extend"], c["nuc_prior"])
        s2, fp, a1, a2 = coracle.align_tb(c["band"], c["truth"], c["read"], c["quals"], c["gap_open"], c["gap_extend"], c["nuc_prior"])
        assert (s, s2, fp, a1, a2) == (c["score"], c["score"], c["first_pos"], c["align_truth"], c["align_read"]), (c["suite"], c["index"])


def test_reference_build_reproduces_its_own_kats(refkernels, kats):
    for isa, k in refkernels.items():
        for c in kats:
            for bits in (16, 32):
                s = k.align(c["band"], c["truth"], c["read"], c["quals"], c["gap_open"], c["gap_extend"], c["nuc_prior"], bits=bits)
                s2, fp, a1, a2 = k.align_tb(c["band"], c["truth"], c["read"], c["quals"], c["gap_open"], c["gap_extend"], c["nuc_prior"], bits=bits)
                assert (s, s2, fp, a1, a2) == (c["score"], c["score"], c["first_pos"], c["align_truth"], c["align_read"]), (isa, c["suite"], c["index"], bits)


def test_c_restatement_matches_reference_kernel_fuzz(coracle, refkernels):
    rng = np.random.default_rng(20260923)
    isas = list(refkernels)
    for it in range(1500):
        band = int(rng.choice([8, 16, 32, 64]))
        L = int(rng.integers(1, 140))
        c = random_alignment_case(rng, band, L)
        nuc = int(rng.integers(2, 5))
        k = refkernels[isas[it % len(isas)]]
        bits = int(rng.choice([16, 32]))
        q = c["quals"].astype(np.int8)
        t, r, m = c["truth"].tobytes(), c["read"].tobytes(), c["snv_mask"].tobytes()
        snv = dict(snv_mask=m, snv_prior=c["snv_prior"]) if it % 4 else {}
        ge = c["gap_extend"] if it % 3 else int(c["gap_extend"][0])
        assert k.align(band, t, r, q, c["gap_open"], ge, nuc, bits=bits, **snv) == coracle.align(band, t, r, q, c["gap_open"], ge, nuc, **snv)
        ref_tb = k.align_tb(band, t, r, q, c["gap_open"], ge, nuc, bits=bits, **snv)
        assert ref_tb == coracle.align_tb(band, t, r, q, c["gap_open"], ge, nuc, **snv)
        if snv:
            W = len(t)
            lhs, rhs = int(rng.integers(0, W // 2 + 1)), int(rng.integers(0, W // 2 + 1))
            a = k.flank_score(band, W, lhs, rhs, r, q, m, c["snv_prior"], c["gap_open"], ge, nuc, ref_tb[1], ref_tb[2], ref_tb[3], bits=bits)
            b = coracle.flank_score(W, lhs, rhs, r, q, m, c["snv_prior"], c["gap_open"], ge, nuc, ref_tb[1], ref_tb[2], ref_tb[3])
            assert a == b


def test_reference_int16_equals_int32_when_not_overflowing(refkernels):
    """Parity domain: the engine computes exact scores; the reference's default int16 lanes agree with its int32 lanes
    whenever the true score fits (adversarial: cheap gaps / expensive mismatches stress the un-initialised band lanes)."""
    k = next(iter(refkernels.values()))
    rng = np.random.default_rng(7)
    for it in range(1500):
        band = int(rng.choice([8, 16, 32]))
        L = int(rng.integers(1, 80))
        c = random_alignment_case(rng, band, L)
        q = rng.integers(60, 121, L).astype(np.int8)
        go = rng.integers(1, 4, len(c["truth"])).astype(np.int8) if it % 2 else rng.integers(40, 46, len(c["truth"])).astype(np.int8)
        ge = np.ones(len(c["truth"]), dtype=np.int8)
        nuc = int(rng.integers(0, 3))
        t, r, m = c["truth"].tobytes(), c["read"].tobytes(), c["snv_mask"].tobytes()
        assert k.align(band, t, r, q, go, ge, nuc, m, c["snv_prior"], bits=16) == k.align(band, t, r, q, go, ge, nuc, m, c["snv_prior"], bits=32)


def test_naive_evaluate_shortcuts(coracle):
    hap = "ACGTTGCAAGCTTAGGCTAACGTTAGCATCGATCGGATCTAGCTAGGATCGAT" * 3
    L, off = 30, 20
    go = np.full(len(hap), 40, dtype=np.int8)
    ge = np.full(len(hap), 3, dtype=np.int8)
    mask = ("N" * len(hap)).encode()
    prior = np.full(len(hap), 100, dtype=np.int8)
    read = hap[off:off + L]
    q = np.full(L, 30, dtype=np.uint8)
    # exact match → 0 (pair_hmm.hpp:289-291)
    assert coracle.try_naive_evaluate(hap, read, q, off, go, ge, mask, prior) == (True, 0)
    # one mismatch, quality <= gap open → the quality (:302-303)
    r1 = list(read); r1[10] = "A" if r1[10] != "A" else "C"; r1 = "".join(r1)
    assert coracle.try_naive_evaluate(hap, r1, q, off, go, ge, mask, prior) == (True, 30)
    # ... capped by the SNV prior when the mask names the read base (:250-263)
    mask2 = bytearray(mask); mask2[off + 10] = ord(r1[10]); prior2 = prior.copy(); prior2[off + 10] = 7
    assert coracle.try_naive_evaluate(hap, r1, q, off, go, ge, bytes(mask2), prior2) == (True, 7)
    # in a flank → 0 (:298)
    assert coracle.try_naive_evaluate(hap, r1, q, off, go, ge, mask, prior, flanks=(off + 11, 0)) == (True, 0)
    # two mismatches → no shortcut
    r2 = list(r1); r2[20] = "A" if r2[20] != "A" else "C"; r2 = "".join(r2)
    assert coracle.try_naive_evaluate(hap, r2, q, off, go, ge, mask, prior)[0] is False
    # evaluate() == -ln10/10 * phred on the shortcut, and the DP otherwise
    assert coracle.evaluate(16, hap, r1, q, off, go, ge, 2, mask, prior) == -C_LN10_DIV_10 * 30
    v, used, raw = coracle.evaluate(16, hap, r2, q, off, go, ge, 2, mask, prior, details=True)
    assert used == 1 and raw == 60 and v == -C_LN10_DIV_10 * 60


def _kmer_map_python(query, target, max_positions=10):
    """Independent restatement of utils/kmer_mapper.hpp:43-159 in pure Python (small inputs only)."""
    K = 6
    code = {"A": 0, "C": 1, "G": 2, "T": 3}
    def h(s):
        return sum(code.get(ch, 0) * 4 ** i for i, ch in enumerate(s))
    if len(query) < K or len(target) < K:
        return []
    table = {}
    for i in range(len(target) - K + 1):
        table.setdefault(h(target[i:i + K]), []).append(i)
    counts = [0] * (len(target) - K + 1)
    max_hit, first_max, num_max = 0, 0, 0
    for qi in range(len(query) - K + 1):
        for ti in table.get(h(query[qi:qi + K]), []):
            if ti >= qi:
                mb = ti - qi
                counts[mb] += 1
                if counts[mb] > max_hit:
                    max_hit, first_max, num_max = counts[mb], mb, 1
                elif counts[mb] == max_hit:
                    num_max += 1
                    first_max = min(first_max, mb)
    out = []
    if max_hit > 0:
        out.append(first_max); first_max += 1; num_max -= 1; max_positions -= 1
        while max_positions > 0 and num_max > 0:
            if counts[first_max] == max_hit:
                out.append(first_max); num_max -= 1; max_positions -= 1
            first_max += 1
    return out


def test_kmer_mapper(coracle):
    rng = np.random.default_rng(3)
    for _ in range(200):
        t = "".join(rng.choice(list("ACGT"), int(rng.integers(20, 200))))
        p = int(rng.integers(0, max(1, len(t) - 10)))
        q = t[p:p + int(rng.integers(6, 60))]
        if rng.random() < 0.5 and len(q) > 8:
            q = q[:4] + "ACGT"[int(rng.integers(0, 4))] + q[5:]
        if rng.random() < 0.3:
            t = t[:len(t) // 2] * 2          # repeats → several equally good positions
        assert coracle.kmer_map(q, t, 10) == _kmer_map_python(q, t, 10)


def test_model_evaluate_mapping_quality_floor(coracle):
    """ln p = log_sum_exp(ln(1 - 10^(-mq/10)) + lnP, -ln10/10 * mq) and the > -1e-15 clamp (haplotype_likelihood_model.cpp:285-303)."""
    hap = "ACGTTGCAAGCTTAGGCTAACGTTAGCATCGATCGGATCTAGCTAGGATCGATACGATCGATCGTAGCTAGCTAGTCGAT"
    n = len(hap)
    args = dict(gap_open=np.full(n, 40, np.int8), gap_extend=np.full(n, 3, np.int8), snv_mask=("N" * n).encode(), snv_prior=np.full(n, 100, np.int8))
    read, q = hap[20:50], np.full(30, 30, np.uint8)
    st, v, _ = coracle.model_evaluate(16, hap, read, q, positions=[], original_pos=20, mapping_quality=60, **args)
    assert st == 0 and v == 0.0            # exact match, clamp to 0
    st, v, _ = coracle.model_evaluate(16, hap, read, q, positions=[], original_pos=20, mapping_quality=0, **args)
    assert st == 0 and v == 0.0            # mq 0: ln_mapped = -inf, lse(-inf, 0) = 0
    st, v, ext = coracle.model_evaluate(16, hap[:40], read, q, positions=[], original_pos=5, mapping_quality=60,
                                        gap_open=args["gap_open"][:40], gap_extend=args["gap_extend"][:40], snv_mask=args["snv_mask"][:40], snv_prior=args["snv_prior"][:40])
    assert st == 1 and ext > 0             # ShortHaplotypeError


# ---------------------------------------------------------------------------------------------------------------------
# The layer above the kernel, pinned to the reference's own code (pair_hmm.hpp, simd_pair_hmm_wrapper.hpp compiled from
# /root/reference behind oracle/ref_hmm_driver.cpp). The reference has no unit tests for this layer.
# ---------------------------------------------------------------------------------------------------------------------
def _hmm_case(rng, hap_len, L, exact_rate=0.25):
    hap = ACGT[rng.integers(0, 4, hap_len)].copy()
    if rng.random() < 0.2:
        hap[rng.integers(0, hap_len)] = ord("N")
    start = int(rng.integers(0, hap_len - L + 1))
    read = np.where(hap[start:start + L] == ord("N"), ord("A"), hap[start:start + L]).astype(np.uint8)
    mode = rng.random()
    if mode > exact_rate:
        n_sub = 1 if mode < exact_rate + 0.3 else int(rng.integers(1, 5))
        for _ in range(n_sub):
            read[rng.integers(0, L)] = ACGT[rng.integers(0, 4)]
        if mode > 0.8 and L > 12:                                   # an indel
            p = int(rng.integers(3, L - 6))
            read = np.concatenate([read[:p], read[p + 2:], ACGT[rng.integers(0, 4, 2)]]) if rng.random() < 0.5 \
                else np.concatenate([read[:p], ACGT[rng.integers(0, 4, 2)], read[p:-2]])
    return dict(hap=hap, read=read, start=start, quals=rng.integers(2, 42, L).astype(np.uint8),
                go=rng.integers(3, 46, hap_len).astype(np.int8), ge=rng.integers(1, 11, hap_len).astype(np.int8),
                mask=np.frombuffer(b"ACGTN", dtype=np.uint8)[rng.integers(0, 5, hap_len)].copy(),
                prior=rng.integers(1, 126, hap_len).astype(np.int8))


def test_band_choice_matches_reference_wrapper(refhmm):
    """simd_pair_hmm_wrapper.hpp:209-241: smallest of 8, 16, ..., 256 that covers the request; beyond 256 it throws."""
    for req in list(range(1, 70)) + [127, 128, 129, 255, 256, 257, 1000]:
        want = next((b for b in (8, 16, 32, 64, 128, 256) if req <= b), -1)
        assert refhmm.band(req) == want and refhmm.band(req, int32=True) == want


def test_c_restatement_evaluate_matches_reference_hmm_evaluate(coracle, refhmm):
    """oracle_evaluate (naive shortcuts, window placement, flank-aware discount, lowest() on out-of-range) against the
    reference's own hmm::evaluate with the MutationModel, over seeded cases that hit every branch."""
    rng = np.random.default_rng(20240923)
    kinds = {0: 0, 1: 0, 2: 0}
    n_lowest = 0
    for it in range(1500):
        band_req = int(rng.choice([3, 8, 12, 16, 30]))
        band = next(b for b in (8, 16, 32) if band_req <= b)
        L = int(rng.integers(8, 60))
        hap_len = int(rng.integers(L + 2 * band + 2, L + 2 * band + 90))
        c = _hmm_case(rng, hap_len, L)
        # mostly the true position (+- a few bases), sometimes anywhere — including offsets whose window leaves the haplotype
        off = int(np.clip(c["start"] + rng.integers(-3, 4), 0, hap_len - 1)) if rng.random() < 0.8 else int(rng.integers(0, hap_len))
        flanks = (0, 0) if rng.random() < 0.4 else (int(rng.integers(0, hap_len // 2)), int(rng.integers(0, hap_len // 2)))
        want = refhmm.evaluate(band_req, c["hap"], c["read"], c["quals"], off, c["go"], c["ge"], c["mask"], c["prior"], flanks)
        got, used, raw = coracle.evaluate(band, c["hap"], c["read"], c["quals"], off, c["go"], c["ge"], 2, c["mask"], c["prior"],
                                          flanks=flanks, details=True)
        assert got == want or abs(got - want) <= 1e-12 * abs(want), (it, band, L, hap_len, off, flanks, got, want, used, raw)
        kinds[used] += 1
        n_lowest += want < -1e300
    assert min(kinds.values()) > 50 and n_lowest > 5, (kinds, n_lowest)      # shortcut, score-only DP, traceback + flank DP, lowest()


def test_c_restatement_align_matches_reference_hmm_align(coracle, refhmm):
    """oracle_model_align at a single in-range mapping position == the reference's hmm::align there: offset, likelihood, CIGAR."""
    rng = np.random.default_rng(77)
    n_indel = 0
    for it in range(600):
        band = int(rng.choice([8, 16]))
        L = int(rng.integers(10, 50))
        hap_len = int(rng.integers(L + 2 * band + 2, L + 2 * band + 60))
        c = _hmm_case(rng, hap_len, L, exact_rate=0.15)
        pos = int(np.clip(c["start"] + rng.integers(-2, 3), band, hap_len - L - band))
        flanks = (0, 0) if rng.random() < 0.5 else (int(rng.integers(0, hap_len // 3)), int(rng.integers(0, hap_len // 3)))
        w_off, w_lk, w_cigar = refhmm.align(band, c["hap"], c["read"], c["quals"], pos, c["go"], c["ge"], c["mask"], c["prior"], flanks)
        st, g_off, g_lk, g_cigar, _ = coracle.model_align(band, c["hap"], c["read"], c["quals"], c["go"], c["ge"], c["mask"], c["prior"],
                                                          [pos], pos, flanks=flanks, use_mapping_quality=False)
        assert st == 0 and (g_off, g_cigar) == (w_off, w_cigar) and abs(g_lk - w_lk) <= 1e-12 * max(abs(w_lk), 1e-300), \
            (it, band, L, pos, flanks, (g_off, g_lk, g_cigar), (w_off, w_lk, w_cigar))
        n_indel += ("I" in w_cigar) or ("D" in w_cigar)
    assert n_indel > 20


def test_c_restatement_kmer_mapper_matches_reference_mapper(coracle, refhmm):
    """oracle_kmer_map against utils/kmer_mapper.hpp itself (compiled from /root/reference), called the way
    HaplotypeLikelihoodArray::populate calls it: repeats (many tied diagonals), non-ACGT bases, reads longer than the
    haplotype, sequences shorter than a k-mer, more than ten maximal diagonals."""
    rng = np.random.default_rng(4242)
    n_multi = n_trunc = 0
    for it in range(1500):
        kind = rng.random()
        tl = int(rng.integers(3, 400))
        if kind < 0.3:                       # low-complexity target: tandem repeat of a short unit
            unit = ACGT[rng.integers(0, 4, int(rng.integers(1, 7)))]
            target = np.tile(unit, tl // len(unit) + 1)[:tl].copy()
        else:
            target = ACGT[rng.integers(0, 4, tl)].copy()
        if rng.random() < 0.2 and tl > 0:
            target[rng.integers(0, tl)] = ord("N")
        ql = int(rng.integers(3, 180))
        if kind < 0.85 and tl > ql:
            s = int(rng.integers(0, tl - ql + 1))
            query = target[s:s + ql].copy()
            for _ in range(int(rng.integers(0, 4))):
                query[rng.integers(0, ql)] = ACGT[rng.integers(0, 4)]
        else:
            query = ACGT[rng.integers(0, 4, ql)].copy()
        want = refhmm.kmer_map(query, target, 10)
        got = coracle.kmer_map(query.tobytes().decode(), target.tobytes().decode(), 10)
        assert list(got) == want, (it, query.tobytes(), target.tobytes(), got, want)
        n_multi += len(want) > 1
        n_trunc += len(want) == 10
    assert n_multi > 100 and n_trunc > 20


def _model_case(rng):
    band_req = int(rng.choice([3, 8, 12, 16, 30]))
    band = next(b for b in (8, 16, 32) if band_req <= b)
    L = int(rng.integers(8, 60))
    # mostly long enough, sometimes too short for read + pads (ShortHaplotypeError / shifted fallback territory)
    hap_len = int(rng.integers(L + 2 * band + 1, L + 2 * band + 80)) if rng.random() < 0.8 else int(rng.integers(max(L // 2, 8), L + 2 * band + 1))
    c = _hmm_case(rng, hap_len, min(L, hap_len), exact_rate=0.3)
    c["band_req"], c["band"] = band_req, band
    c["mask_r"] = np.frombuffer(b"ACGTN", dtype=np.uint8)[rng.integers(0, 5, hap_len)].copy()
    c["prior_r"] = rng.integers(1, 126, hap_len).astype(np.int8)
    c["reverse"] = bool(rng.random() < 0.5)
    c["hap_begin"] = int(rng.integers(0, 1000))
    # the read's own mapped position: near its true origin, or anywhere over the haplotype (edges → fallback shift)
    orig = int(np.clip(c["start"] + rng.integers(-2, 3), 0, hap_len)) if rng.random() < 0.7 else int(rng.integers(0, hap_len + 1))
    c["orig"] = orig
    c["mapq"] = int(rng.choice([0, 3, 20, 40, 60, 255]))
    c["trigger"] = int(rng.choice([-1, -1, 30, 200]))
    c["cap"] = int(rng.choice([120, 50]))
    c["use_mq"] = bool(rng.random() < 0.8)
    c["flanks"] = None if rng.random() < 0.5 else (int(rng.integers(0, hap_len // 2 + 1)), int(rng.integers(0, hap_len // 2 + 1)))
    c["positions"] = None if rng.random() < 0.5 else [int(x) for x in rng.integers(0, hap_len + 5, int(rng.integers(0, 5)))]
    return c


def test_c_restatement_model_evaluate_matches_reference_model(coracle, refhmm):
    """oracle_model_evaluate against the reference's own HaplotypeLikelihoodModel::reset + evaluate
    (haplotype_likelihood_model.cpp compiled from /root/reference): in-range rule, max over mapping positions U original position,
    shifted fallback, ShortHaplotypeError with its required extension, strand-specific SNV arrays, mapping-quality mixing with cap
    trigger, clamp; candidate positions either explicit or mapped by the reference's k-mer mapper as populate() does."""
    rng = np.random.default_rng(31337)
    n_short = n_fallback = n_mapped = 0
    for it in range(2500):
        c = _model_case(rng)
        mask, prior = (c["mask_r"], c["prior_r"]) if c["reverse"] else (c["mask"], c["prior"])
        w = refhmm.model_evaluate(c["band_req"], c["hap"], c["read"], c["quals"], c["go"], c["ge"], c["mask"], c["prior"], c["mask_r"], c["prior_r"],
                                  c["positions"], hap_begin=c["hap_begin"], read_begin=c["hap_begin"] + c["orig"], mapping_quality=c["mapq"],
                                  reverse=c["reverse"], flanks=c["flanks"], use_mapping_quality=c["use_mq"], mapq_cap=c["cap"],
                                  mapq_cap_trigger=c["trigger"])
        positions = c["positions"] if c["positions"] is not None else coracle.kmer_map(c["hap"][:0].tobytes().decode() + c["read"].tobytes().decode(), c["hap"].tobytes().decode(), 10)
        g = coracle.model_evaluate(c["band"], c["hap"], c["read"], c["quals"], c["go"], c["ge"], mask, prior, positions, c["orig"],
                                   mapping_quality=c["mapq"], flanks=c["flanks"], use_mapping_quality=c["use_mq"], mapq_cap=c["cap"],
                                   mapq_cap_trigger=c["trigger"])
        assert g[0] == w[0], (it, c, g, w)
        if w[0] == 1:
            assert g[2] == w[2], (it, c, g, w)
            n_short += 1
        else:
            assert g[1] == w[1] or abs(g[1] - w[1]) <= 1e-12 * abs(w[1]), (it, c, g, w)
        n_mapped += c["positions"] is None
        n_fallback += not (c["band"] <= c["orig"] and c["orig"] + len(c["read"]) + c["band"] <= len(c["hap"]))
    assert n_short > 50 and n_fallback > 300 and n_mapped > 800, (n_short, n_fallback, n_mapped)


def test_c_restatement_model_align_matches_reference_model(coracle, refhmm):
    """oracle_model_align against HaplotypeLikelihoodModel::reset + align (compute_optimal_alignment, :335-431): which candidate
    wins (> for listed positions, >= for the original position), its offset, CIGAR and mixed likelihood, ShortHaplotypeError."""
    rng = np.random.default_rng(99)
    n_short = 0
    for it in range(1200):
        c = _model_case(rng)
        mask, prior = (c["mask_r"], c["prior_r"]) if c["reverse"] else (c["mask"], c["prior"])
        w = refhmm.model_align(c["band_req"], c["hap"], c["read"], c["quals"], c["go"], c["ge"], c["mask"], c["prior"], c["mask_r"], c["prior_r"],
                               c["positions"], hap_begin=c["hap_begin"], read_begin=c["hap_begin"] + c["orig"], mapping_quality=c["mapq"],
                               reverse=c["reverse"], flanks=c["flanks"], use_mapping_quality=c["use_mq"], mapq_cap=c["cap"],
                               mapq_cap_trigger=c["trigger"])
        positions = c["positions"] if c["positions"] is not None else coracle.kmer_map(c["read"].tobytes().decode(), c["hap"].tobytes().decode(), 10)
        g = coracle.model_align(c["band"], c["hap"], c["read"], c["quals"], c["go"], c["ge"], mask, prior, positions, c["orig"],
                                mapping_quality=c["mapq"], flanks=c["flanks"], use_mapping_quality=c["use_mq"], mapq_cap=c["cap"],
                                mapq_cap_trigger=c["trigger"])
        assert g[0] == w[0], (it, c, g, w)
        if w[0] == 1:
            assert g[4] == w[4], (it, c, g, w)
            n_short += 1
        else:
            assert (g[1], g[3]) == (w[1], w[3]) and (g[2] == w[2] or abs(g[2] - w[2]) <= 1e-12 * abs(w[2])), (it, c, g, w)
    assert n_short > 20


def test_model_layer_agrees_on_hostile_inputs_within_the_quality_domain(coracle, refhmm):
    """N / IUPAC / lower-case letters in reads and haplotypes and qualities up to 127 (the int8 range the reference kernel reads):
    the restatement still equals the compiled HaplotypeLikelihoodModel. (Above 127 the reference's own result depends on SIMD
    wrap-around of negative penalties — out of the parity domain, DESIGN.md §2.)"""
    rng = np.random.default_rng(5)
    alphabet = np.frombuffer(b"NRacgtn", dtype=np.uint8)
    for it in range(900):
        c = _model_case(rng)
        L = len(c["read"])
        if it % 3 == 0:
            for _ in range(int(rng.integers(1, 4))):
                c["read"][rng.integers(0, L)] = alphabet[rng.integers(0, len(alphabet))]
        elif it % 3 == 1:
            for _ in range(int(rng.integers(1, 4))):
                c["hap"][rng.integers(0, len(c["hap"]))] = alphabet[rng.integers(0, len(alphabet))]
        else:
            c["quals"] = rng.integers(60, 128, L).astype(np.uint8)
        mask, prior = (c["mask_r"], c["prior_r"]) if c["reverse"] else (c["mask"], c["prior"])
        w = refhmm.model_evaluate(c["band_req"], c["hap"], c["read"], c["quals"], c["go"], c["ge"], c["mask"], c["prior"], c["mask_r"], c["prior_r"],
                                  c["positions"], hap_begin=c["hap_begin"], read_begin=c["hap_begin"] + c["orig"], mapping_quality=c["mapq"],
                                  reverse=c["reverse"], flanks=c["flanks"], use_mapping_quality=c["use_mq"], mapq_cap=c["cap"],
                                  mapq_cap_trigger=c["trigger"])
        positions = c["positions"] if c["positions"] is not None else coracle.kmer_map(c["read"].tobytes().decode("latin1"), c["hap"].tobytes().decode("latin1"), 10)
        g = coracle.model_evaluate(c["band"], c["hap"], c["read"], c["quals"], c["go"], c["ge"], mask, prior, positions, c["orig"],
                                   mapping_quality=c["mapq"], flanks=c["flanks"], use_mapping_quality=c["use_mq"], mapq_cap=c["cap"],
                                   mapq_cap_trigger=c["trigger"])
        assert g[0] == w[0] and ((w[0] == 1 and g[2] == w[2]) or (w[0] == 0 and (g[1] == w[1] or abs(g[1] - w[1]) <= 1e-12 * abs(w[1])))), (it, g, w)


def test_c_restatement_populate_matches_reference_array_populate(coracle, refhmm):
    """oracle_populate — the checker every GPU populate test compares against — equals the reference's own
    HaplotypeLikelihoodArray::populate (haplotype_likelihood_array.cpp compiled from /root/reference: H x S x R loop, inline k-mer
    mapping, model reset / evaluate per haplotype), for several samples (= column ranges of one concatenated batch), with and
    without a flank state, and for the TemplateMap overload (sum over a template's reads)."""
    from helpers import random_region
    rng = np.random.default_rng(606)
    n_short = 0
    for trial in range(14):
        band_req = int(rng.choice([6, 8, 16, 20]))
        band = next(b for b in (8, 16, 32) if band_req <= b)
        haps, reads = random_region(rng, band, n_haps=int(rng.integers(1, 9)), n_reads=int(rng.integers(2, 40)), hap_len=int(rng.choice([150, 260])),
                                    read_len_choices=[30, 60, 100], read_n_rate=0.05, edge_reads=(trial % 2 == 0))
        flanks = (int(rng.integers(0, 70)), int(rng.integers(0, 70))) if trial % 2 else None
        trig, cap = {1: (40, 120), 3: (40, 50), 5: (200, 50)}.get(trial % 6, (-1, 120))
        use_mq = trial % 5 != 4
        cuts = np.sort(rng.integers(0, reads.n + 1, int(rng.integers(0, 4))))
        sample_off = np.concatenate([[0], cuts, [reads.n]]).astype(np.int64)             # empty samples allowed
        rc, want_o, wst = coracle.populate(band, haps, reads, None, flanks, use_mapping_quality=use_mq, mapq_cap=cap, mapq_cap_trigger=trig,
                                           map_positions=True)
        st, got, ext = refhmm.array_populate(band_req, haps, reads, sample_off=sample_off, flanks=flanks, use_mapping_quality=use_mq,
                                             mapq_cap=cap, mapq_cap_trigger=trig)
        short = ((wst & 0xFFFF) == 2).any()
        assert st == (1 if short else 0), (trial, st, rc)
        if short:
            n_short += 1
            continue
        assert np.allclose(got, want_o, rtol=1e-12, atol=0) and np.array_equal(got == 0.0, want_o == 0.0), (trial, np.abs(got - want_o).max())
        # TemplateMap: consecutive reads grouped into templates, two "samples"
        sizes = []
        while sum(sizes) < reads.n:
            sizes.append(min(int(rng.choice([1, 2, 2, 3])), reads.n - sum(sizes)))
        toff = np.concatenate([[0], np.cumsum(sizes)]).astype(np.int64)
        t_cut = int(rng.integers(0, len(sizes) + 1))
        st, got_t, _ = refhmm.array_populate(band_req, haps, reads, sample_off=[0, t_cut, len(sizes)], template_off=toff, flanks=flanks,
                                             use_mapping_quality=use_mq, mapq_cap=cap, mapq_cap_trigger=trig)
        want_t = np.stack([want_o[:, a:b].sum(axis=1) if b - a > 1 else want_o[:, a] for a, b in zip(toff[:-1], toff[1:])], axis=1)
        assert st == 0 and np.allclose(got_t, want_t, rtol=1e-12, atol=1e-300), (trial, np.abs(got_t - want_t).max())
    assert n_short < 10


def test_populate_agrees_with_reference_where_flank_replay_and_dp_differ(coracle, refhmm):
    """CPU twin of the GPU test of the same corner (tests/test_gpu_parity.py): 'N's inside the flanks with qualities / SNV priors
    of 0 and 1, where the reference's flank replay re-adds 2 for a truth-'N' mismatch its DP charged less for. The restatement
    must follow the reference's replay — and the inputs must actually hit the corner (the discounted value differs from what a
    'what the DP charged' discount would give)."""
    from helpers import n_rich_flank_region
    rng = np.random.default_rng(1234)
    for trial in range(4):
        band = [8, 16, 16, 32][trial]
        haps, reads, flanks = n_rich_flank_region(rng)
        rc, want, wst = coracle.populate(band, haps, reads, None, flanks, use_mapping_quality=False, map_positions=True)
        st_r, want_r, _ = refhmm.array_populate(band, haps, reads, flanks=flanks, use_mapping_quality=False)
        assert rc == 0 and st_r == 0 and np.allclose(want, want_r, rtol=1e-12, atol=0), trial
