"""HaplotypeLikelihoodModel::reset (SURVEY.md a11 / N2): the engine's own error models (octopus_b200/csrc/phmm_error_model.cpp, host C++
inside libphmm_b200.so) against the UNMODIFIED reference models + lib/tandem (oracle/_ref/libref_errmodel.so, its answers replayed from
tests/golden/reference_calls.json.xz), array for array — and against the committed golden fixture of error_model_golden.json."""
import json
import os

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLDEN = os.path.join(ROOT, "tests", "golden", "error_model_golden.json")
ACGT = np.frombuffer(b"ACGT", dtype=np.uint8)
LABELS = ["PCR-free.HiSeq-2000", "PCR-free.HiSeq-2500", "PCR-free.HiSeq-4000", "PCR-free.X10", "PCR-free.NovaSeq", "PCR-free.BGISEQ-500",
          "PCR-free.PacBio", "PCR-free.PacBioCCS", "PCR.HiSeq-2000", "PCR.HiSeq-2500", "PCR.HiSeq-4000", "PCR.X10", "PCR.NovaSeq",
          "PCR.BGISEQ-500", "PCR.PacBio", "PCR.PacBioCCS", "10X.HiSeq-2000", "10X.HiSeq-2500", "10X.HiSeq-4000", "10X.X10", "10X.NovaSeq",
          "10X.BGISEQ-500", "MDA.HiSeq-2000", "MDA.HiSeq-2500", "MDA.HiSeq-4000", "MDA.X10", "MDA.NovaSeq", "MDA.BGISEQ-500"]
FIELDS = ("snv_mask_fwd", "snv_prior_fwd", "snv_mask_rev", "snv_prior_rev", "gap_open", "gap_extend")


def repeat_rich_sequence(rng, max_len=400):
    """Random sequence over a random-size alphabet with a few injected tandem repeats (period 1..6) and the odd 'N'."""
    n = int(rng.integers(1, max_len))
    s = ACGT[rng.integers(0, int(rng.integers(1, 5)), n)].copy()
    if rng.random() < 0.1:
        s[rng.integers(0, n)] = ord("N")
    for _ in range(int(rng.integers(0, 4))):
        p, k, at = int(rng.integers(1, 7)), int(rng.integers(2, 30)), int(rng.integers(0, len(s)))
        s = np.concatenate([s[:at], np.tile(ACGT[rng.integers(0, 4, p)], k), s[at:]])
    return s[:max_len + 200]


@pytest.fixture
def ref(request):
    """The original error models + lib/tandem (RefErrorModel), replayed from tests/golden (reference_calls.py)."""
    from reference_calls import reference
    return reference(request, "errmodel")


def test_tandem_repeat_finder_equals_lib_tandem(ref):
    from octopus_b200 import ErrorModel
    m = ErrorModel()
    rng = np.random.default_rng(20260923)
    for _ in range(1500):
        s = repeat_rich_sequence(rng)
        for lo, hi in ((1, 5), (1, 3), (1, 2), (2, 3), (1, 1), (2, 2), (3, 3), (1, 4), (2, 5), (1, 8)):
            assert ref.tandem_repeats(s, lo, hi) == m.tandem_repeats(bytes(s), lo, hi), (bytes(s), lo, hi)
    # edge cases: empty / single base / string shorter than the period / all one letter / min_period 0
    for s in (b"", b"A", b"AC", b"AAAAAAAAAA", b"ACACACACAC", b"ACGACGACGACG", b"NNNNNN"):
        for lo, hi in ((1, 5), (1, 3), (0, 5), (3, 3), (4, 9)):
            assert ref.tandem_repeats(s, lo, hi) == m.tandem_repeats(s, lo, hi), (s, lo, hi)


def test_every_builtin_model_equals_the_reference(ref):
    from octopus_b200 import ErrorModel
    rng = np.random.default_rng(7)
    for label in LABELS + ["pcrf.hiseq-2500", "PCR", "pcr-free", ".X10", "MDA."]:
        m = ErrorModel(label)
        seqs = [repeat_rich_sequence(rng) for _ in range(60)]
        subs = [(rng.random(len(s)) < 0.05).astype(np.uint8) for s in seqs]
        use_sub = rng.random() < 0.5
        block = m.reset(seqs, is_substitution=subs if use_sub else None, n_threads=3)
        for h, s in enumerate(seqs):
            rc, want = ref.reset(s, label, subs[h] if use_sub else None)
            assert rc >= 0, label
            got = block.hap(h)
            assert want == {f: got[f] for f in FIELDS}, (label, bytes(s))
    for bad in ("PCR-free.HiSeq-9000", "nonsense", "10X.PacBio"):
        from octopus_b200 import PhmmError
        with pytest.raises(PhmmError):
            ErrorModel(bad)
        assert ref.reset(b"ACGT", bad)[0] < 0


def test_short_read_models_never_make_an_extension_dearer_than_the_opening():
    """gap_open[x] >= gap_extend[x] at every position of every short-read model's output (HiSeq / X10 / NovaSeq / BGISEQ, all
    library preparations): the precondition of the DP kernels' shorter deletion update (phmm_device.cuh dp_pair, OGE). The PacBio
    models break it inside long homopolymers, as a custom model may: such arrays raise kFlagOpenBelowExtend on the device and the
    call runs the general update. This test records which built-in models are on which side."""
    from octopus_b200 import ErrorModel
    rng = np.random.default_rng(99)
    seqs = [repeat_rich_sequence(rng, 600) for _ in range(150)]
    for period in (1, 2, 3, 4, 5, 6):                       # long pure repeats: the lowest opening penalties of every table
        seqs.append(np.tile(ACGT[rng.integers(0, 4, period)], 400 // period))
    violating = set()
    for label in LABELS:
        block = ErrorModel(label).reset(seqs, n_threads=3)
        if any((block.hap(h)["gap_open"] < block.hap(h)["gap_extend"]).any() for h in range(len(seqs))):
            violating.add(label)
    assert violating and all("PacBio" in label for label in violating), violating


def test_custom_model_text_equals_the_reference(ref):
    from octopus_b200 import ErrorModel, PhmmError
    rng = np.random.default_rng(11)
    motifs = ["A", "C", "G", "T", "AC", "AG", "CG", "GC", "AT", "N", "NN", "NNN", "AAC", "ACG", "NNNN", "ACGT"]
    for _ in range(60):
        rng.shuffle(motifs)
        lines = ["# a custom model"]
        for mo in motifs[:int(rng.integers(1, len(motifs)))]:
            lines.append(mo + ":" + ",".join(str(x) for x in sorted(rng.integers(1, 60, int(rng.integers(1, 40))).tolist(), reverse=True)))
        if rng.random() < 0.6:
            for mo in motifs[:int(rng.integers(1, 6))]:
                lines.append(mo + "+:" + ",".join(str(x) for x in rng.integers(1, 12, int(rng.integers(1, 20))).tolist()))
        rng.shuffle(lines)
        text = "\n".join(lines) + ("\n" if rng.random() < 0.7 else "")
        m = ErrorModel(custom_model_text=text)
        for _ in range(20):
            s = repeat_rich_sequence(rng, 250)
            rc, want = ref.reset(s, custom_model_text=text)
            assert rc == 1
            got = m.reset([s]).hap(0)
            assert want == {f: got[f] for f in FIELDS}, (text, bytes(s))
    for bad in ("A+:3,4\n", "A:\n", ":3\n", "A:3,x\n", "AC 3,4\n"):
        with pytest.raises(PhmmError):
            ErrorModel(custom_model_text=bad)
        assert ref.reset(b"ACGT", custom_model_text=bad)[0] < 0, bad


def test_golden_fixture():
    """Committed vectors generated from the compiled reference (tests/golden/make_error_model_golden.py): this is what pins the
    models where /root/reference is absent (the GPU box)."""
    from octopus_b200 import ErrorModel
    with open(GOLDEN) as f:
        cases = json.load(f)["cases"]
    assert len(cases) >= 100
    models = {}
    for c in cases:
        key = (c["label"], c.get("custom"))
        if key not in models:
            models[key] = ErrorModel(c["label"], custom_model_text=c.get("custom"))
        sub = None if c["substitutions"] is None else [np.asarray(c["substitutions"], dtype=np.uint8)]
        got = models[key].reset([c["sequence"]], is_substitution=sub).hap(0)
        for f in FIELDS:
            want = np.frombuffer(c[f].encode(), dtype=np.uint8) if "mask" in f else np.asarray(c[f], dtype=np.int8).view(np.uint8)
            assert np.array_equal(got[f].view(np.uint8), want), (c["label"], f, c["sequence"])
        assert np.array_equal(models[key].tandem_repeats(c["sequence"], 1, 5), np.asarray(c["repeats_1_5"], dtype=np.uint32).reshape(-1, 3))
