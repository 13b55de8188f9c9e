"""phmm_populate_regions_ex: many regions in one call with paired-read templates (populate(TemplateMap), Octopus's default read
linkage) and explicit candidate positions, through the C ABI, the Python API and the C++ adapter's RegionBatch."""
import ctypes as C
import os
import re
import subprocess
import sys

import numpy as np
import pytest

from helpers import random_region

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REGIONS_SRC = os.path.join(ROOT, "tests", "cpp", "test_regions.cpp")
REGIONS_EXE = os.path.join(ROOT, "tests", "cpp", "test_regions")


# ---------------------------------------------------------------------------------------------------------------------
# helpers
# ---------------------------------------------------------------------------------------------------------------------
def _template_sizes(rng, n_reads):
    """Templates of 1-3 consecutive reads (pairs mostly, singletons and triples included): the region-local template_off."""
    sizes = []
    while sum(sizes) < n_reads:
        sizes.append(min(int(rng.choice([1, 2, 2, 2, 3])), n_reads - sum(sizes)))
    return np.concatenate([[0], np.cumsum(sizes)]).astype(np.int64)


def _ragged_regions(rng, band, n_regions, edge_reads=False, max_haps=45, max_reads=70):
    hap_blocks, read_blocks, toffs = [], [], []
    for g in range(n_regions):
        h, r = random_region(rng, band, n_haps=int(rng.integers(1, max_haps + 1)), n_reads=int(rng.integers(1, max_reads + 1)),
                             hap_len=2 * band + int(rng.choice([200, 260, 330])), read_len_choices=[40, 76, 100, 150], read_n_rate=0.05,
                             edge_reads=edge_reads and g % 2 == 0)
        hap_blocks.append(h); read_blocks.append(r); toffs.append(_template_sizes(rng, r.n))
    return hap_blocks, read_blocks, toffs


def _templates_alone(engine, cfg, haps, reads, toff, flank=None, positions=None):
    """phmm_populate_templates for one region, with its per-read statuses (the C entry point: a short haplotype does not raise here)."""
    from octopus_b200 import _lib
    toff = np.ascontiguousarray(toff, dtype=np.int64)
    out = np.empty((haps.n, len(toff) - 1), dtype=np.float64)
    st = np.empty((haps.n, reads.n), dtype=np.int32)
    hs, rs, cs = haps.c_struct(), reads.c_struct(), cfg.c_struct()
    fs = None if flank is None else _lib.FlankState(1, int(flank[0]), int(flank[1]))
    keep = None if positions is None else (np.ascontiguousarray(positions[0], dtype=np.int64), np.ascontiguousarray(positions[1], dtype=np.int32))
    ps = None if keep is None else _lib.Positions(keep[0].ctypes.data, keep[1].ctypes.data)
    rc = engine._lib.phmm_populate_templates(engine._h, C.byref(cs), C.byref(hs), C.byref(rs), toff.ctypes.data, len(toff) - 1,
                                             C.byref(ps) if ps is not None else None, C.byref(fs) if fs is not None else None,
                                             out.ctypes.data, st.ctypes.data, _lib.SPACE_HOST)
    return rc, out, st


def _sum_templates(per_read, toff):
    """The template values from per-read values: a sum in read order from 0.0, one addition at a time (std::accumulate)."""
    out = np.zeros((per_read.shape[0], len(toff) - 1))
    for t in range(len(toff) - 1):
        for r in range(int(toff[t]), int(toff[t + 1])):
            out[:, t] = out[:, t] + per_read[:, r]
    return out


def _positions_lists(rng, haps, reads, max_len=12):
    """Candidate lists of 0..max_len positions per (haplotype, read) pair, some of them beyond either end of the haplotype."""
    lists = []
    for h in range(haps.n):
        row = []
        for r in range(reads.n):
            p0 = int(reads.begin[r])
            ps = {int(p0 + rng.integers(-15, 16)) for _ in range(int(rng.integers(0, max_len + 1)))}
            if ps and rng.random() < 0.2:
                ps.add(int(rng.choice([-7, haps.length(h) + 3])))           # outside the haplotype
            row.append(sorted(ps)[:max_len])
        lists.append(row)
    return lists


def _pack_lists(list_of_region_lists):
    """CSR over the regions' [H_g][R_g] slots back to back (what phmm_populate_regions_ex takes)."""
    off, flat = [0], []
    for lists in list_of_region_lists:
        for row in lists:
            for ps in row:
                flat.extend(ps)
                off.append(len(flat))
    return np.asarray(off, np.int64), np.asarray(flat if flat else [0], np.int32)


# ---------------------------------------------------------------------------------------------------------------------
# CPU
# ---------------------------------------------------------------------------------------------------------------------
def test_region_templates_struct_matches_header():
    from octopus_b200 import _lib
    assert C.sizeof(_lib.RegionTemplates) == 16
    header = open(os.path.join(ROOT, "include", "phmm_b200.h")).read()
    body = re.search(r"typedef struct \{([^}]*)\} phmm_region_templates;", header).group(1)
    assert re.findall(r"const (\w+)\*\s+(\w+);", body) == [("int32_t", "template_first"), ("int64_t", "template_off")]
    assert [f for f, _ in _lib.RegionTemplates._fields_] == ["template_first", "template_off"]


def test_concat_templates_matches_concat_blocks():
    from octopus_b200.batch import concat_blocks, concat_templates, pack_haplotypes, pack_reads
    s = np.frombuffer(b"ACGTACGTAC", np.uint8)
    hap = lambda: pack_haplotypes([s], [s], [np.full(10, 40, np.int8)], [s], [np.full(10, 40, np.int8)], [np.full(10, 30, np.int8)],   # noqa: E731
                                  [np.full(10, 3, np.int8)])
    reads = lambda n: pack_reads([s[:4]] * n, [np.full(4, 30, np.uint8)] * n)   # noqa: E731
    local = [np.array([0, 2, 3]), np.array([0, 1]), np.array([0, 2, 2, 5])]       # an empty template is allowed
    haps, rb, hf, rf = concat_blocks([hap(), hap(), hap()], [reads(3), reads(1), reads(5)])
    toff, tf = concat_templates(local)
    assert toff.dtype == np.int64 and tf.dtype == np.int32
    assert toff.tolist() == [0, 2, 3, 4, 6, 6, 9] and tf.tolist() == [0, 2, 3, 6]
    assert rb.n == toff[-1]
    for g in range(3):          # each region's templates cover exactly its reads
        assert toff[tf[g]] == rf[g] and toff[tf[g + 1]] == rf[g + 1]
    with pytest.raises(ValueError):
        concat_templates([np.array([0, 2, 1])])


def _build_regions_exe():
    from octopus_b200 import build
    build.build()
    subprocess.run(["g++", "-std=c++14", "-O1", "-I", os.path.join(ROOT, "include"), "-I", os.path.join(ROOT, "octopus_b200", "cpp"),
                    REGIONS_SRC, "-o", REGIONS_EXE, "-L", os.path.join(ROOT, "octopus_b200"), "-lphmm_b200",
                    "-Wl,-rpath," + os.path.join(ROOT, "octopus_b200")], check=True)


def test_region_batch_compiles_against_the_abi():
    _build_regions_exe()
    assert os.path.exists(REGIONS_EXE)


# ---------------------------------------------------------------------------------------------------------------------
# GPU
# ---------------------------------------------------------------------------------------------------------------------
MODES = {"dp_only": dict(disable_naive_shortcut=True, map_positions=False), "mapper": dict(map_positions=True),
         "flank": dict(map_positions=True)}


@pytest.mark.gpu
@pytest.mark.parametrize("band", [8, 16, 32, 64])
@pytest.mark.parametrize("mode", sorted(MODES))
def test_region_templates_equal_one_call_per_region(engine, coracle, band, mode):
    """Ragged regions (1-45 haplotypes, 1-70 reads, templates of 1-3 reads) in one call: each region's [H_g, T_g] equals that region's
    own phmm_populate_templates bit for bit, the per-read statuses are equal, the values are the sums of the region's per-read values
    in read order (exactly) and agree with the oracle."""
    from octopus_b200 import HaplotypeLikelihoodModel
    from octopus_b200.batch import concat_blocks, concat_templates
    from test_gpu_parity import _close
    rng = np.random.default_rng(1000 + band + 7 * sorted(MODES).index(mode))
    hap_blocks, read_blocks, toffs = _ragged_regions(rng, band, int(rng.integers(3, 8)), edge_reads=True)
    flanks = [(int(rng.integers(0, 80)), int(rng.integers(0, 80))) if (mode == "flank" and g % 3) else None for g in range(len(hap_blocks))]
    haps, reads, hf, rf = concat_blocks(hap_blocks, read_blocks)
    toff, tf = concat_templates(toffs)
    cfg = HaplotypeLikelihoodModel.Config(max_indel_error=band, **MODES[mode])
    flat, off, st = engine.populate_regions(cfg, haps, reads, hf, rf, flank_states=flanks, want_status=True, templates=(toff, tf))
    mats = engine.split_regions(flat, off, hf, tf)
    sts = engine.split_regions(st, None, hf, rf)
    for g, (h, r) in enumerate(zip(hap_blocks, read_blocks)):
        rc, one, one_st = _templates_alone(engine, cfg, h, r, toffs[g], flanks[g])
        assert np.array_equal(sts[g], one_st), (band, mode, g)
        assert np.array_equal(mats[g], one), (band, mode, g)
        per_read, pst = engine.populate(cfg, h, r, None, flanks[g], want_status=True)
        assert np.array_equal(pst, one_st) and np.array_equal(_sum_templates(per_read, toffs[g]), one), (band, mode, g)
        _, want, wst = coracle.populate(band, h, r, None, flanks[g], dp_only=cfg.disable_naive_shortcut, map_positions=cfg.map_positions)
        ok_reads = wst == 0
        ok = np.stack([ok_reads[:, a:b].all(axis=1) for a, b in zip(toffs[g][:-1], toffs[g][1:])], axis=1)
        good, worst = _close(mats[g][ok], _sum_templates(want, toffs[g])[ok])
        assert good, (band, mode, g, worst)


# The answers of HaplotypeLikelihoodArray::populate(TemplateMap) compiled from Octopus (oracle/_ref, built only where the Octopus
# sources are) on _reference_case(), recorded in tests/golden/region_templates_reference.json with a digest of the inputs:
#   python tests/test_gpu_region_templates.py --record        (needs oracle/_ref)
REF_GOLDEN = os.path.join(ROOT, "tests", "golden", "region_templates_reference.json")


def _reference_case():
    """Three regions, one with two samples (a sample = a column range of the region's templates), two with a flank state."""
    rng = np.random.default_rng(4242)
    hap_blocks, read_blocks, toffs = _ragged_regions(rng, 16, 3, max_haps=8, max_reads=40)
    flanks = [None, (40, 35), (20, 60)]
    sample_offs = [[0, (len(t) - 1) // 2, len(t) - 1] if g == 0 else [0, len(t) - 1] for g, t in enumerate(toffs)]
    return dict(band_req=12, hap_blocks=hap_blocks, read_blocks=read_blocks, toffs=toffs, flanks=flanks, sample_offs=sample_offs)


def _case_digest(case):
    import hashlib
    h = hashlib.blake2b(digest_size=16)
    h.update(repr((case["band_req"], case["flanks"], case["sample_offs"])).encode())
    for blk in case["hap_blocks"] + case["read_blocks"]:
        for name, a in sorted(blk.arrays().items()):
            h.update(name.encode()); h.update(np.ascontiguousarray(a).tobytes())
    for t in case["toffs"]:
        h.update(np.ascontiguousarray(t, dtype=np.int64).tobytes())
    return h.hexdigest()


def _live_reference(case):
    from oracle.oracle import RefHMM
    ref = RefHMM()
    out = []
    for g in range(len(case["hap_blocks"])):
        st, m, _ = ref.array_populate(case["band_req"], case["hap_blocks"][g], case["read_blocks"][g], sample_off=case["sample_offs"][g],
                                      template_off=case["toffs"][g], flanks=case["flanks"][g])
        out.append((int(st), m))
    return out


def _recorded_reference():
    import json
    with open(REF_GOLDEN) as f:
        rec = json.load(f)
    return rec["digest"], [(r["status"], np.asarray(r["values"], dtype=np.float64).reshape(r["shape"])) for r in rec["regions"]]


def test_recorded_reference_answers_belong_to_the_inputs():
    """The recorded answers were taken on exactly _reference_case()'s inputs, and (where oracle/_ref is built) are still what the
    compiled Octopus code returns."""
    from oracle.oracle import RefHMM
    case = _reference_case()
    digest, recorded = _recorded_reference()
    assert digest == _case_digest(case), "the inputs changed: re-record tests/golden/region_templates_reference.json"
    if RefHMM.available():
        for (st, m), (st_r, m_r) in zip(_live_reference(case), recorded):
            assert st == st_r and m.tobytes() == m_r.tobytes()


@pytest.mark.gpu
def test_region_templates_match_the_compiled_reference(engine):
    """Each region's [H_g, T_g] matrix of one many-regions call against HaplotypeLikelihoodArray::populate(TemplateMap) compiled from
    Octopus (the recorded answers)."""
    from octopus_b200 import HaplotypeLikelihoodModel
    from octopus_b200.batch import concat_blocks, concat_templates
    from test_gpu_parity import _close
    case = _reference_case()
    digest, recorded = _recorded_reference()
    assert digest == _case_digest(case)
    haps, reads, hf, rf = concat_blocks(case["hap_blocks"], case["read_blocks"])
    toff, tf = concat_templates(case["toffs"])
    cfg = HaplotypeLikelihoodModel.Config(max_indel_error=case["band_req"])
    flat, off = engine.populate_regions(cfg, haps, reads, hf, rf, flank_states=case["flanks"], templates=(toff, tf))
    mats = engine.split_regions(flat, off, hf, tf)
    for g, (st, want) in enumerate(recorded):
        assert st == 0 and mats[g].shape == want.shape
        ok, worst = _close(mats[g], want)
        assert ok and np.array_equal(mats[g] == 0.0, want == 0.0), (g, worst)


@pytest.mark.gpu
def test_explicit_positions_across_regions(engine):
    """Candidate lists of 0-12 positions (some outside the haplotype) over several regions, with and without templates: each region
    equals phmm_populate / phmm_populate_templates with the same lists; malformed offsets are refused."""
    from octopus_b200 import HaplotypeLikelihoodModel, PhmmError
    from octopus_b200.batch import concat_blocks, concat_templates, pack_positions
    rng = np.random.default_rng(919)
    for band, dp_only in ((8, False), (16, True), (32, False)):
        hap_blocks, read_blocks, toffs = _ragged_regions(rng, band, 5, max_haps=12, max_reads=30)
        lists = [_positions_lists(rng, h, r) for h, r in zip(hap_blocks, read_blocks)]
        flanks = [(30, 30) if g % 2 else None for g in range(5)]
        haps, reads, hf, rf = concat_blocks(hap_blocks, read_blocks)
        toff, tf = concat_templates(toffs)
        positions = _pack_lists(lists)
        cfg = HaplotypeLikelihoodModel.Config(max_indel_error=band, disable_naive_shortcut=dp_only)
        flat, off, st = engine.populate_regions(cfg, haps, reads, hf, rf, flank_states=flanks, want_status=True, positions=positions)
        tflat, toff_out, tst = engine.populate_regions(cfg, haps, reads, hf, rf, flank_states=flanks, want_status=True, templates=(toff, tf),
                                                       positions=positions)
        assert np.array_equal(st, tst)
        mats, sts = engine.split_regions(flat, off, hf, rf), engine.split_regions(st, off, hf, rf)
        tmats = engine.split_regions(tflat, toff_out, hf, tf)
        for g, (h, r) in enumerate(zip(hap_blocks, read_blocks)):
            p = pack_positions(lists[g], h.n, r.n)
            one, one_st = engine.populate(cfg, h, r, p, flanks[g], want_status=True)
            assert np.array_equal(mats[g], one) and np.array_equal(sts[g], one_st), (band, g)
            rc, tone, tone_st = _templates_alone(engine, cfg, h, r, toffs[g], flanks[g], p)
            assert np.array_equal(tmats[g], tone) and np.array_equal(sts[g], tone_st), (band, g)
        bad_off = positions[0].copy()
        bad_off[len(bad_off) // 2] = bad_off[-1] + 5                      # not non-decreasing
        for tpl in (None, (toff, tf)):
            with pytest.raises(PhmmError) as ei:
                engine.populate_regions(cfg, haps, reads, hf, rf, templates=tpl, positions=(bad_off, positions[1]))
            assert ei.value.code == -1


@pytest.mark.gpu
def test_region_templates_in_device_memory(engine):
    """Torch CUDA blocks, device template_off and device out give the bytes of the host call; a device template crossing a region
    boundary is refused with PHMM_ERR_INVALID (validated on the device)."""
    import torch
    from octopus_b200 import HaplotypeLikelihoodModel, PhmmError
    from octopus_b200.batch import concat_blocks, concat_templates
    rng = np.random.default_rng(31337)
    hap_blocks, read_blocks, toffs = _ragged_regions(rng, 16, 6)
    flanks = [(25, 50) if g % 2 else None for g in range(6)]
    haps, reads, hf, rf = concat_blocks(hap_blocks, read_blocks)
    toff, tf = concat_templates(toffs)
    cfg = HaplotypeLikelihoodModel.Config(max_indel_error=16)
    want, off, wst = engine.populate_regions(cfg, haps, reads, hf, rf, flank_states=flanks, want_status=True, templates=(toff, tf))
    dh, dr = haps.to_device(), reads.to_device()
    dtoff = torch.as_tensor(toff, device="cuda:0")
    out = torch.full((int(off[-1]),), 7.0, dtype=torch.float64, device="cuda:0")
    got, off2, gst = engine.populate_regions(cfg, dh, dr, hf, rf, flank_states=flanks, out=out, want_status=True, templates=(dtoff, tf))
    assert got.data_ptr() == out.data_ptr() and np.array_equal(off, off2)
    assert got.cpu().numpy().tobytes() == want.tobytes() and np.array_equal(gst.cpu().numpy(), wst)
    bad = toff.copy()
    g = 2
    bad[tf[g + 1]] += 1                     # region g's last template takes the first read of region g + 1
    if bad[tf[g + 1]] > bad[tf[g + 1] + 1]:
        bad[tf[g + 1] + 1] = bad[tf[g + 1]]
    with pytest.raises(PhmmError) as ei:
        engine.populate_regions(cfg, dh, dr, hf, rf, templates=(torch.as_tensor(bad, device="cuda:0"), tf))
    assert ei.value.code == -1
    with pytest.raises(PhmmError) as ei:     # the same offsets from the host are refused on the host
        engine.populate_regions(cfg, haps, reads, hf, rf, templates=(bad, tf))
    assert ei.value.code == -1
    again = engine.populate_regions(cfg, dh, dr, hf, rf, flank_states=flanks, templates=(dtoff, tf))[0]   # the engine is still usable
    assert again.cpu().numpy().tobytes() == want.tobytes()


@pytest.mark.gpu
def test_short_haplotype_in_one_region(engine):
    """A short haplotype in one region: the call reports ShortHaplotypeError, only that region's statuses carry PHMM_STATUS_SHORT_HAP,
    and every other region equals its single-region result."""
    from octopus_b200 import HaplotypeLikelihoodModel, ShortHaplotypeError
    from octopus_b200.batch import concat_blocks, concat_templates, pack_haplotypes, pack_reads
    rng = np.random.default_rng(55)
    hap_blocks, read_blocks, toffs = _ragged_regions(rng, 8, 5, max_haps=10, max_reads=30)
    s = np.frombuffer(b"ACGT", np.uint8)[rng.integers(0, 4, 60)]
    k = 3
    hap_blocks[k] = pack_haplotypes([s, s], [s, s], [np.full(60, 50, np.int8)] * 2, [s, s], [np.full(60, 50, np.int8)] * 2,
                                    [np.full(60, 30, np.int8)] * 2, [np.full(60, 3, np.int8)] * 2)
    read_blocks[k] = pack_reads([s[5:55], s[10:40], s[2:52]], [np.full(50, 30, np.uint8), np.full(30, 30, np.uint8), np.full(50, 30, np.uint8)],
                                begin=np.array([5, 10, 2]))
    toffs[k] = np.array([0, 2, 3], dtype=np.int64)
    haps, reads, hf, rf = concat_blocks(hap_blocks, read_blocks)
    toff, tf = concat_templates(toffs)
    cfg = HaplotypeLikelihoodModel.Config(max_indel_error=8)
    with pytest.raises(ShortHaplotypeError):
        engine.populate_regions(cfg, haps, reads, hf, rf, templates=(toff, tf))
    flat, off, st = engine.populate_regions(cfg, haps, reads, hf, rf, want_status=True, templates=(toff, tf))
    mats, sts = engine.split_regions(flat, off, hf, tf), engine.split_regions(st, None, hf, rf)
    for g, (h, r) in enumerate(zip(hap_blocks, read_blocks)):
        rc, one, one_st = _templates_alone(engine, cfg, h, r, toffs[g])
        assert np.array_equal(sts[g], one_st), g
        if g == k:
            assert rc == -4 and ((sts[g] & 0xFFFF) == 2).any()
            continue
        assert rc == 0 and not ((sts[g] & 0xFFFF) == 2).any() and np.array_equal(mats[g], one), g


@pytest.mark.gpu
def test_cpp_region_batch_equals_populate_per_region():
    """RegionBatch (C++ adapter): TemplateMap regions (one with two samples), ReadMap regions and a mixed batch each equal
    HaplotypeLikelihoodArray::populate per region; a short-haplotype region is reported while the others are filled."""
    _build_regions_exe()
    out = subprocess.run([REGIONS_EXE], capture_output=True, text=True, timeout=300)
    assert out.returncode == 0 and "REGIONS ok" in out.stdout, out.stdout + out.stderr
    assert int(out.stdout.split("short_regions=")[1].split()[0]) == 6          # the short region of each of the 6 batches


if __name__ == "__main__" and "--record" in sys.argv:
    import json
    sys.path.insert(0, ROOT)
    case = _reference_case()
    regions = [{"status": st, "shape": list(m.shape), "values": [float(x) for x in m.ravel()]} for st, m in _live_reference(case)]
    with open(REF_GOLDEN, "w") as f:
        json.dump({"what": "HaplotypeLikelihoodArray::populate(TemplateMap) compiled from Octopus on _reference_case()",
                   "digest": _case_digest(case), "regions": regions}, f, indent=0)
        f.write("\n")
