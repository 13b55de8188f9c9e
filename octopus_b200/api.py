"""Host-side mirror of the reference interface for this path, over the C ABI (include/phmm_b200.h).

Names and argument meaning follow the reference:
  * ``PairHMMEngine.align_scores``            ↔ simd::PairHMM::align  (simd_pair_hmm.hpp:454-470), batched
  * ``HaplotypeLikelihoodModel.Config``       ↔ HaplotypeLikelihoodModel::Config (haplotype_likelihood_model.hpp:36-44)
  * ``HaplotypeLikelihoodArray.populate``     ↔ HaplotypeLikelihoodArray::populate (haplotype_likelihood_array.cpp:51-103)
  * ``ShortHaplotypeError``                   ↔ HaplotypeLikelihoodModel::ShortHaplotypeError (:123-139)
Every computing call goes through libphmm_b200.so to the GPU; nothing here computes likelihoods on the CPU.
"""
import ctypes as C

import numpy as np

from . import _lib
from .batch import HaplotypeBlock, ReadBlock


class PhmmError(RuntimeError):
    def __init__(self, code, message):
        super().__init__("phmm error %d: %s" % (code, message))
        self.code = code


class ShortHaplotypeError(PhmmError):
    """Haplotype is too short for alignment (reference: thrown out of populate, caller.cpp:1182-1188 skips the region)."""


class TooLargeBandSizeError(PhmmError):
    """Requested band > 256 (simd_pair_hmm_wrapper.hpp:45-61)."""


def _is_torch(x):
    return hasattr(x, "data_ptr")


class PairHMMEngine:
    """One engine handle (not re-entrant; one per host thread, like the reference's per-thread model copies)."""

    def __init__(self, device=-1):
        self._lib = _lib.load()
        h = C.c_void_p()
        rc = self._lib.phmm_create(C.byref(h), int(device))
        if rc != _lib.PHMM_OK:
            raise PhmmError(rc, self._lib.phmm_last_error(None).decode())
        self._h = h

    def close(self):
        if getattr(self, "_h", None):
            self._lib.phmm_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    def _raise(self, rc):
        msg = self._lib.phmm_last_error(self._h).decode()
        if rc == _lib.PHMM_ERR_SHORT_HAPLOTYPE:
            raise ShortHaplotypeError(rc, msg)
        if rc == _lib.PHMM_ERR_BAND:
            raise TooLargeBandSizeError(rc, msg)
        raise PhmmError(rc, msg)

    # -- stream ordering -----------------------------------------------------------------------------------------
    def wait_event(self, event):
        """Make the engine's stream wait (on the device) for a CUDA event — a torch.cuda.Event or a raw cudaEvent_t — recorded
        after work on another stream that still reads a buffer the next call will overwrite (phmm_wait_event)."""
        handle = getattr(event, "cuda_event", event)
        rc = self._lib.phmm_wait_event(self._h, C.c_void_p(int(handle)))
        if rc != _lib.PHMM_OK:
            self._raise(rc)

    def reserve_sms(self, n):
        """Keep the first n SMs free of persistent DP blocks, for a collective running beside the next call (phmm_reserve_sms)."""
        rc = self._lib.phmm_reserve_sms(self._h, int(n))
        if rc != _lib.PHMM_OK:
            self._raise(rc)

    def stream_handle(self):
        return int(self._lib.phmm_engine_stream(self._h) or 0)

    # -- statistics of the last call -------------------------------------------------------------------------
    def launch_count(self, total=False):
        return int(self._lib.phmm_launch_count(self._h, int(total)))

    def last_dp_kernel_ms(self):
        return float(self._lib.phmm_last_dp_kernel_ms(self._h))

    def last_dp_cells(self):
        return int(self._lib.phmm_last_dp_cells(self._h))

    # -- raw kernel boundary -----------------------------------------------------------------------------------
    def align_scores(self, band, haps: HaplotypeBlock, reads: ReadBlock, tasks, nuc_prior=2, precision_bits=16):
        """tasks: (n, 4) int32 rows (read, hap, win_off, reverse). Returns the integer score of every task, i.e.
        reference ``hmm.align(hap_window, read, quals, L+2*band-1, L, snv_mask, snv_prior, gap_open, gap_extend, nuc_prior)``."""
        dev = haps.on_device
        assert dev == reads.on_device, "haplotypes and reads must live in the same memory space"
        hs, rs = haps.c_struct(), reads.c_struct()
        if dev:
            import torch
            t = tasks if _is_torch(tasks) else torch.as_tensor(np.ascontiguousarray(tasks, dtype=np.int32), device=haps.seq.device)
            t = t.to(torch.int32).contiguous()
            n = t.shape[0]
            out = torch.empty(n, dtype=torch.int32, device=t.device)
            tp, op = t.data_ptr(), out.data_ptr()
        else:
            t = np.ascontiguousarray(tasks, dtype=np.int32).reshape(-1, 4)
            n = t.shape[0]
            out = np.empty(n, dtype=np.int32)
            tp, op = t.ctypes.data, out.ctypes.data
        rc = self._lib.phmm_align_scores(self._h, int(band), int(precision_bits), int(nuc_prior), C.byref(hs), C.byref(rs),
                                         tp, n, op, _lib.SPACE_DEVICE if dev else _lib.SPACE_HOST)
        if rc != _lib.PHMM_OK:
            self._raise(rc)
        return out

    def align(self, band, truth, target, quals, gap_open, gap_extend, nuc_prior=2, snv_mask=None, snv_prior=None):
        """Per-call seam with traceback ↔ simd::PairHMM::align(..., first_pos, align1, align2) (simd_pair_hmm.hpp:472-509).
        Returns (score, first_pos, aligned_truth, aligned_target). gap_extend may be a scalar (the reference's scalar overload)."""
        def as_bytes(x):
            if isinstance(x, str):
                return x.encode()
            if isinstance(x, (bytes, bytearray)):
                return bytes(x)
            return np.ascontiguousarray(np.asarray(x)).view(np.uint8).tobytes()
        t, r = as_bytes(truth), as_bytes(target)
        q = np.ascontiguousarray(np.asarray(quals, dtype=np.int8))
        go = np.ascontiguousarray(np.asarray(gap_open, dtype=np.int8))
        if np.ndim(gap_extend) == 0:
            ge, gep, ges = None, None, int(gap_extend)
        else:
            ge = np.ascontiguousarray(np.asarray(gap_extend, dtype=np.int8)); gep, ges = ge.ctypes.data, 0
        if snv_mask is not None:
            m = as_bytes(snv_mask)
            sp = np.ascontiguousarray(np.asarray(snv_prior, dtype=np.int8)); spp = sp.ctypes.data
        else:
            m, spp = None, None
        n = 2 * (len(r) + band) + 1
        a1, a2 = C.create_string_buffer(n + 8), C.create_string_buffer(n + 8)
        score, fp = C.c_int(0), C.c_int(0)
        rc = self._lib.phmm_align_traceback(self._h, int(band), t, r, q.ctypes.data, len(t), len(r), m, spp, go.ctypes.data, gep, ges,
                                            int(nuc_prior), C.byref(score), C.byref(fp), a1, a2)
        if rc != _lib.PHMM_OK:
            self._raise(rc)
        return score.value, fp.value, a1.value.decode(), a2.value.decode()

    def align_reads(self, config, haps: HaplotypeBlock, reads: ReadBlock, pairs, positions=None, flank_state=None, cigar_stride=None):
        """HaplotypeLikelihoodModel::align for explicit (read, haplotype) pairs (host blocks). pairs: (n, 2) int32 rows (read, hap);
        positions: None or (off[n+1], pos) CSR over the pair list. Returns (mapping_position[n], likelihood[n], cigars[list of str], status[n])."""
        assert not haps.on_device and not reads.on_device
        pr = np.ascontiguousarray(pairs, dtype=np.int32).reshape(-1, 2)
        n = pr.shape[0]
        hs, rs = haps.c_struct(), reads.c_struct()
        cfg = config.c_struct()
        if cigar_stride is None:
            cigar_stride = 4 * int(np.diff(reads.off).max()) + 64
        pstruct = None
        if positions is not None:
            off = np.ascontiguousarray(positions[0], dtype=np.int64)
            pos = np.ascontiguousarray(positions[1], dtype=np.int32)
            pstruct = _lib.Positions(off.ctypes.data, pos.ctypes.data)
        fstruct = None if flank_state is None else _lib.FlankState(1, int(flank_state[0]), int(flank_state[1]))
        mp = np.zeros(n, dtype=np.int64)
        lk = np.zeros(n, dtype=np.float64)
        st = np.zeros(n, dtype=np.int32)
        cg = np.zeros(n * cigar_stride, dtype=np.uint8)
        rc = self._lib.phmm_align_reads(self._h, C.byref(cfg), C.byref(hs), C.byref(rs), pr.ctypes.data, n,
                                        C.byref(pstruct) if pstruct is not None else None, C.byref(fstruct) if fstruct is not None else None,
                                        mp.ctypes.data, lk.ctypes.data, cg.ctypes.data, cigar_stride, st.ctypes.data, _lib.SPACE_HOST)
        if rc != _lib.PHMM_OK:
            self._raise(rc)
        cigars = [bytes(cg[j * cigar_stride:(j + 1) * cigar_stride]).split(b"\0", 1)[0].decode() for j in range(n)]
        return mp, lk, cigars, st

    def align_pairs(self, config, truths: HaplotypeBlock, targets: ReadBlock, pairs, target_offsets, flank_state=None, cigar_stride=None):
        """hmm::align batched (phmm_align_pairs): pair j = (target pairs[j][0], truth pairs[j][1]) at target_offsets[j]. Host blocks.
        Returns (target_offset[n], likelihood[n], cigars, status[n])."""
        assert not truths.on_device and not targets.on_device
        pr = np.ascontiguousarray(pairs, dtype=np.int32).reshape(-1, 2)
        n = pr.shape[0]
        offs = np.ascontiguousarray(target_offsets, dtype=np.int32)
        assert len(offs) == n
        hs, rs, cfg = truths.c_struct(), targets.c_struct(), config.c_struct()
        if cigar_stride is None:
            cigar_stride = 4 * int(np.diff(targets.off).max()) + 64
        fstruct = None if flank_state is None else _lib.FlankState(1, int(flank_state[0]), int(flank_state[1]))
        mp, lk, st = np.zeros(n, dtype=np.int64), np.zeros(n, dtype=np.float64), np.zeros(n, dtype=np.int32)
        cg = np.zeros(n * cigar_stride, dtype=np.uint8)
        rc = self._lib.phmm_align_pairs(self._h, C.byref(cfg), C.byref(hs), C.byref(rs), pr.ctypes.data, offs.ctypes.data, n,
                                        C.byref(fstruct) if fstruct is not None else None,
                                        mp.ctypes.data, lk.ctypes.data, cg.ctypes.data, cigar_stride, st.ctypes.data, _lib.SPACE_HOST)
        if rc != _lib.PHMM_OK:
            self._raise(rc)
        cigars = [bytes(cg[j * cigar_stride:(j + 1) * cigar_stride]).split(b"\0", 1)[0].decode() for j in range(n)]
        return mp, lk, cigars, st

    def genotype_likelihoods(self, lnl, genotypes):
        """ConstantMixtureGenotypeLikelihoodModel::evaluate for every row of `genotypes` ((G, ploidy) haplotype indices) over the
        (H, R) matrix `lnl` (numpy on the host, or a torch CUDA tensor left where populate produced it). Returns G doubles."""
        if _is_torch(lnl):
            import torch
            m = lnl.contiguous()
            gt = torch.as_tensor(np.ascontiguousarray(genotypes, dtype=np.int32), device=m.device)
            out = torch.empty(gt.shape[0], dtype=torch.float64, device=m.device)
            rc = self._lib.phmm_genotype_likelihoods(self._h, m.data_ptr(), m.shape[0], m.shape[1], gt.data_ptr(), gt.shape[0], gt.shape[1],
                                                     out.data_ptr(), _lib.SPACE_DEVICE)
        else:
            m = np.ascontiguousarray(lnl, dtype=np.float64)
            gt = np.ascontiguousarray(genotypes, dtype=np.int32)
            out = np.empty(gt.shape[0], dtype=np.float64)
            rc = self._lib.phmm_genotype_likelihoods(self._h, m.ctypes.data, m.shape[0], m.shape[1], gt.ctypes.data, gt.shape[0], gt.shape[1],
                                                     out.ctypes.data, _lib.SPACE_HOST)
        if rc != _lib.PHMM_OK:
            self._raise(rc)
        return out

    # -- batch boundary ----------------------------------------------------------------------------------------
    def populate_templates(self, config, haps: HaplotypeBlock, reads: ReadBlock, template_off, flank_state=None, positions=None):
        """HaplotypeLikelihoodArray::populate(TemplateMap): host blocks; template t = reads [template_off[t], template_off[t+1]).
        Returns the (H, T) matrix: each entry the sum of the template's reads' ln-likelihoods. positions: as in ``populate``."""
        assert not haps.on_device and not reads.on_device
        toff = np.ascontiguousarray(template_off, dtype=np.int64)
        T = len(toff) - 1
        hs, rs, cfg = haps.c_struct(), reads.c_struct(), config.c_struct()
        fstruct = None if flank_state is None else _lib.FlankState(1, int(flank_state[0]), int(flank_state[1]))
        pstruct, keep = None, None
        if positions is not None:
            keep = (np.ascontiguousarray(positions[0], dtype=np.int64), np.ascontiguousarray(positions[1], dtype=np.int32))
            pstruct = _lib.Positions(keep[0].ctypes.data, keep[1].ctypes.data)
        out = np.empty((haps.n, T), dtype=np.float64)
        rc = self._lib.phmm_populate_templates(self._h, C.byref(cfg), C.byref(hs), C.byref(rs), toff.ctypes.data, T,
                                               C.byref(pstruct) if pstruct is not None else None,
                                               C.byref(fstruct) if fstruct is not None else None, out.ctypes.data, None, _lib.SPACE_HOST)
        if rc != _lib.PHMM_OK:
            self._raise(rc)
        return out

    def populate_regions(self, config, haps: HaplotypeBlock, reads: ReadBlock, hap_first, read_first, flank_states=None, out=None, want_status=False,
                         templates=None, positions=None):
        """Many regions in one call (phmm_populate_regions / phmm_populate_regions_ex): region g owns haplotypes [hap_first[g], hap_first[g+1])
        and reads [read_first[g], read_first[g+1]). Returns the flat result vector (the regions' [H_g, R_g] matrices back to back) and the
        per-region offsets into it; ``split_regions`` cuts it into matrices. flank_states: None or a list of (lhs, rhs) / None.

        templates: None, or (template_off, template_first) as ``batch.concat_templates`` returns them — region g owns the templates
        [template_first[g], template_first[g+1]), template t the reads [template_off[t], template_off[t+1]). The result then holds the
        regions' [H_g, T_g] matrices of template values (``split_regions(flat, off, hap_first, template_first)``); the status stays per
        read ([H_g, R_g]: ``split_regions(status, None, hap_first, read_first)``). template_first is host memory in every case.
        positions: None, or (off, pos), a CSR of candidate positions over the per-read result slots (the status layout)."""
        dev = haps.on_device
        assert dev == reads.on_device
        hf = np.ascontiguousarray(hap_first, dtype=np.int32)
        rf = np.ascontiguousarray(read_first, dtype=np.int32)
        G = len(hf) - 1
        tf = None if templates is None else np.ascontiguousarray(templates[1], dtype=np.int32)
        off = self.region_offsets(hf, rf if tf is None else tf)
        total = int(off[-1])
        n_status = int(self.region_offsets(hf, rf)[-1])
        keep = []

        def in_space(a, dtype):
            if dev:
                import torch
                t = a if _is_torch(a) else torch.as_tensor(np.ascontiguousarray(a, dtype=dtype), device=haps.seq.device)
                keep.append(t)
                return t.data_ptr()
            a = np.ascontiguousarray(a, dtype=dtype)
            keep.append(a)
            return a.ctypes.data
        tstruct = None if tf is None else _lib.RegionTemplates(tf.ctypes.data, in_space(templates[0], np.int64))
        pstruct = None if positions is None else _lib.Positions(in_space(positions[0], np.int64), in_space(positions[1], np.int32))
        fl = None
        if flank_states is not None:
            fl = (_lib.FlankState * G)()
            for g, f in enumerate(flank_states):
                if f is not None:
                    fl[g] = _lib.FlankState(1, int(f[0]), int(f[1]))
        regs = _lib.Regions(G, hf.ctypes.data, rf.ctypes.data, C.addressof(fl) if fl is not None else None)
        hs, rs = haps.c_struct(), reads.c_struct()
        cfg = config.c_struct() if hasattr(config, "c_struct") else config
        status = None
        if dev:
            import torch
            if out is None:
                out = torch.empty(total, dtype=torch.float64, device=haps.seq.device)
            if want_status:
                status = torch.empty(n_status, dtype=torch.int32, device=haps.seq.device)
            op, sp = out.data_ptr(), (status.data_ptr() if want_status else None)
        else:
            if out is None:
                out = np.empty(total, dtype=np.float64)
            if want_status:
                status = np.empty(n_status, dtype=np.int32)
            op, sp = out.ctypes.data, (status.ctypes.data if want_status else None)
        space = _lib.SPACE_DEVICE if dev else _lib.SPACE_HOST
        if tstruct is None and pstruct is None:
            rc = self._lib.phmm_populate_regions(self._h, C.byref(cfg), C.byref(hs), C.byref(rs), C.byref(regs), op, sp, space)
        else:
            rc = self._lib.phmm_populate_regions_ex(self._h, C.byref(cfg), C.byref(hs), C.byref(rs), C.byref(regs),
                                                    C.byref(tstruct) if tstruct is not None else None,
                                                    C.byref(pstruct) if pstruct is not None else None, op, sp, space)
        if rc != _lib.PHMM_OK and not (rc == _lib.PHMM_ERR_SHORT_HAPLOTYPE and want_status):
            self._raise(rc)
        return (out, off, status) if want_status else (out, off)

    @staticmethod
    def region_offsets(hap_first, col_first):
        """Where each region's [H_g, C_g] matrix starts in a flat populate_regions result (C_g: reads, or templates)."""
        sizes = np.diff(np.asarray(hap_first, dtype=np.int64)) * np.diff(np.asarray(col_first, dtype=np.int64))
        return np.concatenate([[0], np.cumsum(sizes)]).astype(np.int64)

    @staticmethod
    def split_regions(flat, off, hap_first, col_first):
        """The per-region [H_g, C_g] views of a populate_regions result: col_first is read_first for per-read results (and the status),
        template_first for template values. off: the offsets populate_regions returned, or None (computed from the widths)."""
        if off is None:
            off = PairHMMEngine.region_offsets(hap_first, col_first)
        return [flat[int(off[g]):int(off[g + 1])].reshape(int(hap_first[g + 1] - hap_first[g]), int(col_first[g + 1] - col_first[g]))
                for g in range(len(off) - 1)]

    def populate(self, config, haps: HaplotypeBlock, reads: ReadBlock, positions=None, flank_state=None, out=None,
                 want_status=False):
        """Returns the (H, R) matrix of ln-likelihoods (numpy float64, or a torch CUDA tensor for device-resident blocks).
        positions: None or (off[H*R+1] int64, pos int32) CSR in [H][R] order. flank_state: None or (lhs_flank, rhs_flank)."""
        dev = haps.on_device
        assert dev == reads.on_device, "haplotypes and reads must live in the same memory space"
        H, R = haps.n, reads.n
        hs, rs = haps.c_struct(), reads.c_struct()
        cfg = config.c_struct() if hasattr(config, "c_struct") else config
        keep = []
        pstruct = None
        if positions is not None:
            off, pos = positions
            if dev:
                import torch
                off = off if _is_torch(off) else torch.as_tensor(np.ascontiguousarray(off, dtype=np.int64), device=haps.seq.device)
                pos = pos if _is_torch(pos) else torch.as_tensor(np.ascontiguousarray(pos, dtype=np.int32), device=haps.seq.device)
                pstruct = _lib.Positions(off.data_ptr(), pos.data_ptr())
            else:
                off = np.ascontiguousarray(off, dtype=np.int64)
                pos = np.ascontiguousarray(pos, dtype=np.int32)
                pstruct = _lib.Positions(off.ctypes.data, pos.ctypes.data)
            keep += [off, pos]
        fstruct = None
        if flank_state is not None:
            fstruct = _lib.FlankState(1, int(flank_state[0]), int(flank_state[1]))
        status = None
        if dev:
            import torch
            if out is None:
                out = torch.empty((H, R), dtype=torch.float64, device=haps.seq.device)
            if want_status:
                status = torch.empty((H, R), dtype=torch.int32, device=haps.seq.device)
            op, sp = out.data_ptr(), (status.data_ptr() if want_status else None)
            if tuple(out.shape) != (H, R) or out.dtype != torch.float64 or (R > 1 and out.stride(1) != 1):
                raise ValueError("out must be a float64 [H, R] tensor with unit column stride")
            if H > 1 and out.stride(0) != R:
                # a column window of a wider matrix — possibly another GPU's (octopus_b200.peer): phmm_populate_ld
                rc = self._lib.phmm_populate_ld(self._h, C.byref(cfg), C.byref(hs), C.byref(rs),
                                                C.byref(pstruct) if pstruct is not None else None,
                                                C.byref(fstruct) if fstruct is not None else None, op, int(out.stride(0)), sp)
                if rc != _lib.PHMM_OK and not (rc == _lib.PHMM_ERR_SHORT_HAPLOTYPE and want_status):
                    self._raise(rc)
                return (out, status) if want_status else out
        else:
            if out is None:
                out = np.empty((H, R), dtype=np.float64)
            if want_status:
                status = np.empty((H, R), dtype=np.int32)
            op, sp = out.ctypes.data, (status.ctypes.data if want_status else None)
        rc = self._lib.phmm_populate(self._h, C.byref(cfg), C.byref(hs), C.byref(rs),
                                     C.byref(pstruct) if pstruct is not None else None,
                                     C.byref(fstruct) if fstruct is not None else None,
                                     op, sp, _lib.SPACE_DEVICE if dev else _lib.SPACE_HOST)
        if rc != _lib.PHMM_OK:
            if rc == _lib.PHMM_ERR_SHORT_HAPLOTYPE and want_status:
                return out, status
            self._raise(rc)
        return (out, status) if want_status else out


class ErrorModel:
    """The reference's sequencing-error models behind HaplotypeLikelihoodModel::reset (haplotype_likelihood_model.cpp:60-78):
    make_error_model(label) / make_error_model(file) (core/models/error/error_model_factory.cpp:531-589). ``reset`` turns
    haplotype sequences into the HaplotypeBlock the engine consumes (host C++ inside libphmm_b200.so, no GPU involved)."""

    def __init__(self, label=None, custom_model_text=None):
        self._lib = _lib.load()
        h = C.c_void_p()
        if custom_model_text is not None:
            rc = self._lib.phmm_error_model_create_custom(C.byref(h), custom_model_text.encode() if isinstance(custom_model_text, str) else custom_model_text)
        else:
            rc = self._lib.phmm_error_model_create(C.byref(h), None if label is None else label.encode())
        if rc != _lib.PHMM_OK:
            raise PhmmError(rc, self._lib.phmm_error_model_last_error().decode())
        self._h = h

    def __del__(self):
        try:
            if getattr(self, "_h", None):
                self._lib.phmm_error_model_destroy(self._h)
                self._h = None
        except Exception:
            pass

    def tandem_repeats(self, sequence, min_period=1, max_period=5):
        """tandem::extract_exact_tandem_repeats (lib/tandem/tandem.hpp:504-521): (n, 3) uint32 rows (pos, length, period)."""
        s = np.ascontiguousarray(np.frombuffer(sequence.encode() if isinstance(sequence, str) else bytes(sequence), dtype=np.uint8))
        cap = 4 * len(s) + 16
        while True:
            out = np.zeros((cap, 3), dtype=np.uint32)
            n = self._lib.phmm_tandem_repeats(s.ctypes.data, len(s), int(min_period), int(max_period), out.ctypes.data, cap)
            if n < 0:
                raise PhmmError(n, self._lib.phmm_error_model_last_error().decode())
            if n <= cap:
                return out[:n]
            cap = n

    def reset(self, sequences, begin=None, is_substitution=None, n_threads=0):
        """HaplotypeLikelihoodModel::reset for every haplotype: sequences (list of str / bytes / uint8 arrays) → HaplotypeBlock
        with the SNV masks / priors and gap penalties the reference's models assign. ``is_substitution``: optional list of
        per-base flag arrays (bases that are substitutions in Haplotype::cigar())."""
        parts = [np.frombuffer(x.encode() if isinstance(x, str) else bytes(x), dtype=np.uint8) if not isinstance(x, np.ndarray) else
                 np.ascontiguousarray(x).view(np.uint8).reshape(-1) for x in sequences]
        off = np.zeros(len(parts) + 1, dtype=np.int64)
        np.cumsum([len(x) for x in parts], out=off[1:])
        seq = np.ascontiguousarray(np.concatenate(parts)) if parts else np.zeros(0, dtype=np.uint8)
        return self.reset_block(off, seq, begin, None if is_substitution is None else
                                np.ascontiguousarray(np.concatenate([np.asarray(x, dtype=np.uint8) for x in is_substitution])), n_threads)

    def reset_block(self, off, seq, begin=None, is_substitution=None, n_threads=0):
        off = np.ascontiguousarray(off, dtype=np.int64)
        seq = np.ascontiguousarray(seq, dtype=np.uint8)
        total = int(off[-1])
        mf, mr = np.empty(total, dtype=np.uint8), np.empty(total, dtype=np.uint8)
        pf, pr, go, ge = (np.empty(total, dtype=np.int8) for _ in range(4))
        rc = self._lib.phmm_reset_haplotypes(self._h, len(off) - 1, off.ctypes.data, seq.ctypes.data,
                                             None if is_substitution is None else is_substitution.ctypes.data,
                                             mf.ctypes.data, pf.ctypes.data, mr.ctypes.data, pr.ctypes.data, go.ctypes.data, ge.ctypes.data, int(n_threads))
        if rc != _lib.PHMM_OK:
            raise PhmmError(rc, self._lib.phmm_error_model_last_error().decode())
        return HaplotypeBlock(off, seq, mf, pf, mr, pr, go, ge, begin)


class HaplotypeLikelihoodModel:
    """Configuration holder with the reference's names (the per-haplotype state lives in the HaplotypeBlock)."""

    class Config:
        def __init__(self, use_mapping_quality=True, mapping_quality_cap_trigger=None, mapping_quality_cap=120,
                     use_flank_state=True, max_indel_error=8, use_int_scores=False, nuc_prior=2,
                     disable_naive_shortcut=False, map_positions=True):
            self.use_mapping_quality = use_mapping_quality
            self.mapping_quality_cap_trigger = mapping_quality_cap_trigger
            self.mapping_quality_cap = mapping_quality_cap
            self.use_flank_state = use_flank_state
            self.max_indel_error = max_indel_error
            self.use_int_scores = use_int_scores
            self.nuc_prior = nuc_prior
            self.disable_naive_shortcut = disable_naive_shortcut
            self.map_positions = map_positions   # run the reference's k-mer mapper on the device when no positions are given

        def c_struct(self):
            trig = self.mapping_quality_cap_trigger
            # haplotype_likelihood_model.cpp:50-52: a trigger >= the cap is dropped
            if trig is not None and trig >= self.mapping_quality_cap:
                trig = None
            return _lib.Config(int(self.max_indel_error), int(self.use_int_scores), int(self.use_mapping_quality),
                               int(self.mapping_quality_cap), -1 if trig is None else int(trig),
                               int(self.use_flank_state), int(self.nuc_prior), int(self.disable_naive_shortcut),
                               int(self.map_positions))

    def __init__(self, config=None):
        self.config = config or HaplotypeLikelihoodModel.Config()

    def pad_requirement(self):
        """hmm_.band_size() (haplotype_likelihood_model.cpp:55-58): smallest of 8,16,...,256 >= max_indel_error."""
        b = 8
        while b < self.config.max_indel_error:
            b *= 2
        return b


class HaplotypeLikelihoodArray:
    """likelihoods_[haplotype][sample][read or template] (haplotype_likelihood_array.hpp:34-175).

    All samples of a populate() go to the GPU as one batch: their reads are concatenated, one engine call fills one
    [H, R_total] matrix and a sample is a column range of it (views, no copies)."""

    mapperKmerSize = 6          # haplotype_likelihood_array.hpp:103
    maxMappingPositions = 10    # :104

    def __init__(self, likelihood_model=None, engine=None):
        self.likelihood_model = likelihood_model or HaplotypeLikelihoodModel()
        self._engine = engine
        self.likelihoods = None     # [H, sum of the samples' widths]
        self._samples = []
        self._off = [0]
        self._primed = None

    @property
    def engine(self):
        if self._engine is None:
            self._engine = PairHMMEngine()
        return self._engine

    @staticmethod
    def _concat_reads(blocks):
        if len(blocks) == 1:
            return blocks[0]
        off = [np.zeros(1, dtype=np.int64)]
        base = 0
        for b in blocks:
            off.append(b.off[1:] + base)
            base += int(b.off[-1])
        return ReadBlock(np.concatenate(off), np.concatenate([b.bases for b in blocks]), np.concatenate([b.quals for b in blocks]),
                         np.concatenate([b.mapq for b in blocks]), np.concatenate([b.reverse for b in blocks]),
                         np.concatenate([b.begin for b in blocks]))

    def _set_samples(self, names, widths):
        self._samples = list(names)
        self._off = [0]
        for w in widths:
            self._off.append(self._off[-1] + int(w))
        self._primed = None

    def populate(self, reads, haplotypes: HaplotypeBlock, flank_state=None, positions=None):
        """populate(ReadMap, haplotypes, flank_state) (haplotype_likelihood_array.cpp:51-103). ``reads``: a dict
        {sample: ReadBlock} in sample order, or one ReadBlock (a single unnamed sample, left primed)."""
        if isinstance(reads, ReadBlock):
            self._set_samples([""], [reads.n])
            self.likelihoods = self.engine.populate(self.likelihood_model.config, haplotypes, reads, positions, flank_state)
            self._primed = 0
            return self
        names = list(reads.keys())
        blocks = [reads[k] for k in names]
        self._set_samples(names, [b.n for b in blocks])
        self.likelihoods = self.engine.populate(self.likelihood_model.config, haplotypes, self._concat_reads(blocks), positions, flank_state)
        return self

    def populate_templates(self, templates, haplotypes: HaplotypeBlock, flank_state=None):
        """populate(TemplateMap, ...) (:105-199). ``templates``: {sample: (ReadBlock, template_off)} — template t of the sample
        owns its reads [template_off[t], template_off[t+1]); one value per (haplotype, template)."""
        names = list(templates.keys())
        blocks, toff, base = [], [np.zeros(1, dtype=np.int64)], 0
        for k in names:
            rb, off = templates[k]
            off = np.asarray(off, dtype=np.int64)
            assert off[0] == 0 and off[-1] == rb.n, "template offsets must cover the sample's reads"
            blocks.append(rb)
            toff.append(off[1:] + base)
            base += rb.n
        self._set_samples(names, [len(templates[k][1]) - 1 for k in names])
        self.likelihoods = self.engine.populate_templates(self.likelihood_model.config, haplotypes, self._concat_reads(blocks),
                                                          np.concatenate(toff), flank_state)
        return self

    # -- accessors (haplotype_likelihood_array.cpp:200-291) ----------------------------------------------------
    def samples(self):
        return list(self._samples)

    def _sample_index(self, sample):
        try:
            return self._samples.index(sample)
        except ValueError:
            raise KeyError(sample) from None      # the reference's unordered_map::at

    def num_likelihoods(self, sample=None):
        s = self._primed_index() if sample is None else self._sample_index(sample)
        return self._off[s + 1] - self._off[s]

    def __call__(self, sample, haplotype_index):
        s = self._sample_index(sample)
        return self.likelihoods[haplotype_index, self._off[s]:self._off[s + 1]]

    def __getitem__(self, haplotype_index):
        """likelihoods_[haplotype][primed sample] (:224-236)."""
        s = self._primed_index()
        return self.likelihoods[haplotype_index, self._off[s]:self._off[s + 1]]

    def extract_sample(self, sample):
        s = self._sample_index(sample)
        return self.likelihoods[:, self._off[s]:self._off[s + 1]]

    def is_empty(self):
        return self.likelihoods is None

    def clear(self):
        self.likelihoods = None
        self._set_samples([], [])

    def is_primed(self):
        return self._primed is not None

    def prime(self, sample):
        self._primed = self._sample_index(sample)

    def unprime(self):
        self._primed = None

    def _primed_index(self):
        if self._primed is None:
            raise RuntimeError("HaplotypeLikelihoodArray is not primed")      # an assert in the reference
        return self._primed

    def reset(self, haplotypes_to_keep):
        """reset(haplotypes) (:331-360): keep a subset of the haplotypes, given by their ascending old indices."""
        keep = [int(h) for h in haplotypes_to_keep]
        if not keep:
            self.clear()
            return
        assert all(a < b for a, b in zip(keep, keep[1:])) and 0 <= keep[0] and keep[-1] < self.likelihoods.shape[0]
        self.likelihoods = self.likelihoods[keep]

    def merge_samples(self, samples=None, new_sample=None):
        """merge_samples (:362-409): a one-sample array holding the chosen samples' likelihoods back to back; primed."""
        samples = self.samples() if samples is None else list(samples)
        idx = [self._sample_index(s) for s in samples]
        out = HaplotypeLikelihoodArray(self.likelihood_model, self._engine)
        parts = [self.likelihoods[:, self._off[s]:self._off[s + 1]] for s in idx]
        if isinstance(self.likelihoods, np.ndarray):
            out.likelihoods = np.concatenate(parts, axis=1)
        else:                                                   # device-resident matrix (torch tensor)
            import torch
            out.likelihoods = torch.cat(parts, dim=1)
        out._set_samples(["".join(samples) if new_sample is None else new_sample], [out.likelihoods.shape[1]])
        out._primed = 0
        return out
