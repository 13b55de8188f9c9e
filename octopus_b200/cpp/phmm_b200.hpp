// phmm_b200.hpp — C++ host-side adapter over the C ABI (include/phmm_b200.h), mirroring the reference's own
// interface for the pair-HMM path so that Octopus code compiles against it unchanged:
//
//   octopus_b200::GpuPairHMM<Band>   satisfies the duck-typed PairHMM concept that octopus::hmm::evaluate / align are
//                                    templated on (src/core/models/pairhmm/pair_hmm.hpp:373-380, 397-406, 441-451, 471-483,
//                                    542-551, 590-601; canonical signatures simd_pair_hmm.hpp:433-549):
//                                    band_size(), name(), 4 x align(), calculate_flank_score().
//   octopus_b200::HaplotypeLikelihoodArray  the batch seam: populate(reads, haplotypes, flank_state) fills the
//                                    [haplotype][read] matrix (haplotype_likelihood_array.hpp:65-72, .cpp:51-103) and throws
//                                    ShortHaplotypeError exactly where the reference does (haplotype_likelihood_model.cpp:238-256).
//
// Header-only; link with -lphmm_b200. All likelihood arithmetic runs on the GPU behind the C ABI; the only host
// arithmetic here is calculate_flank_score, which in the reference too is a scalar replay of two alignment strings
// (simd_pair_hmm.hpp:352-430), not part of the DP.
#ifndef PHMM_B200_HPP
#define PHMM_B200_HPP

#include <algorithm>
#include <cstddef>
#include <cstdint>
#include <cstdlib>
#include <memory>
#include <new>
#include <stdexcept>
#include <string>
#include <utility>
#include <vector>

#include "phmm_b200.h"

namespace octopus_b200 {

class Error : public std::runtime_error
{
public:
    Error(int code, const std::string& what) : std::runtime_error {what}, code_ {code} {}
    int code() const noexcept { return code_; }
private:
    int code_;
};

// HaplotypeLikelihoodModel::ShortHaplotypeError (haplotype_likelihood_model.hpp:123-139)
class ShortHaplotypeError : public std::runtime_error
{
public:
    ShortHaplotypeError(std::size_t haplotype_index, unsigned required_extension)
    : std::runtime_error {"Haplotype is too short for alignment"}, haplotype_index_ {haplotype_index}, required_extension_ {required_extension} {}
    std::size_t haplotype_index() const noexcept { return haplotype_index_; }
    unsigned required_extension() const noexcept { return required_extension_; }
private:
    std::size_t haplotype_index_;
    unsigned required_extension_;
};

// simd::PairHMMWrapper::TooLargeBandSizeError (simd_pair_hmm_wrapper.hpp:45-61)
class TooLargeBandSizeError : public std::runtime_error
{
public:
    explicit TooLargeBandSizeError(unsigned band) : std::runtime_error {"Band size too large"}, band_ {band} {}
    unsigned band() const noexcept { return band_; }
private:
    unsigned band_;
};

class Engine
{
public:
    explicit Engine(int device = -1)
    {
        phmm_engine* e = nullptr;
        const int rc = phmm_create(&e, device);
        if (rc != PHMM_OK) throw Error {rc, phmm_last_error(nullptr)};
        handle_.reset(e, [] (phmm_engine* p) { phmm_destroy(p); });
    }
    phmm_engine* get() const noexcept { return handle_.get(); }
    void check(int rc) const
    {
        if (rc == PHMM_OK) return;
        throw Error {rc, phmm_last_error(handle_.get())};
    }
private:
    std::shared_ptr<phmm_engine> handle_;
};

// Page-locked storage for the batch blocks: a std::allocator over phmm_host_alloc (cudaHostAlloc) that falls back to malloc where
// no GPU is usable. The blocks below are vectors of this allocator, so a populate() copies straight from / to pinned memory.
template <typename T>
struct PinnedAllocator
{
    using value_type = T;
    PinnedAllocator() = default;
    template <typename U> PinnedAllocator(const PinnedAllocator<U>&) noexcept {}
    T* allocate(std::size_t n)
    {
        // one tag word in front of the block remembers where it came from
        const std::size_t bytes = n * sizeof(T) + kHeader;
        char* p = static_cast<char*>(phmm_host_alloc(bytes));
        const bool pinned = p != nullptr;
        if (!p) p = static_cast<char*>(std::malloc(bytes));
        if (!p) throw std::bad_alloc {};
        *reinterpret_cast<std::size_t*>(p) = pinned ? 1 : 0;
        return reinterpret_cast<T*>(p + kHeader);
    }
    void deallocate(T* q, std::size_t) noexcept
    {
        char* p = reinterpret_cast<char*>(q) - kHeader;
        if (*reinterpret_cast<std::size_t*>(p)) phmm_host_free(p); else std::free(p);
    }
    template <typename U> bool operator==(const PinnedAllocator<U>&) const noexcept { return true; }
    template <typename U> bool operator!=(const PinnedAllocator<U>&) const noexcept { return false; }
private:
    static constexpr std::size_t kHeader = 64;   // keeps the payload 64-byte aligned
};
template <typename T> using pinned_vector = std::vector<T, PinnedAllocator<T>>;

// The reference's sequencing-error models (core/models/error/error_model_factory.cpp:531-589), i.e. what
// HaplotypeLikelihoodModel::reset runs per haplotype (haplotype_likelihood_model.cpp:60-78) — bit-identical, in the library.
class ErrorModel
{
public:
    explicit ErrorModel(const std::string& label = "PCR-free.HiSeq-2500")
    {
        phmm_error_model* m = nullptr;
        const int rc = phmm_error_model_create(&m, label.c_str());
        if (rc != PHMM_OK) throw Error {rc, phmm_error_model_last_error()};
        handle_.reset(m, [] (phmm_error_model* p) { phmm_error_model_destroy(p); });
    }
    static ErrorModel from_custom_model_text(const std::string& text)   // the contents of a --sequence-error-model file
    {
        phmm_error_model* m = nullptr;
        const int rc = phmm_error_model_create_custom(&m, text.c_str());
        if (rc != PHMM_OK) throw Error {rc, phmm_error_model_last_error()};
        ErrorModel result {std::shared_ptr<phmm_error_model>(m, [] (phmm_error_model* p) { phmm_error_model_destroy(p); })};
        return result;
    }
    const phmm_error_model* get() const noexcept { return handle_.get(); }
private:
    explicit ErrorModel(std::shared_ptr<phmm_error_model> h) : handle_ {std::move(h)} {}
    std::shared_ptr<phmm_error_model> handle_;
};

// ---------------------------------------------------------------------------------------------------------------------
// Per-call seam
// ---------------------------------------------------------------------------------------------------------------------
template <int BandSize>
class GpuPairHMM
{
public:
    using ScoreType = int;
    constexpr static char gap_label = '-';

    explicit GpuPairHMM(Engine engine = Engine {}) : engine_ {std::move(engine)} {}

    constexpr static const char* name() noexcept { return "B200"; }
    constexpr static int band_size() noexcept { return BandSize; }

    // score only, no SNV model (simd_pair_hmm.hpp:438-452)
    template <typename GapExtend>
    int align(const char* truth, const char* target, const std::int8_t* qualities, int truth_len, int target_len,
              const std::int8_t* gap_open, GapExtend gap_extend, short nuc_prior) const noexcept
    {
        int first_pos;
        return run(truth, target, qualities, truth_len, target_len, nullptr, nullptr, gap_open, gap_extend, nuc_prior, first_pos, nullptr, nullptr);
    }
    // score only, SNV model (:454-470)
    template <typename GapExtend>
    int align(const char* truth, const char* target, const std::int8_t* qualities, int truth_len, int target_len,
              const char* snv_mask, const std::int8_t* snv_prior, const std::int8_t* gap_open, GapExtend gap_extend, short nuc_prior) const noexcept
    {
        int first_pos;
        return run(truth, target, qualities, truth_len, target_len, snv_mask, snv_prior, gap_open, gap_extend, nuc_prior, first_pos, nullptr, nullptr);
    }
    // traceback, no SNV model (:472-489)
    template <typename GapExtend>
    int align(const char* truth, const char* target, const std::int8_t* qualities, int truth_len, int target_len,
              const std::int8_t* gap_open, GapExtend gap_extend, short nuc_prior, int& first_pos, char* align1, char* align2) const noexcept
    {
        return run(truth, target, qualities, truth_len, target_len, nullptr, nullptr, gap_open, gap_extend, nuc_prior, first_pos, align1, align2);
    }
    // traceback, SNV model (:491-509)
    template <typename GapExtend>
    int align(const char* truth, const char* target, const std::int8_t* qualities, int truth_len, int target_len,
              const char* snv_mask, const std::int8_t* snv_prior, const std::int8_t* gap_open, GapExtend gap_extend, short nuc_prior,
              int& first_pos, char* align1, char* align2) const noexcept
    {
        return run(truth, target, qualities, truth_len, target_len, snv_mask, snv_prior, gap_open, gap_extend, nuc_prior, first_pos, align1, align2);
    }

    // simd_pair_hmm.hpp:530-549 (SNV overload): replay of the alignment strings; scalar on the host in the reference too
    template <typename GapExtend>
    int calculate_flank_score(int truth_len, int lhs_flank_len, int rhs_flank_len, const char* target, const std::int8_t* quals,
                              const char* snv_mask, const std::int8_t* snv_prior, const std::int8_t* gap_open, GapExtend gap_extend,
                              short nuc_prior, int first_pos, const char* aln1, const char* aln2, int& target_mask_size) const noexcept
    {
        enum { M, I, D };
        int prev = M, truth_idx = first_pos, target_idx = 0, result = 0;
        const int rhs_begin = truth_len - rhs_flank_len;
        target_mask_size = 0;
        for (int a = 0; aln1[a]; ++a) {
            int st = M;
            if (aln1[a] == gap_label) st = I; else if (aln2[a] == gap_label) st = D;
            const bool in_flank = truth_idx < lhs_flank_len || truth_idx >= rhs_begin;
            if (st == M) {
                if (in_flank) {
                    if (aln1[a] != aln2[a]) {
                        if (aln1[a] != 'N') {
                            int q = quals[target_idx];
                            if (snv_mask[truth_idx] == target[target_idx] && snv_prior[truth_idx] < q) q = snv_prior[truth_idx];
                            result += q;
                        } else result += 2;
                    }
                    ++target_mask_size;
                }
                ++truth_idx; ++target_idx;
            } else if (st == I) {
                if (in_flank) { result += (prev == I ? get(gap_extend, truth_idx - 1) : gap_open[truth_idx - 1]) + nuc_prior; ++target_mask_size; }
                ++target_idx;
            } else {
                if (in_flank) result += prev == D ? get(gap_extend, truth_idx) : gap_open[truth_idx];
                ++truth_idx;
            }
            prev = st;
        }
        return result;
    }

private:
    Engine engine_;

    static int get(const std::int8_t* v, int i) noexcept { return v[i]; }
    template <typename T> static int get(T v, int) noexcept { return static_cast<int>(v); }
    static const std::int8_t* ext_ptr(const std::int8_t* p) noexcept { return p; }
    template <typename T> static const std::int8_t* ext_ptr(T) noexcept { return nullptr; }
    static int ext_scalar(const std::int8_t*) noexcept { return 0; }
    template <typename T> static int ext_scalar(T v) noexcept { return static_cast<int>(v); }

    template <typename GapExtend>
    int run(const char* truth, const char* target, const std::int8_t* quals, int truth_len, int target_len,
            const char* snv_mask, const std::int8_t* snv_prior, const std::int8_t* gap_open, GapExtend gap_extend, short nuc_prior,
            int& first_pos, char* align1, char* align2) const noexcept
    {
        int score = 0;
        std::vector<char> a1, a2;
        if (!align1) { a1.assign(2 * (target_len + BandSize) + 1, 0); a2 = a1; align1 = a1.data(); align2 = a2.data(); }
        const int rc = phmm_align_traceback(engine_.get(), BandSize, truth, target, quals, truth_len, target_len, snv_mask, snv_prior,
                                            gap_open, ext_ptr(gap_extend), ext_scalar(gap_extend), nuc_prior, &score, &first_pos, align1, align2);
        if (rc != PHMM_OK) first_pos = -1;   // the reference signals failure through first_pos (simd_pair_hmm.hpp:176-199)
        return score;
    }
};

// ---------------------------------------------------------------------------------------------------------------------
// Batch seam
// ---------------------------------------------------------------------------------------------------------------------
struct HaplotypeBlock   // what HaplotypeLikelihoodModel::reset derives per haplotype (haplotype_likelihood_model.cpp:60-78)
{
    pinned_vector<std::int64_t> off {0};
    pinned_vector<char> seq, snv_mask_fwd, snv_mask_rev;
    pinned_vector<std::int8_t> snv_prior_fwd, snv_prior_rev, gap_open, gap_extend;
    pinned_vector<std::int64_t> begin;
    pinned_vector<std::uint8_t> is_substitution;   // only used by reset(): bases that are substitutions in Haplotype::cigar()

    // Sequences only; reset(model) then fills the penalty arrays (the reference's likelihood_model_.reset(haplotype) per haplotype).
    void add(const std::string& sequence, std::int64_t mapped_begin = 0, const std::vector<bool>* substitutions = nullptr)
    {
        seq.insert(seq.end(), sequence.begin(), sequence.end());
        is_substitution.resize(seq.size(), 0);
        if (substitutions) for (std::size_t i = 0; i < substitutions->size() && i < sequence.size(); ++i) is_substitution[seq.size() - sequence.size() + i] = (*substitutions)[i] ? 1 : 0;
        begin.push_back(mapped_begin);
        off.push_back(static_cast<std::int64_t>(seq.size()));
    }
    void reset(const ErrorModel& model, int n_threads = 0)
    {
        const std::size_t n = seq.size();
        snv_mask_fwd.resize(n); snv_mask_rev.resize(n); snv_prior_fwd.resize(n); snv_prior_rev.resize(n); gap_open.resize(n); gap_extend.resize(n);
        is_substitution.resize(n, 0);
        const int rc = phmm_reset_haplotypes(model.get(), static_cast<std::int32_t>(size()), off.data(), seq.data(), is_substitution.data(),
                                             snv_mask_fwd.data(), snv_prior_fwd.data(), snv_mask_rev.data(), snv_prior_rev.data(),
                                             gap_open.data(), gap_extend.data(), n_threads);
        if (rc != PHMM_OK) throw Error {rc, phmm_error_model_last_error()};
    }

    void add(const std::string& sequence, const std::vector<char>& fwd_mask, const std::vector<std::int8_t>& fwd_priors,
             const std::vector<char>& rev_mask, const std::vector<std::int8_t>& rev_priors,
             const std::vector<std::int8_t>& open, const std::vector<std::int8_t>& extend, std::int64_t mapped_begin = 0)
    {
        seq.insert(seq.end(), sequence.begin(), sequence.end());
        snv_mask_fwd.insert(snv_mask_fwd.end(), fwd_mask.begin(), fwd_mask.end());
        snv_mask_rev.insert(snv_mask_rev.end(), rev_mask.begin(), rev_mask.end());
        snv_prior_fwd.insert(snv_prior_fwd.end(), fwd_priors.begin(), fwd_priors.end());
        snv_prior_rev.insert(snv_prior_rev.end(), rev_priors.begin(), rev_priors.end());
        gap_open.insert(gap_open.end(), open.begin(), open.end());
        gap_extend.insert(gap_extend.end(), extend.begin(), extend.end());
        begin.push_back(mapped_begin);
        off.push_back(static_cast<std::int64_t>(seq.size()));
    }
    void append(const HaplotypeBlock& other)   // the penalty arrays of both blocks must be filled
    {
        const auto base = static_cast<std::int64_t>(seq.size());
        seq.insert(seq.end(), other.seq.begin(), other.seq.end());
        snv_mask_fwd.insert(snv_mask_fwd.end(), other.snv_mask_fwd.begin(), other.snv_mask_fwd.end());
        snv_mask_rev.insert(snv_mask_rev.end(), other.snv_mask_rev.begin(), other.snv_mask_rev.end());
        snv_prior_fwd.insert(snv_prior_fwd.end(), other.snv_prior_fwd.begin(), other.snv_prior_fwd.end());
        snv_prior_rev.insert(snv_prior_rev.end(), other.snv_prior_rev.begin(), other.snv_prior_rev.end());
        gap_open.insert(gap_open.end(), other.gap_open.begin(), other.gap_open.end());
        gap_extend.insert(gap_extend.end(), other.gap_extend.begin(), other.gap_extend.end());
        begin.insert(begin.end(), other.begin.begin(), other.begin.end());
        for (std::size_t i = 1; i < other.off.size(); ++i) off.push_back(base + other.off[i]);
    }
    std::size_t size() const noexcept { return off.size() - 1; }
    phmm_haplotypes view() const noexcept
    {
        return phmm_haplotypes {static_cast<std::int32_t>(size()), off.data(), seq.data(), snv_mask_fwd.data(), snv_prior_fwd.data(),
                                snv_mask_rev.data(), snv_prior_rev.data(), gap_open.data(), gap_extend.data(), begin.data()};
    }
};

struct ReadBlock   // AlignedRead fields on the path (basics/aligned_read.hpp:36-39,120-146)
{
    pinned_vector<std::int64_t> off {0};
    pinned_vector<char> bases;
    pinned_vector<std::uint8_t> quals, mapq, reverse;
    pinned_vector<std::int64_t> begin;

    void add(const std::string& sequence, const std::vector<std::uint8_t>& base_qualities, std::uint8_t mapping_quality,
             bool is_marked_reverse_mapped, std::int64_t mapped_begin)
    {
        bases.insert(bases.end(), sequence.begin(), sequence.end());
        quals.insert(quals.end(), base_qualities.begin(), base_qualities.end());
        mapq.push_back(mapping_quality);
        reverse.push_back(is_marked_reverse_mapped ? 1 : 0);
        begin.push_back(mapped_begin);
        off.push_back(static_cast<std::int64_t>(bases.size()));
    }
    void append(const ReadBlock& other)
    {
        const auto base = static_cast<std::int64_t>(bases.size());
        bases.insert(bases.end(), other.bases.begin(), other.bases.end());
        quals.insert(quals.end(), other.quals.begin(), other.quals.end());
        mapq.insert(mapq.end(), other.mapq.begin(), other.mapq.end());
        reverse.insert(reverse.end(), other.reverse.begin(), other.reverse.end());
        begin.insert(begin.end(), other.begin.begin(), other.begin.end());
        for (std::size_t i = 1; i < other.off.size(); ++i) off.push_back(base + other.off[i]);
    }
    std::size_t size() const noexcept { return off.size() - 1; }
    phmm_reads view() const noexcept
    {
        return phmm_reads {static_cast<std::int32_t>(size()), off.data(), bases.data(), quals.data(), mapq.data(), reverse.data(), begin.data()};
    }
};

struct TemplateBlock   // AlignedTemplate containers: template t owns the reads [off[t], off[t+1]) (basics/aligned_template.hpp)
{
    ReadBlock reads;
    pinned_vector<std::int64_t> off {0};
    void add(const ReadBlock& template_reads) { reads.append(template_reads); off.push_back(static_cast<std::int64_t>(reads.size())); }
    std::size_t size() const noexcept { return off.size() - 1; }
};

struct FlankState { std::int64_t lhs_flank, rhs_flank; };   // HaplotypeLikelihoodModel::FlankState

using SampleName = std::string;

// A read-only view of one likelihoods_[haplotype][sample] vector (the reference returns const std::vector<double>&).
struct LikelihoodSpan
{
    const double* first = nullptr;
    std::size_t count = 0;
    const double* begin() const noexcept { return first; }
    const double* end() const noexcept { return first + count; }
    std::size_t size() const noexcept { return count; }
    bool empty() const noexcept { return count == 0; }
    double operator[](std::size_t i) const noexcept { return first[i]; }
    operator std::vector<double>() const { return std::vector<double>(first, first + count); }
};

// HaplotypeLikelihoodArray (haplotype_likelihood_array.hpp:34-175): likelihoods_[haplotype][sample][read or template].
// All samples of a populate() go to the GPU as ONE batch (their reads are concatenated; one phmm_populate call fills one
// [H][R_total] matrix), a sample is a column range of that matrix.
class HaplotypeLikelihoodArray
{
public:
    using LogProbability = double;
    using LikelihoodVector = std::vector<LogProbability>;
    using ReadMap = std::vector<std::pair<SampleName, ReadBlock>>;                 // config/common.hpp:33-37, in sample order
    using TemplateMap = std::vector<std::pair<SampleName, TemplateBlock>>;

    explicit HaplotypeLikelihoodArray(phmm_config config, Engine engine = Engine {}) : engine_ {std::move(engine)}, config_ {config}
    {
        if (config.max_indel_error > 256) throw TooLargeBandSizeError {static_cast<unsigned>(config.max_indel_error)};
    }
    static phmm_config default_config() noexcept { phmm_config c; phmm_default_config(&c); return c; }

    // populate(const ReadMap&, haplotypes, flank_state) — haplotype_likelihood_array.cpp:51-103.
    // positions: optional candidate mapping positions (CSR over [H][R_total]); without them the device k-mer mapper runs
    // (config.map_positions), as the reference maps inline (:89-92).
    void populate(const ReadMap& reads, const HaplotypeBlock& haplotypes, const FlankState* flank_state = nullptr,
                  const phmm_positions* positions = nullptr)
    {
        ReadBlock all;
        begin_samples(reads.size());
        for (const auto& p : reads) { add_sample(p.first, p.second.size()); all.append(p.second); }
        run(all, nullptr, haplotypes, flank_state, positions);
    }
    // single unnamed sample, primed (what the reference's single-sample callers see after prime())
    void populate(const ReadBlock& reads, const HaplotypeBlock& haplotypes, const FlankState* flank_state = nullptr,
                  const phmm_positions* positions = nullptr)
    {
        begin_samples(1);
        add_sample(SampleName {}, reads.size());
        run(reads, nullptr, haplotypes, flank_state, positions);
        primed_ = 0;
    }
    // populate(const TemplateMap&, ...) — haplotype_likelihood_array.cpp:105-199: one value per (haplotype, template)
    void populate(const TemplateMap& templates, const HaplotypeBlock& haplotypes, const FlankState* flank_state = nullptr)
    {
        ReadBlock all;
        pinned_vector<std::int64_t> template_off {0};
        begin_samples(templates.size());
        for (const auto& p : templates) {
            add_sample(p.first, p.second.size());
            const auto base = static_cast<std::int64_t>(all.size());
            all.append(p.second.reads);
            for (std::size_t t = 1; t < p.second.off.size(); ++t) template_off.push_back(base + p.second.off[t]);
        }
        run(all, &template_off, haplotypes, flank_state, nullptr);
    }

    // accessors (haplotype_likelihood_array.cpp:200-291)
    std::size_t num_likelihoods(const SampleName& sample) const { return width(sample_index(sample)); }
    std::size_t num_likelihoods() const { return width(primed()); }
    LikelihoodSpan operator()(const SampleName& sample, std::size_t haplotype_index) const { return span(haplotype_index, sample_index(sample)); }
    LikelihoodSpan operator[](std::size_t haplotype_index) const { return span(haplotype_index, primed()); }
    const std::vector<SampleName>& samples() const noexcept { return samples_; }
    std::size_t num_haplotypes() const noexcept { return num_haplotypes_; }
    std::vector<LikelihoodVector> extract_sample(const SampleName& sample) const
    {
        const auto s = sample_index(sample);
        std::vector<LikelihoodVector> result;
        for (std::size_t h = 0; h < num_haplotypes_; ++h) result.push_back(span(h, s));
        return result;
    }
    bool is_empty() const noexcept { return likelihoods_.empty(); }
    void clear() noexcept { likelihoods_.clear(); samples_.clear(); sample_off_.assign(1, 0); num_haplotypes_ = 0; unprime(); }
    bool is_primed() const noexcept { return primed_ >= 0; }
    void prime(const SampleName& sample) const { primed_ = static_cast<std::ptrdiff_t>(sample_index(sample)); }
    void unprime() const noexcept { primed_ = -1; }

    // reset(haplotypes) (:331-360): keep a subset of the haplotypes — here by their (ascending) old indices
    void reset(const std::vector<std::size_t>& haplotypes_to_keep)
    {
        if (haplotypes_to_keep.empty()) { clear(); return; }
        const std::size_t w = total_width();
        std::size_t dst = 0, prev = 0;
        for (const std::size_t h : haplotypes_to_keep) {
            if (h >= num_haplotypes_ || (dst > 0 && h <= prev)) throw std::invalid_argument {"reset: haplotype indices must be ascending and in range"};
            if (h != dst) std::copy_n(likelihoods_.begin() + static_cast<std::ptrdiff_t>(h * w), w, likelihoods_.begin() + static_cast<std::ptrdiff_t>(dst * w));
            prev = h; ++dst;
        }
        num_haplotypes_ = dst;
        likelihoods_.resize(dst * w);
    }
    // merge_samples (:362-409): one sample holding the chosen samples' likelihoods back to back; the result is primed
    HaplotypeLikelihoodArray merge_samples(const std::vector<SampleName>& samples, const SampleName* new_sample = nullptr) const
    {
        SampleName name;
        if (new_sample) name = *new_sample; else for (const auto& s : samples) name += s;
        HaplotypeLikelihoodArray result {config_, engine_};
        std::vector<std::size_t> idx;
        std::size_t total = 0;
        for (const auto& s : samples) { idx.push_back(sample_index(s)); total += width(idx.back()); }
        result.begin_samples(1);
        result.add_sample(name, total);
        result.num_haplotypes_ = num_haplotypes_;
        result.likelihoods_.resize(num_haplotypes_ * total);
        auto dst = result.likelihoods_.begin();
        for (std::size_t h = 0; h < num_haplotypes_; ++h) {
            for (const std::size_t s : idx) { const auto src = span(h, s); dst = std::copy(src.begin(), src.end(), dst); }
        }
        result.primed_ = 0;
        return result;
    }
    HaplotypeLikelihoodArray merge_samples(const SampleName* new_sample = nullptr) const { return merge_samples(samples_, new_sample); }

    const double* data() const noexcept { return likelihoods_.data(); }   // [haplotype][all samples' columns], row-major

private:
    friend class RegionBatch;   // fills arrays from the result of one many-regions call (fill_from)

    Engine engine_;
    phmm_config config_;
    pinned_vector<double> likelihoods_;
    pinned_vector<std::int32_t> status_;
    std::vector<SampleName> samples_;
    std::vector<std::size_t> sample_off_ {0};
    std::size_t num_haplotypes_ = 0;
    mutable std::ptrdiff_t primed_ = -1;

    // samples_ / sample_off_ already set: the [num_haplotypes][total width] values, row-major
    void fill_from(std::size_t num_haplotypes, const double* values)
    {
        num_haplotypes_ = num_haplotypes;
        likelihoods_.assign(values, values + num_haplotypes * total_width());
    }
    void begin_samples(std::size_t n) { samples_.clear(); samples_.reserve(n); sample_off_.assign(1, 0); unprime(); }
    void add_sample(const SampleName& name, std::size_t n) { samples_.push_back(name); sample_off_.push_back(sample_off_.back() + n); }
    std::size_t total_width() const noexcept { return sample_off_.back(); }
    std::size_t width(std::size_t s) const noexcept { return sample_off_[s + 1] - sample_off_[s]; }
    std::size_t sample_index(const SampleName& sample) const
    {
        for (std::size_t s = 0; s < samples_.size(); ++s) if (samples_[s] == sample) return s;
        throw std::out_of_range {"HaplotypeLikelihoodArray: unknown sample " + sample};   // the reference's unordered_map::at
    }
    std::size_t primed() const
    {
        if (primed_ < 0) throw std::logic_error {"HaplotypeLikelihoodArray: not primed"};   // an assert in the reference
        return static_cast<std::size_t>(primed_);
    }
    LikelihoodSpan span(std::size_t h, std::size_t s) const
    {
        if (h >= num_haplotypes_) throw std::out_of_range {"HaplotypeLikelihoodArray: haplotype index"};
        return LikelihoodSpan {likelihoods_.data() + h * total_width() + sample_off_[s], width(s)};
    }
    void run(const ReadBlock& reads, const pinned_vector<std::int64_t>* template_off, const HaplotypeBlock& haplotypes,
             const FlankState* flank_state, const phmm_positions* positions)
    {
        const auto hv = haplotypes.view();
        const auto rv = reads.view();
        num_haplotypes_ = haplotypes.size();
        likelihoods_.resize(num_haplotypes_ * total_width());        // every element is written by the call (no zero fill; the storage is page-locked and kept)
        if (num_haplotypes_ == 0 || reads.size() == 0) return;
        pinned_vector<std::int32_t>& status = status_;               // page-locked scratch kept across calls: allocating pinned memory costs milliseconds
        status.resize(num_haplotypes_ * reads.size());
        phmm_flank_state fs {flank_state ? 1 : 0, flank_state ? flank_state->lhs_flank : 0, flank_state ? flank_state->rhs_flank : 0};
        const int rc = template_off
            ? phmm_populate_templates(engine_.get(), &config_, &hv, &rv, template_off->data(), static_cast<std::int32_t>(template_off->size() - 1),
                                      positions, &fs, likelihoods_.data(), status.data(), PHMM_SPACE_HOST)
            : phmm_populate(engine_.get(), &config_, &hv, &rv, positions, &fs, likelihoods_.data(), status.data(), PHMM_SPACE_HOST);
        if (rc == PHMM_ERR_SHORT_HAPLOTYPE) {
            for (std::size_t i = 0; i < status.size(); ++i) {
                if ((status[i] & 0xFFFF) == PHMM_STATUS_SHORT_HAP) throw ShortHaplotypeError {i / reads.size(), static_cast<unsigned>(static_cast<std::uint32_t>(status[i]) >> 16)};
            }
        }
        engine_.check(rc);
    }
};

// Many independent regions in ONE engine call (phmm_populate_regions_ex): a batch front end for a caller that has several regions
// ready at once (Octopus's region tasks). Each region is what one HaplotypeLikelihoodArray::populate call takes — a ReadMap or a
// TemplateMap (the two kinds may be mixed: a ReadMap region then rides along as one-read templates, whose sums are the reads' values
// exactly), its haplotypes (penalty arrays filled) and an optional flank state. run() yields one array per region, in the order added,
// with the samples, widths and values populate() gives for that region alone. A region with a short haplotype is reported in its
// result (as ShortHaplotypeError would report it) and the other regions are filled all the same.
class RegionBatch
{
public:
    using ReadMap = HaplotypeLikelihoodArray::ReadMap;
    using TemplateMap = HaplotypeLikelihoodArray::TemplateMap;

    struct Result
    {
        HaplotypeLikelihoodArray likelihoods;
        bool short_haplotype = false;           // populate() would have thrown ShortHaplotypeError {haplotype_index, required_extension}
        std::size_t haplotype_index = 0;
        unsigned required_extension = 0;
        void check() const { if (short_haplotype) throw ShortHaplotypeError {haplotype_index, required_extension}; }
    };

    explicit RegionBatch(phmm_config config, Engine engine = Engine {}) : config_ {config}, engine_ {std::move(engine)}
    {
        if (config.max_indel_error > 256) throw TooLargeBandSizeError {static_cast<unsigned>(config.max_indel_error)};
    }

    // Each add() copies the region into the batch's page-locked blocks and returns its index.
    std::size_t add(const ReadMap& reads, const HaplotypeBlock& haplotypes, const FlankState* flank_state = nullptr)
    {
        std::size_t n_reads = 0;
        for (const auto& p : reads) n_reads += p.second.size();
        Region g = begin_region(haplotypes, n_reads, flank_state, false);
        for (const auto& p : reads) {
            g.samples.push_back(p.first); g.widths.push_back(p.second.size());
            if (g.in_call()) reads_.append(p.second);
        }
        regions_.push_back(std::move(g));
        return regions_.size() - 1;
    }
    std::size_t add(const TemplateMap& templates, const HaplotypeBlock& haplotypes, const FlankState* flank_state = nullptr)
    {
        for (const auto& p : templates) {
            const TemplateBlock& tb = p.second;
            if (tb.off.empty() || tb.off.front() != 0 || static_cast<std::size_t>(tb.off.back()) != tb.reads.size() ||
                !std::is_sorted(tb.off.begin(), tb.off.end())) throw std::invalid_argument {"RegionBatch: template offsets must cover the sample's reads"};
        }
        std::size_t n_reads = 0;
        for (const auto& p : templates) n_reads += p.second.reads.size();
        Region g = begin_region(haplotypes, n_reads, flank_state, true);
        for (const auto& p : templates) {
            g.samples.push_back(p.first); g.widths.push_back(p.second.size());
            if (!g.in_call()) continue;
            const auto base = static_cast<std::int64_t>(reads_.size() - g.read0);
            for (std::size_t t = 1; t < p.second.off.size(); ++t) g.template_off.push_back(base + p.second.off[t]);
            reads_.append(p.second.reads);
        }
        regions_.push_back(std::move(g));
        return regions_.size() - 1;
    }
    std::size_t size() const noexcept { return regions_.size(); }
    void clear() { regions_.clear(); haps_ = HaplotypeBlock {}; reads_ = ReadBlock {}; }

    std::vector<Result> run()
    {
        std::vector<Result> results;
        results.reserve(regions_.size());
        bool any_templates = false;
        std::vector<std::int32_t> hap_first {0}, read_first {0}, template_first {0};
        std::vector<phmm_flank_state> flanks;
        pinned_vector<std::int64_t> template_off {0};
        std::size_t n_out = 0, n_status = 0;
        for (const Region& g : regions_) any_templates = any_templates || g.templated;
        for (const Region& g : regions_) {
            if (!g.in_call()) continue;
            hap_first.push_back(static_cast<std::int32_t>(g.hap0 + g.n_haps));
            read_first.push_back(static_cast<std::int32_t>(g.read0 + g.n_reads));
            flanks.push_back(g.flank);
            if (any_templates) {
                const std::size_t base = g.read0;
                if (g.templated) for (std::size_t t = 1; t < g.template_off.size(); ++t) template_off.push_back(static_cast<std::int64_t>(base) + g.template_off[t]);
                else for (std::size_t r = 1; r <= g.n_reads; ++r) template_off.push_back(static_cast<std::int64_t>(base + r));
                template_first.push_back(static_cast<std::int32_t>(template_off.size() - 1));
            }
            n_out += g.n_haps * g.width();
            n_status += g.n_haps * g.n_reads;
        }
        int rc = PHMM_OK;
        if (flanks.size()) {
            out_.resize(n_out);
            status_.resize(n_status);
            const auto hv = haps_.view();
            const auto rv = reads_.view();
            const phmm_regions regions {static_cast<std::int32_t>(flanks.size()), hap_first.data(), read_first.data(), flanks.data()};
            const phmm_region_templates templates {template_first.data(), template_off.data()};
            rc = phmm_populate_regions_ex(engine_.get(), &config_, &hv, &rv, &regions, any_templates ? &templates : nullptr, nullptr,
                                          out_.data(), status_.data(), PHMM_SPACE_HOST);
            if (rc != PHMM_ERR_SHORT_HAPLOTYPE) engine_.check(rc);
        }
        std::size_t out_at = 0, status_at = 0;
        for (const Region& g : regions_) {
            Result res {HaplotypeLikelihoodArray {config_, engine_}};
            HaplotypeLikelihoodArray& a = res.likelihoods;
            a.begin_samples(g.samples.size());
            for (std::size_t s = 0; s < g.samples.size(); ++s) a.add_sample(g.samples[s], g.widths[s]);
            if (!g.in_call()) {
                const std::vector<double> zeros(g.n_haps * g.width(), 0.0);   // no reads: every template sums to 0
                a.fill_from(g.n_haps, zeros.data());
            } else {
                a.fill_from(g.n_haps, out_.data() + out_at);
                if (rc == PHMM_ERR_SHORT_HAPLOTYPE) {
                    for (std::size_t i = 0; i < g.n_haps * g.n_reads; ++i) {
                        const std::int32_t st = status_[status_at + i];
                        if ((st & 0xFFFF) == PHMM_STATUS_SHORT_HAP) {
                            res.short_haplotype = true;
                            res.haplotype_index = i / g.n_reads;
                            res.required_extension = static_cast<unsigned>(static_cast<std::uint32_t>(st) >> 16);
                            break;
                        }
                    }
                }
                out_at += g.n_haps * g.width();
                status_at += g.n_haps * g.n_reads;
            }
            results.push_back(std::move(res));
        }
        return results;
    }

private:
    struct Region
    {
        std::vector<SampleName> samples;
        std::vector<std::size_t> widths;
        std::size_t hap0 = 0, n_haps = 0, read0 = 0, n_reads = 0;
        bool templated = false;
        phmm_flank_state flank {0, 0, 0};
        std::vector<std::int64_t> template_off {0};   // over the region's reads
        std::size_t width() const { std::size_t w = 0; for (const std::size_t x : widths) w += x; return w; }
        bool in_call() const { return n_haps > 0 && n_reads > 0; }
    };
    phmm_config config_;
    Engine engine_;
    HaplotypeBlock haps_;
    ReadBlock reads_;
    std::vector<Region> regions_;
    pinned_vector<double> out_;            // page-locked result buffers kept across runs
    pinned_vector<std::int32_t> status_;

    // a region without haplotypes or reads stays out of the call and out of the blocks (run() fills its array)
    Region begin_region(const HaplotypeBlock& haplotypes, std::size_t n_reads, const FlankState* flank_state, bool templated)
    {
        Region g;
        g.templated = templated;
        if (flank_state) g.flank = phmm_flank_state {1, flank_state->lhs_flank, flank_state->rhs_flank};
        g.hap0 = haps_.size(); g.n_haps = haplotypes.size();
        g.read0 = reads_.size(); g.n_reads = n_reads;
        if (g.in_call()) haps_.append(haplotypes);
        return g;
    }
};

// ---------------------------------------------------------------------------------------------------------------------
// hmm::PairHMM<Parameters, BandSize, Score> (src/core/models/pairhmm/pair_hmm.hpp:892-1032) over the GPU kernel
// ---------------------------------------------------------------------------------------------------------------------
// The reference's class bundles a kernel object with a `const Parameters*` and forwards to the free templates hmm::evaluate /
// hmm::align. Those templates are the reference's own code, so this type exists only where its header has been included before
// this one (Octopus's build; tests/cpp/test_dropin.cpp): it differs from octopus::hmm::PairHMM in the kernel member alone.
// The kernel is GpuPairHMM with a RUNTIME band, like simd::PairHMMWrapper (simd_pair_hmm_wrapper.hpp:218-241: smallest of
// 8, 16, ..., 256 that holds the request; TooLargeBandSizeError beyond).
class GpuPairHMMDyn
{
public:
    using ScoreType = int;
    constexpr static char gap_label = '-';
    GpuPairHMMDyn() = default;
    explicit GpuPairHMMDyn(unsigned min_band_size, Engine engine = Engine {}) : engine_ {std::move(engine)} { reset(min_band_size); }
    void reset(unsigned min_band_size)
    {
        for (int b = 8; b <= 256; b <<= 1) if (min_band_size <= static_cast<unsigned>(b)) { band_ = b; return; }
        throw TooLargeBandSizeError {min_band_size};
    }
    constexpr static const char* name() noexcept { return "B200"; }
    int band_size() const noexcept { return band_; }
    template <typename GapExtend>
    int align(const char* truth, const char* target, const std::int8_t* qualities, int truth_len, int target_len,
              const std::int8_t* gap_open, GapExtend gap_extend, short nuc_prior) const noexcept
    { int fp; return run(truth, target, qualities, truth_len, target_len, nullptr, nullptr, gap_open, gap_extend, nuc_prior, fp, nullptr, nullptr); }
    template <typename GapExtend>
    int align(const char* truth, const char* target, const std::int8_t* qualities, int truth_len, int target_len,
              const char* snv_mask, const std::int8_t* snv_prior, const std::int8_t* gap_open, GapExtend gap_extend, short nuc_prior) const noexcept
    { int fp; return run(truth, target, qualities, truth_len, target_len, snv_mask, snv_prior, gap_open, gap_extend, nuc_prior, fp, nullptr, nullptr); }
    template <typename GapExtend>
    int align(const char* truth, const char* target, const std::int8_t* qualities, int truth_len, int target_len,
              const std::int8_t* gap_open, GapExtend gap_extend, short nuc_prior, int& first_pos, char* align1, char* align2) const noexcept
    { return run(truth, target, qualities, truth_len, target_len, nullptr, nullptr, gap_open, gap_extend, nuc_prior, first_pos, align1, align2); }
    template <typename GapExtend>
    int align(const char* truth, const char* target, const std::int8_t* qualities, int truth_len, int target_len,
              const char* snv_mask, const std::int8_t* snv_prior, const std::int8_t* gap_open, GapExtend gap_extend, short nuc_prior,
              int& first_pos, char* align1, char* align2) const noexcept
    { return run(truth, target, qualities, truth_len, target_len, snv_mask, snv_prior, gap_open, gap_extend, nuc_prior, first_pos, align1, align2); }
    template <typename... Args>
    int calculate_flank_score(Args&&... args) const noexcept { return GpuPairHMM<8> {engine_}.calculate_flank_score(std::forward<Args>(args)...); }   // band-independent replay
private:
    Engine engine_;
    int band_ = 8;
    static const std::int8_t* ext_ptr(const std::int8_t* p) noexcept { return p; }
    template <typename T> static const std::int8_t* ext_ptr(T) noexcept { return nullptr; }
    static int ext_scalar(const std::int8_t*) noexcept { return 0; }
    template <typename T> static int ext_scalar(T v) noexcept { return static_cast<int>(v); }
    template <typename GapExtend>
    int run(const char* truth, const char* target, const std::int8_t* quals, int truth_len, int target_len,
            const char* snv_mask, const std::int8_t* snv_prior, const std::int8_t* gap_open, GapExtend gap_extend, short nuc_prior,
            int& first_pos, char* align1, char* align2) const noexcept
    {
        int score = 0;
        std::vector<char> a1, a2;
        if (!align1) { a1.assign(2 * (target_len + band_) + 1, 0); a2 = a1; align1 = a1.data(); align2 = a2.data(); }
        const int rc = phmm_align_traceback(engine_.get(), band_, truth, target, quals, truth_len, target_len, snv_mask, snv_prior,
                                            gap_open, ext_ptr(gap_extend), ext_scalar(gap_extend), nuc_prior, &score, &first_pos, align1, align2);
        if (rc != PHMM_OK) first_pos = -1;
        return score;
    }
};

#ifdef pair_hmm_hpp   // the include guard of the reference's src/core/models/pairhmm/pair_hmm.hpp
template <typename Parameters, int BandSize = 0>
class PairHMM
{
public:
    using ParameterType = Parameters;
    PairHMM() = default;
    explicit PairHMM(unsigned min_band_size) { reset(min_band_size); }
    PairHMM(const Parameters& params, unsigned min_band_size = 8) { reset(min_band_size); set(params); }
    int band_size() const noexcept { return hmm_.band_size(); }
    void set(const Parameters& params) noexcept { params_ = std::addressof(params); }
    template <typename Sequence1, typename Sequence2>
    double evaluate(const Sequence1& target, const Sequence2& truth, const std::vector<std::uint8_t>& target_base_qualities, const std::size_t target_offset) const noexcept
    { return octopus::hmm::evaluate(truth, target, target_base_qualities, target_offset, hmm_, *params_); }
    template <typename Sequence1, typename Sequence2>
    void align(const Sequence1& target, const Sequence2& truth, const std::vector<std::uint8_t>& target_base_qualities, const std::size_t target_offset,
               octopus::hmm::Alignment& result) const
    { octopus::hmm::align(truth, target, target_base_qualities, target_offset, hmm_, *params_, result); }
    template <typename Sequence1, typename Sequence2>
    octopus::hmm::Alignment align(const Sequence1& target, const Sequence2& truth, const std::vector<std::uint8_t>& target_base_qualities, const std::size_t target_offset) const
    { octopus::hmm::Alignment result {}; this->align(target, truth, target_base_qualities, target_offset, result); return result; }
private:
    GpuPairHMMDyn hmm_ {BandSize > 0 ? static_cast<unsigned>(BandSize) : 8u};
    const Parameters* params_ = nullptr;
    void reset(unsigned min_band_size) { if (BandSize == 0) hmm_.reset(min_band_size); }
};
#endif

} // namespace octopus_b200

#endif
