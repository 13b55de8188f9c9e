// The C++ adapter's many-regions front end (RegionBatch): built by tests/test_gpu_region_templates.py with g++ -std=c++14 and run on
// the GPU. Every region of a batch must come back with exactly what HaplotypeLikelihoodArray::populate gives for that region alone:
// the same samples, widths and bytes, or the same ShortHaplotypeError. Prints "REGIONS ..." and exits 0 when all of them agree.
#include <cstdio>
#include <cstring>
#include <random>
#include <string>
#include <vector>
#include "phmm_b200.hpp"

using namespace octopus_b200;

namespace {

std::mt19937_64 rng {20261017};
int uniform(int lo, int hi) { return std::uniform_int_distribution<int> {lo, hi}(rng); }   // [lo, hi]

struct Region
{
    HaplotypeBlock haps;
    std::vector<std::pair<std::string, TemplateBlock>> samples;   // as templates; the ReadMap form uses the same reads
    bool flank = false;
    FlankState fs {0, 0};
};

ReadBlock one_read(const std::string& hap, int L, int band)
{
    const int p = uniform(band, (int)hap.size() - L - band);
    std::string s = hap.substr((std::size_t)p, (std::size_t)L);
    if (uniform(0, 2) == 0) s[(std::size_t)uniform(0, L - 1)] = "ACGT"[uniform(0, 3)];
    std::vector<std::uint8_t> q((std::size_t)L);
    for (auto& x : q) x = (std::uint8_t)uniform(20, 40);
    ReadBlock r;
    r.add(s, q, (std::uint8_t)uniform(20, 60), uniform(0, 1) == 1, p);
    return r;
}

Region make_region(const ErrorModel& model, int n_haps, int n_samples, int band, int hap_len = 300, bool short_hap = false)
{
    Region g;
    std::string base((std::size_t)hap_len, 'A');
    for (auto& c : base) c = "ACGT"[uniform(0, 3)];
    for (int h = 0; h < n_haps; ++h) {
        std::string s = base;
        for (int k = 0; k < 3; ++k) s[(std::size_t)uniform(0, hap_len - 1)] = "ACGT"[uniform(0, 3)];
        g.haps.add(s);
    }
    g.haps.reset(model);
    for (int smp = 0; smp < n_samples; ++smp) {
        TemplateBlock tb;
        const int n_templates = uniform(1, 25);
        for (int t = 0; t < n_templates; ++t) {
            ReadBlock members;
            for (int k = uniform(1, 3); k > 0; --k) {
                const std::string hap(g.haps.seq.begin() + g.haps.off[0], g.haps.seq.begin() + g.haps.off[1]);
                members.append(short_hap ? [&] { ReadBlock r; r.add(hap.substr(5, 50), std::vector<std::uint8_t>(50, 30), 60, false, 5); return r; }()
                                         : one_read(hap, uniform(0, 1) ? 100 : 76, band));
            }
            tb.add(members);
        }
        g.samples.emplace_back("S" + std::to_string(smp), std::move(tb));
    }
    if (uniform(0, 1)) { g.flank = true; g.fs = FlankState {uniform(0, 60), uniform(0, 60)}; }
    return g;
}

HaplotypeLikelihoodArray::ReadMap read_map(const Region& g)
{
    HaplotypeLikelihoodArray::ReadMap m;
    for (const auto& s : g.samples) m.emplace_back(s.first, s.second.reads);
    return m;
}

struct Expected { bool is_short = false; std::size_t hap = 0; unsigned ext = 0; HaplotypeLikelihoodArray array; };

Expected alone(const phmm_config& cfg, const Engine& engine, const Region& g, bool templates)
{
    Expected x {false, 0, 0, HaplotypeLikelihoodArray {cfg, engine}};
    try {
        if (templates) x.array.populate(HaplotypeLikelihoodArray::TemplateMap(g.samples.begin(), g.samples.end()), g.haps, g.flank ? &g.fs : nullptr);
        else x.array.populate(read_map(g), g.haps, g.flank ? &g.fs : nullptr);
    } catch (const ShortHaplotypeError& e) {
        x.is_short = true; x.hap = e.haplotype_index(); x.ext = e.required_extension();
    }
    return x;
}

bool same(const RegionBatch::Result& got, const Expected& want, const char* what, std::size_t g)
{
    if (got.short_haplotype != want.is_short || (want.is_short && (got.haplotype_index != want.hap || got.required_extension != want.ext))) {
        std::printf("MISMATCH %s region %zu: short haplotype %d/%d\n", what, g, (int)got.short_haplotype, (int)want.is_short);
        return false;
    }
    if (want.is_short) return true;
    const auto& a = got.likelihoods;
    const auto& b = want.array;
    if (a.samples() != b.samples() || a.num_haplotypes() != b.num_haplotypes()) { std::printf("MISMATCH %s region %zu: shape\n", what, g); return false; }
    std::size_t width = 0;
    for (const auto& s : b.samples()) {
        if (a.num_likelihoods(s) != b.num_likelihoods(s)) { std::printf("MISMATCH %s region %zu: width of %s\n", what, g, s.c_str()); return false; }
        width += b.num_likelihoods(s);
    }
    if (std::memcmp(a.data(), b.data(), a.num_haplotypes() * width * sizeof(double)) != 0) { std::printf("MISMATCH %s region %zu: values\n", what, g); return false; }
    return true;
}

}  // namespace

int main()
{
    try {
        Engine engine;
        ErrorModel model;
        bool ok = true;
        int n_short = 0;
        for (const int band : {8, 16}) {
            auto cfg = HaplotypeLikelihoodArray::default_config();
            cfg.max_indel_error = band;
            std::vector<Region> regions;
            regions.push_back(make_region(model, 5, 2, band));              // two samples
            regions.push_back(make_region(model, 1, 1, band));
            regions.push_back(make_region(model, 12, 1, band));
            regions.push_back(make_region(model, 3, 1, band, 60, true));     // ShortHaplotypeError
            regions.push_back(make_region(model, 7, 3, band));
            for (const int mode : {0, 1, 2}) {                              // TemplateMap batch, ReadMap batch, mixed batch
                RegionBatch batch {cfg, engine};
                std::vector<Expected> want;
                for (std::size_t g = 0; g < regions.size(); ++g) {
                    const bool templates = mode == 0 || (mode == 2 && g % 2 == 0);
                    if (templates) batch.add(HaplotypeLikelihoodArray::TemplateMap(regions[g].samples.begin(), regions[g].samples.end()), regions[g].haps,
                                             regions[g].flank ? &regions[g].fs : nullptr);
                    else batch.add(read_map(regions[g]), regions[g].haps, regions[g].flank ? &regions[g].fs : nullptr);
                    want.push_back(alone(cfg, engine, regions[g], templates));
                }
                const auto got = batch.run();
                const char* what = mode == 0 ? "templates" : mode == 1 ? "reads" : "mixed";
                for (std::size_t g = 0; g < regions.size(); ++g) {
                    ok = same(got[g], want[g], what, g) && ok;
                    n_short += got[g].short_haplotype ? 1 : 0;
                }
            }
        }
        if (!ok) return 1;
        std::printf("REGIONS ok short_regions=%d\n", n_short);
        return 0;
    } catch (const std::exception& e) {
        std::printf("ERROR %s\n", e.what());
        return 2;
    }
}
