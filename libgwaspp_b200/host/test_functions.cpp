#include "test_functions.h"

#include <cassert>
#include <cstdio>
#include <iostream>
#include <time.h>

namespace libgwaspp {
namespace genetics {

GeneticData::GeneticData(int m, int n, int device)
    : n_markers(m), n_individs(n), geno_tbl(new DeviceGenoTable(m, n, device)), ccs(new CaseControlSet(n)) {}
GeneticData::GeneticData(const std::string &tped_path, int device)
    : n_markers(0), n_individs(0), geno_tbl(new DeviceGenoTable(tped_path, device)), ccs(nullptr) {
    n_markers = geno_tbl->row_size();
    n_individs = geno_tbl->column_size();
    ccs = new CaseControlSet(n_individs);
}
GeneticData::~GeneticData() { delete geno_tbl; delete ccs; }

void GeneticData::setCaseControlSet(const std::set<int> &cases, const std::set<int> &controls) {
    ccs->reset();
    std::set<int> co(controls);
    for (int c : cases)                      // an index in both sets stays a case (genetic_data.cpp:149-154)
        if (co.erase(c)) std::cout << "Index: " << c << " found in both Case/Controls; Removing from controls" << std::endl;
    ccs->setCases(cases);
    ccs->setControls(co);
}

}  // namespace genetics

namespace algorithms {

namespace {
struct Lap {
    timespec t0;
    Lap() { clock_gettime(CLOCK_MONOTONIC, &t0); }
    double seconds() const { timespec t1; clock_gettime(CLOCK_MONOTONIC, &t1); return (t1.tv_sec - t0.tv_sec) + 1e-9 * (t1.tv_nsec - t0.tv_nsec); }
};
// "%lu.%09lus" as PRINT_LAPSE does with NANO_TIME (src/util/time/timing.h:45-52,100-106)
void print_lapse(std::ostream &out, const char *prefix, double s) {
    char buf[64];
    unsigned long sec = (unsigned long)s, ns = (unsigned long)((s - (double)sec) * 1e9);
    snprintf(buf, sizeof buf, "%lu.%09lus", sec, ns);
    out << prefix << buf;
}
}  // namespace

void compute(void (*f)(GeneticData *, std::ostream *), GeneticData *gd, std::ostream *out) {
    Lap lap;
    if (out == NULL) out = &std::cout;
    f(gd, out);
    print_lapse(std::cout, "Total runtime: ", lap.seconds());
    std::cout << std::endl;
}

void compute_maf_perform(GeneticData *gd, std::ostream *) {
    const int M = gd->getGenotypedMarkersCount();
    DeviceGenoTable &gt = *gd->getGenotypeTable();
    std::vector<uint> c((size_t)M * 4);
    int rc = gwasdev_counts(gt.handle(), 0, (uint64_t)M, 0, c.data());
    assert(rc == GWASDEV_OK); (void)rc;
    double tot, maf;
    for (int i = 0; i < M; ++i) { frequency_table ft; memcpy(ft.freq, &c[4 * (size_t)i], 16); MinorAlleleFrequency(ft, tot, maf); }
}

void select_cc_maf(GeneticData *gd, std::ostream *out) {
    const int M = gd->getGenotypedMarkersCount();
    DeviceGenoTable &gt = *gd->getGenotypeTable();
    Lap sel;
    gt.selectCaseControl(*gd->getCaseControlSet());
    *out << (int)-1;
    print_lapse(*out, "\t", sel.seconds());
    *out << std::endl;
    Lap scan;
    std::vector<frequency_table> ca, co;
    gt.scanCaseControl(ca, co);
    const double per = scan.seconds() / (M > 0 ? M : 1);      // one batched scan: report its per-SNP share
    double tot, maf;
    for (int i = 0; i < M; ++i) {
        *out << (int)i;
        print_lapse(*out, "\t", per);
        *out << std::endl;
        MinorAlleleFrequency(ca[i], tot, maf);
        MinorAlleleFrequency(co[i], tot, maf);
    }
}

void inline_cc_maf(GeneticData *gd, std::ostream *out) {
    const int M = gd->getGenotypedMarkersCount();
    DeviceGenoTable &gt = *gd->getGenotypeTable();
    CaseControlSet &ccs = *gd->getCaseControlSet();
    Lap scan;
    CaseControlGenotypeDistribution first;
    if (M > 0) gt.getCaseControlGenotypeDistribution(0, ccs, first);     // uploads the masks when they changed
    std::vector<uint> c((size_t)M * 8);
    int rc = gwasdev_counts(gt.handle(), 0, (uint64_t)M, 1, c.data());
    assert(rc == GWASDEV_OK); (void)rc;
    const double per = scan.seconds() / (M > 0 ? M : 1);
    double tot, maf;
    for (int i = 0; i < M; ++i) {
        *out << (int)i;
        print_lapse(*out, "\t", per);
        *out << std::endl;
        frequency_table a, b;
        memcpy(a.freq, &c[8 * (size_t)i], 16); memcpy(b.freq, &c[8 * (size_t)i + 4], 16);
        MinorAlleleFrequency(a, tot, maf);
        MinorAlleleFrequency(b, tot, maf);
    }
}

void inline_maf_print(GeneticData *gd, std::ostream *out) {
    const int M = gd->getGenotypedMarkersCount(), N = gd->getGenotypedIndividualsCount();
    DeviceGenoTable &gt = *gd->getGenotypeTable();
    std::vector<uint> c((size_t)M * 4);
    int rc = gwasdev_counts(gt.handle(), 0, (uint64_t)M, 0, c.data());
    assert(rc == GWASDEV_OK); (void)rc;
    double tot, maf;
    for (int i = 0; i < M; ++i) {
        frequency_table ft;
        memcpy(ft.freq, &c[4 * (size_t)i], 16);
        MinorAlleleFrequency(ft, tot, maf);
        *out << (int)(N - tot) << "\t" << ft.aa << "\t" << ft.ab << "\t" << ft.bb << std::endl;
    }
}

void genotype_dist_performance(GeneticData *gd, std::ostream *out) {
    const int M = gd->getGenotypedMarkersCount();
    DeviceGenoTable &gt = *gd->getGenotypeTable();
    Lap scan;
    std::vector<uint> c((size_t)M * 4);
    int rc = gwasdev_counts(gt.handle(), 0, (uint64_t)M, 0, c.data());
    assert(rc == GWASDEV_OK); (void)rc;
    const double per = scan.seconds() / (M > 0 ? M : 1);
    for (int i = 0; i < M; ++i) { *out << (int)i; print_lapse(*out, "\t", per); *out << std::endl; }
}

// genetics/genotype/common_genotype_func.cpp:37-55 without the header row
void printContingencyTable(const CONTIN_TABLE_T &ct, std::ostream &out) {
    out << std::dec;
    for (int i = 0; i < 4; ++i) {
        for (int j = 0; j < 4; ++j) out << "\t" << ct.contin[i * 4 + j];
        out << std::endl;
    }
}

namespace {
const size_t PAIR_BATCH = 1u << 18;
// all pairs i < j of M markers in the reference's loop order, PAIR_BATCH at a time
template <class F> void for_pair_batches(uint M, F f) {
    std::vector<uint> pi, pj;
    pi.reserve(PAIR_BATCH); pj.reserve(PAIR_BATCH);
    uint64_t k0 = 0;
    for (uint i = 0; i < M; ++i)
        for (uint j = i + 1; j < M; ++j) {
            pi.push_back(i); pj.push_back(j);
            if (pi.size() == PAIR_BATCH) { f(k0, pi, pj); k0 += pi.size(); pi.clear(); pj.clear(); }
        }
    if (!pi.empty()) f(k0, pi, pj);
}
// EpistasisDebug / EpistasisPerformance build their own set: cases 0, 2, .., 398; controls 1, 3, .., 399 (:270-279)
void fixed_epistasis_set(CaseControlSet &ccs) {
    std::set<int> cases, ctrls;
    for (int i = 0; i < 200; ++i) { cases.insert(i << 1); ctrls.insert((i << 1) + 1); }
    ccs.setCases(cases);
    ccs.setControls(ctrls);
}
}  // namespace

void ContingencyDebug(GeneticData *gd, std::ostream *out) {
    DeviceGenoTable &gt = *gd->getGenotypeTable();
    std::vector<uint> tab;
    for_pair_batches((uint)gd->getGenotypedMarkersCount(), [&](uint64_t, const std::vector<uint> &pi, const std::vector<uint> &pj) {
        tab.resize(pi.size() * 32);
        int rc = gwasdev_pair_tables(gt.handle(), pi.size(), pi.data(), pj.data(), 0, tab.data());
        assert(rc == GWASDEV_OK); (void)rc;
        for (size_t q = 0; q < pi.size(); ++q) {
            *out << (int)pi[q] << " x " << (int)pj[q] << "\n";
            printContingencyTable(*reinterpret_cast<const CONTIN_TABLE_T *>(&tab[32 * q]), *out);
            *out << "\n";
        }
    });
}

namespace {
// one timing line per pair (k, lapse): the batched call's time is shared out evenly
void timed_tables(GeneticData *gd, std::ostream *out, int mode) {
    DeviceGenoTable &gt = *gd->getGenotypeTable();
    std::vector<uint> tab;
    for_pair_batches((uint)gd->getGenotypedMarkersCount(), [&](uint64_t k0, const std::vector<uint> &pi, const std::vector<uint> &pj) {
        tab.resize(pi.size() * 32);
        Lap lap;
        int rc = gwasdev_pair_tables(gt.handle(), pi.size(), pi.data(), pj.data(), mode, tab.data());
        assert(rc == GWASDEV_OK); (void)rc;
        const double per = lap.seconds() / (double)pi.size();
        for (size_t q = 0; q < pi.size(); ++q) { *out << (int)(k0 + q); print_lapse(*out, "\t", per); *out << std::endl; }
    });
}
}  // namespace

void ContingencyPerformance(GeneticData *gd, std::ostream *out) { timed_tables(gd, out, 0); }

void ContingencyCCPerformance(GeneticData *gd, std::ostream *out) {
    DeviceGenoTable &gt = *gd->getGenotypeTable();
    gt.selectCaseControl(*gd->getCaseControlSet());      // pre-select, margins are computed on first use (:150-156)
    timed_tables(gd, out, 3);
}

void EpistasisDebug(GeneticData *gd, std::ostream *out) {
    DeviceGenoTable &gt = *gd->getGenotypeTable();
    CaseControlSet ccs(gd->getGenotypedIndividualsCount());
    fixed_epistasis_set(ccs);
    gt.selectCaseControl(ccs);
    std::vector<uint> tab;
    std::vector<double> ll, pval;
    for_pair_batches((uint)gd->getGenotypedMarkersCount(), [&](uint64_t, const std::vector<uint> &pi, const std::vector<uint> &pj) {
        tab.resize(pi.size() * 32); ll.resize(pi.size()); pval.resize(pi.size());
        int rc = gwasdev_pair_tables(gt.handle(), pi.size(), pi.data(), pj.data(), 1, tab.data());
        assert(rc == GWASDEV_OK);
        rc = gwasdev_epi_pairs(gt.handle(), pi.size(), pi.data(), pj.data(), 1, ll.data(), pval.data());
        assert(rc == GWASDEV_OK); (void)rc;
        for (size_t q = 0; q < pi.size(); ++q) {
            *out << (int)pi[q] << " x " << (int)pj[q] << std::endl;
            *out << "Cases\n";
            printContingencyTable(*reinterpret_cast<const CONTIN_TABLE_T *>(&tab[32 * q]), *out);
            *out << "\nControls\n";
            printContingencyTable(*reinterpret_cast<const CONTIN_TABLE_T *>(&tab[32 * q + 16]), *out);
            out->flush();
            printf("\nLog likelihood: %f; p-value: %g\n\n", ll[q], pval[q]);      // to stdout, as the reference does (:302)
        }
    });
}

void EpistasisPerformance(GeneticData *gd, std::ostream *out) {
    DeviceGenoTable &gt = *gd->getGenotypeTable();
    CaseControlSet ccs(gd->getGenotypedIndividualsCount());
    fixed_epistasis_set(ccs);
    gt.selectCaseControl(ccs);
    std::vector<double> ll, pval;
    Lap lap;
    for_pair_batches((uint)gd->getGenotypedMarkersCount(), [&](uint64_t, const std::vector<uint> &pi, const std::vector<uint> &pj) {
        ll.resize(pi.size()); pval.resize(pi.size());
        int rc = gwasdev_epi_pairs(gt.handle(), pi.size(), pi.data(), pj.data(), 1, ll.data(), pval.data());
        assert(rc == GWASDEV_OK); (void)rc;
    });
    *out << "Case/Control Contingencies " << gd->getGenotypedMarkersCount() << ": ";
    print_lapse(std::cout, "", lap.seconds());
    std::cout << std::endl;
}

void computeMargins(DeviceGenoTable &gt, int nIndivids, marginal_information *&pMargins, int &nMarkerCount) {
    (void)nIndivids;
    nMarkerCount = gt.row_size();
    if (pMargins != NULL) delete[] pMargins;
    pMargins = new marginal_information[nMarkerCount];
    std::vector<marginal_information> tmp;
    gt.computeMargins(tmp);
    memcpy(pMargins, tmp.data(), sizeof(marginal_information) * (size_t)nMarkerCount);
}

void computeGTest(DeviceGenoTable &gt, marginal_information *, uint, std::vector<SNPInteractionPair> &passingThreshold,
                  std::vector<double> &zval) {
    std::vector<gwasdev_hit> hits(passingThreshold.size());
    for (size_t k = 0; k < hits.size(); ++k) { hits[k].i = passingThreshold[k].first.first; hits[k].j = passingThreshold[k].first.second; hits[k].stat = passingThreshold[k].second; }
    std::vector<double> stat;
    gt.gtestPairs(hits, stat, zval);
    for (size_t k = 0; k < hits.size(); ++k) passingThreshold[k].second = stat[k];
}

void computeBoost(GeneticData *gd, std::ostream *out) {
    CaseControlSet &ccs = *gd->getCaseControlSet();
    const int nIndivids = (int)(ccs.getCaseCount() + ccs.getControlCount());
    DeviceGenoTable &gt = *gd->getGenotypeTable();
    gt.selectCaseControl(ccs);
    const double thresholdRecord = 30.0;
    *out << "Pre-screening " << gt.row_size() << " SNP interactions" << std::endl;
    Lap lap;
    std::vector<gwasdev_hit> hits;
    gt.screenPairs(thresholdRecord, hits);                // margins + exhaustive screen + exact re-score on the device
    print_lapse(*out, "", lap.seconds());
    *out << std::endl;
    std::vector<SNPInteractionPair> passingThreshold;
    for (const gwasdev_hit &h : hits) passingThreshold.push_back(SNPInteractionPair(SNPPair(h.i, h.j), h.stat));
    *out << "Located " << passingThreshold.size() << " potential interactions" << std::endl;
    *out << "Performing deeper analysis of SNPs" << std::endl;
    std::vector<double> zval;
    computeGTest(gt, NULL, (uint)nIndivids, passingThreshold, zval);
    int idx = 0;
    char buf[256];
    for (size_t k = 0; k < passingThreshold.size(); ++k) {
        if (passingThreshold[k].second > thresholdRecord) {      // false for NaN: a G-test fit that never converged
            snprintf(buf, sizeof buf, "%7d\t%7d\t%7d\t%f\t%f\t%f\t%f", idx++, (int)passingThreshold[k].first.first,
                     (int)passingThreshold[k].first.second, 0.0, 0.0, passingThreshold[k].second, zval[k]);
            *out << buf << std::endl;
        }
    }
}

}  // namespace algorithms
}  // namespace libgwaspp
