// TEST INFRASTRUCTURE ONLY (oracle/).  Stand-in for include/ORBVocabulary.h in the adapter build of oracle/dbowref_wrap.cpp
// (oracle/Makefile target `adapt`): the vocabulary calls the wrapper makes are answered by the CPU restatement (liborbport.so
// sources, linked in), which tests/test_oracle_dbow_ref.py pins to DBoW2.  The product's KeyFrameDatabase adapter itself does not
// use the vocabulary.
#pragma once
#include <cstdint>
#include <cstring>
#include <string>
#include <vector>

#include <opencv2/core/core.hpp>

#include "Thirdparty/DBoW2/DBoW2/BowVector.h"
#include "Thirdparty/DBoW2/DBoW2/FeatureVector.h"

extern "C" {
void* orbport_voc_load_text(const char* path);
void orbport_voc_free(void* h);
int orbport_voc_nodes(void* h);
void orbport_voc_export(void* h, int32_t* parent, uint8_t* is_leaf, int32_t* word_id, uint8_t* desc, double* weight, int* k, int* L);
void orbport_compute_bow(void* h, const uint8_t* desc, int n, int levelsup, uint32_t* bow_word, double* bow_value, int32_t* n_bow,
                         uint32_t* fv_node, int32_t* fv_start, uint32_t* fv_idx, int32_t* n_nodes);
double orbport_bow_score_l1(const uint32_t* w1, const double* v1, int n1, const uint32_t* w2, const double* v2, int n2, int32_t* common,
                            uint32_t* first);
}

namespace ORB_SLAM2 {

class ORBVocabulary {
public:
    ORBVocabulary() = default;
    ORBVocabulary(const ORBVocabulary&) = delete;
    ORBVocabulary& operator=(const ORBVocabulary&) = delete;
    ~ORBVocabulary() { if (h_) orbport_voc_free(h_); }

    bool loadFromTextFile(const std::string& path) {
        h_ = orbport_voc_load_text(path.c_str());
        if (!h_) return false;
        const int n = orbport_voc_nodes(h_);
        std::vector<int32_t> parent(n), word(n);
        std::vector<uint8_t> leaf(n), desc((size_t)n * 32);
        std::vector<double> weight(n);
        int k = 0, L = 0;
        orbport_voc_export(h_, parent.data(), leaf.data(), word.data(), desc.data(), weight.data(), &k, &L);
        words_ = 0;
        for (uint8_t l : leaf) words_ += l != 0;
        return true;
    }

    unsigned int size() const { return words_; }

    void transform(const std::vector<cv::Mat>& features, DBoW2::BowVector& bow, DBoW2::FeatureVector& fv, int levelsup) const {
        const int n = (int)features.size();
        std::vector<uint8_t> desc((size_t)n * 32);
        for (int i = 0; i < n; i++) std::memcpy(&desc[(size_t)i * 32], features[i].data, 32);
        const size_t m = n > 0 ? n : 1;
        std::vector<uint32_t> bw(m), fnode(m), fidx(m);
        std::vector<double> bv(m);
        std::vector<int32_t> fstart(m + 1);
        int32_t nb = 0, nn = 0;
        orbport_compute_bow(h_, desc.data(), n, levelsup, bw.data(), bv.data(), &nb, fnode.data(), fstart.data(), fidx.data(), &nn);
        bow.clear();
        fv.clear();
        for (int i = 0; i < nb; i++) bow.insert(bow.end(), std::make_pair(bw[i], bv[i]));
        for (int a = 0; a < nn; a++)
            fv.insert(fv.end(), std::make_pair(fnode[a], std::vector<unsigned int>(fidx.begin() + fstart[a], fidx.begin() + fstart[a + 1])));
    }

    double score(const DBoW2::BowVector& a, const DBoW2::BowVector& b) const {
        std::vector<uint32_t> wa, wb;
        std::vector<double> va, vb;
        for (const auto& e : a) { wa.push_back(e.first); va.push_back(e.second); }
        for (const auto& e : b) { wb.push_back(e.first); vb.push_back(e.second); }
        return orbport_bow_score_l1(wa.data(), va.data(), (int)wa.size(), wb.data(), vb.data(), (int)wb.size(), nullptr, nullptr);
    }

private:
    void* h_ = nullptr;
    unsigned int words_ = 0;
};

}  // namespace ORB_SLAM2
