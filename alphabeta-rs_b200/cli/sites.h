// sites.h — the [S][L] site arrays of a pedigree's measured samples, read as abfit_pedigree_build reads the methylome
// files (node files relative to the CWD), shared by the command-line tools that need the sites themselves
// (`alphabeta --site-bootstrap`, `regions`).
#pragma once
#include <cstdio>
#include <fstream>
#include <sstream>
#include <string>
#include <vector>

#include "../../include/abfit.h"

// The site arrays of the measured samples and the (i, j) samples of every pedigree row.  Every sample must list the same
// number of sites; with `coords` the samples must list the same (chromosome, position) sequence as well, and coords
// receives it (the first sample's sites).  Errors are printed as "Error: <what>: ..." and return false.
static bool read_sites(const std::string &nodes, const std::string &edges, int32_t n_pairs, int32_t &S, int64_t &L,
                       std::vector<uint8_t> &st, std::vector<double> &po, std::vector<double> &me, std::vector<int32_t> &pairs,
                       const char *what = "--site-bootstrap", std::vector<abfit_cg_site> *coords = nullptr)
{
    std::vector<char> files(1 << 20);
    std::vector<double> pr((size_t)n_pairs * 5);
    int32_t np = 0;
    if (abfit_pedigree_graph(nodes.c_str(), edges.c_str(), &S, files.data(), (int32_t)files.size(), &np, pr.data(), n_pairs) ||
        np != n_pairs) {
        std::printf("Error: %s\n", abfit_last_error());
        return false;
    }
    pairs.resize((size_t)n_pairs * 2);
    for (int32_t r = 0; r < n_pairs; ++r) {
        pairs[2 * r] = (int32_t)pr[5 * r];
        pairs[2 * r + 1] = (int32_t)pr[5 * r + 1];
    }
    std::istringstream names(std::string(files.data()));
    std::string fn;
    std::vector<std::vector<uint8_t>> s_st;
    std::vector<std::vector<double>> s_po, s_me;
    std::vector<abfit_cg_site> sites;
    std::vector<int64_t> line_off;
    while (std::getline(names, fn)) {
        std::ifstream f(fn, std::ios::binary);
        if (!f) {
            std::printf("Error: Could not open node file: %s\n", fn.c_str());
            return false;
        }
        const std::string image((std::istreambuf_iterator<char>(f)), std::istreambuf_iterator<char>());
        int64_t cap = 1, n = 0;
        for (char ch : image) cap += ch == '\n';
        s_st.emplace_back((size_t)cap);
        s_po.emplace_back((size_t)cap);
        s_me.emplace_back((size_t)cap);
        if (coords) {
            sites.resize((size_t)cap);
            line_off.resize((size_t)cap);
        }
        if (abfit_parse_methylome_buffer(image.data(), (int64_t)image.size(), 0, 0, cap, coords ? sites.data() : nullptr,
                                         s_po.back().data(), s_st.back().data(), s_me.back().data(),
                                         coords ? line_off.data() : nullptr, nullptr, &n)) {
            std::printf("Error: %s\n", abfit_last_error());
            return false;
        }
        s_st.back().resize((size_t)n);
        if (coords) {
            sites.resize((size_t)n);
            if (s_st.size() == 1) {
                *coords = sites;
            } else {
                // the first site where this sample and the first one differ, and its line in this file
                size_t k = 0;
                while (k < sites.size() && k < coords->size() && sites[k].chromosome == (*coords)[k].chromosome &&
                       sites[k].start == (*coords)[k].start)
                    ++k;
                if (k < sites.size() || k < coords->size()) {
                    int64_t line = 1;
                    const int64_t end = k < sites.size() ? line_off[k] : (int64_t)image.size();
                    for (int64_t i = 0; i < end; ++i) line += image[(size_t)i] == '\n';
                    std::printf("Error: %s: %s differs from the first sample at line %lld (site %zu): every sample must list the "
                                "same (chromosome, position) sequence\n", what, fn.c_str(), (long long)line, k);
                    return false;
                }
            }
        }
        if (s_st.size() > 1 && s_st.back().size() != s_st[0].size()) {
            std::printf("Error: %s: %s lists %lld sites, the first sample %lld; the site-block bootstrap needs "
                        "every sample to list the same sites\n", what, fn.c_str(), (long long)n, (long long)s_st[0].size());
            return false;
        }
    }
    if ((int32_t)s_st.size() != S) {
        std::printf("Error: %s: expected %d methylome files\n", what, S);
        return false;
    }
    L = (int64_t)s_st[0].size();
    st.resize((size_t)S * L);
    po.resize((size_t)S * L);
    me.resize((size_t)S * L);
    for (int32_t s = 0; s < S; ++s) {
        std::copy(s_st[s].begin(), s_st[s].begin() + L, st.begin() + (size_t)s * L);
        std::copy(s_po[s].begin(), s_po[s].begin() + L, po.begin() + (size_t)s * L);
        std::copy(s_me[s].begin(), s_me[s].begin() + L, me.begin() + (size_t)s * L);
    }
    return true;
}
