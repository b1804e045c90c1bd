// TEST-ONLY host build of the play and root-noise helpers of the tree search (cn_chess_ai_b200/csrc/xq_search.cuh, xq_search_play_device,
// xq_search_root_noise_device), compiled with -ffp-contract=off like search_shim.cpp: the visit-count weights and the list-order sampled
// choice, the uniform draw of XQ_PICK_SAMPLE, and the log-Gamma / Dirichlet draw of one root.  Never loaded by the product package.
#include <cstdint>

#include "../../cn_chess_ai_b200/csrc/xq_search.cuh"

using namespace xq;

extern "C" {
// the weights of n root edges and the edge the play kernel samples with the draw u (-1 if no edge has a positive weight)
int sp_sample(const int32_t* visits, int n, float tau, float u, float* weights) {
    int nmax = 0;
    for (int k = 0; k < n; ++k) nmax = visits[k] > nmax ? visits[k] : nmax;
    if (nmax == 0) return -1;
    for (int k = 0; k < n; ++k) weights[k] = search_play_weight(visits[k], nmax, tau);
    return search_play_sample([&](int k) { return weights[k]; }, n, u);
}

float sp_uniform(uint64_t seed, uint64_t env_id, uint32_t ctr) { return policy_uniform(rng(seed, env_id, ctr)); }
uint64_t sp_rng(uint64_t seed, uint64_t env_id, uint32_t ctr) { return rng(seed, env_id, ctr); }

// lg[0 .. n) and eta[0 .. n) of one root drawn from base = xq_rng(seed, env id, root ctr)
void sp_dirichlet(uint64_t base, int n, float alpha, float* lg, float* eta) {
    for (int k = 0; k < n; ++k) lg[k] = search_log_gamma(base, k, alpha);
    search_dirichlet(base, n, alpha, eta);
}
}
