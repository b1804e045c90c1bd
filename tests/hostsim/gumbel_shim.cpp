// TEST-ONLY host build of the Gumbel root-search helpers of the tree search (cn_chess_ai_b200/csrc/xq_search.cuh, xq_gumbel_*), compiled
// with -ffp-contract=off like search_shim.cpp: the Gumbel draw, the considered set, the Sequential Halving sequence, the completed Q and
// sigma, the improved policy and its weights, the root rule and the action to play.  Never loaded by the product package.
#include <cstdint>

#include "../../cn_chess_ai_b200/csrc/xq_search.cuh"

using namespace xq;

extern "C" {
float gb_draw(uint64_t base, int k) { return gumbel_draw(base, k); }
uint64_t gb_rng(uint64_t seed, uint64_t env_id, uint32_t ctr) { return rng(seed, env_id, ctr); }
void gb_considered(const float* key, int n, int m, uint8_t* out) {
    for (int k = 0; k < n; ++k) out[k] = gumbel_considered(key, n, m, k) ? 1 : 0;
}
int gb_seq(int m, int n, int i) { return gumbel_seq(m, n, i); }
float gb_vmix(const int32_t* N, const float* W, const float* P, int n, float vhat) { return gumbel_vmix(N, W, P, n, vhat); }
void gb_root_scores(const int32_t* N, const float* W, const float* P, const float* g, const float* logit, int n, float vhat, float c_visit,
                    float c_scale, float* z, float* score) {
    gumbel_root_scores(N, W, P, g, logit, n, vhat, c_visit, c_scale, z, score);
}
// pi' and the weights of the logits z[0 .. n), as gumbel_policy_warp computes them
void gb_policy(const float* z, int n, float* p, uint32_t* w) {
    float zm = -INFINITY;
    for (int k = 0; k < n; ++k) zm = fmaxf(zm, z[k]);
    float s = 0.f;
    for (int k = 0; k < n; ++k) { p[k] = gumbel_exp(z[k], zm); s = s_add(s, p[k]); }
    for (int k = 0; k < n; ++k) { p[k] = s_div(p[k], s); w[k] = gumbel_weight(p[k]); }
}
int gb_pick(const uint8_t* cons, const int32_t* cnt, const float* score, int n, int target) {
    bool c[128];
    for (int k = 0; k < n; ++k) c[k] = cons[k] != 0;
    return gumbel_pick(c, cnt, score, n, target);
}
int gb_action(const uint8_t* cons, const int32_t* nv, const float* score, int n) {
    bool c[128];
    for (int k = 0; k < n; ++k) c[k] = cons[k] != 0;
    return gumbel_action(c, nv, score, n);
}
}
