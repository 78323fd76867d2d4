// Host build of the opt-in root exploration sampler of sigma-zero_b200/csrc/tree.cuh -- test infrastructure only.
// Lets the tests recompute, without a GPU, the Dirichlet sample the device mixes into a root's priors.  Never loaded by the product.
#include <algorithm>
#include <vector>
#include "../../sigma-zero_b200/csrc/tree.cuh"

using namespace szb;

extern "C" {
// log-gamma draws of the children `moves` [n] (in the order given) for the key (seed, global game id, root ply)
void hx_dirichlet_log(uint64_t seed, uint64_t game_id, int ply, int n, const uint16_t* moves, double alpha, double* log_out) {
    const uint64_t key = dir_root_key(seed, game_id, ply);
    for (int k = 0; k < n; k++) log_out[k] = dir_log_gamma(key, moves[k], alpha);
}
// the Dirichlet sample over those children, reduced as the device reduces it (child k to lane k mod 32)
void hx_dirichlet(uint64_t seed, uint64_t game_id, int ply, int n, const uint16_t* moves, double alpha, double* eta_out) {
    std::vector<double> l(n);
    hx_dirichlet_log(seed, game_id, ply, n, moves, alpha, l.data());
    double mx = -INFINITY, part[32] = {0};
    for (int k = 0; k < n; k++) mx = std::max(mx, l[k]);
    for (int k = 0; k < n; k++) part[k & 31] = d_add(part[k & 31], exp(d_add(l[k], -mx)));
    const double total = dir_combine([&](int t) { return part[t]; });
    for (int k = 0; k < n; k++) eta_out[k] = exp(d_add(l[k], -mx)) / total;
}
}
