// Where every model block of the Newton-KKT operator sits in K, shared by the derivative
// kernels (kkt_vjp.cu, jvp.cu).
//
// Block k of node i / edge e is the column-major rows x cols matrix of array G at element
// offset off, placed at K[ra:, cb:] of the full [x | y | z] vector (its transpose at
// K[cb:, ra:]); s is the factor the derivative kernels apply: -1 for off-diagonal blocks,
// -1/2 for the symmetric Hessian blocks (ra == cb), whose symmetric part is what K holds.
// The table is generic over the struct of arrays (gradients or tangents): both name their
// arrays after the model blocks.
#pragma once

#include <cuda_runtime.h>

#include "structure.hpp"

namespace sipoc {

constexpr int kKktNodeBlocks = 7;   // node_hxx, node_jc, node_jg, node_hxt, node_jct, node_jgt, node_htt
constexpr int kKktEdgeBlocks = 15;  // the nine stagewise edge blocks and the six theta ones
constexpr int kKktNodeHtt = 6;      // the theta x theta blocks: index in the lists above
constexpr int kKktEdgeHtt = 14;
constexpr int kKktNodeTheta = 3;    // first theta block of each list
constexpr int kKktEdgeTheta = 9;

template <class Ptr>
struct KktBlock {
  Ptr G;
  int off, rows, cols, ra, cb;
  double s;
};

template <class Arrays>
__device__ __forceinline__ KktBlock<decltype(Arrays::node_hxx)> kkt_node_block(
    const DevTables &t, const Arrays &g, int k, int i) {
  const int n = t.n[i], c = t.node_c[i], gg = t.node_g[i], p = t.theta_dim;
  const int xs = t.x_state[i], yc = t.x_dim + t.y_node_c[i], zn = t.x_dim + t.y_dim + t.z_node[i];
  const int th = t.sx_dim;
  switch (k) {
    case 0: return {g.node_hxx, t.nn_off[i], n, n, xs, xs, -0.5};
    case 1: return {g.node_jc, t.jc_node_off[i], c, n, yc, xs, -1.0};
    case 2: return {g.node_jg, t.jg_node_off[i], gg, n, zn, xs, -1.0};
    case 3: return {g.node_hxt, t.n_off[i] * p, n, p, xs, th, -1.0};
    case 4: return {g.node_jct, t.node_c_off[i] * p, c, p, yc, th, -1.0};
    case 5: return {g.node_jgt, t.node_g_off[i] * p, gg, p, zn, th, -1.0};
    default: return {g.node_htt, i * p * p, p, p, th, th, -0.5};
  }
}

template <class Arrays>
__device__ __forceinline__ KktBlock<decltype(Arrays::node_hxx)> kkt_edge_block(
    const DevTables &t, const Arrays &g, int k, int e) {
  const int par = t.parents[e], ch = t.children[e], p = t.theta_dim;
  const int np = t.n[par], nc = t.n[ch], m = t.m[e], c = t.edge_c[e], gg = t.edge_g[e];
  const int xp = t.x_state[par], xu = t.x_control[e], yd = t.x_dim + t.y_dyn[ch],
            yc = t.x_dim + t.y_edge_c[e], ze = t.x_dim + t.y_dim + t.z_edge[e];
  const int th = t.sx_dim;
  switch (k) {
    case 0: return {g.edge_hxx, t.hxx_edge_off[e], np, np, xp, xp, -0.5};
    case 1: return {g.edge_hxu, t.nm_off[e], np, m, xp, xu, -1.0};
    case 2: return {g.edge_huu, t.mm_off[e], m, m, xu, xu, -0.5};
    case 3: return {g.edge_A, t.a_off[e], nc, np, yd, xp, -1.0};
    case 4: return {g.edge_B, t.b_off[e], nc, m, yd, xu, -1.0};
    case 5: return {g.edge_jcx, t.jcx_off[e], c, np, yc, xp, -1.0};
    case 6: return {g.edge_jcu, t.jcu_off[e], c, m, yc, xu, -1.0};
    case 7: return {g.edge_jgx, t.jgx_off[e], gg, np, ze, xp, -1.0};
    case 8: return {g.edge_jgu, t.jgu_off[e], gg, m, ze, xu, -1.0};
    case 9: return {g.edge_hxt, t.pn_off[e] * p, np, p, xp, th, -1.0};
    case 10: return {g.edge_hut, t.m_off[e] * p, m, p, xu, th, -1.0};
    case 11: return {g.edge_dynt, t.cn_off[e] * p, nc, p, yd, th, -1.0};
    case 12: return {g.edge_jct, t.edge_c_off[e] * p, c, p, yc, th, -1.0};
    case 13: return {g.edge_jgt, t.edge_g_off[e] * p, gg, p, ze, th, -1.0};
    default: return {g.edge_htt, e * p * p, p, p, th, th, -0.5};
  }
}

}  // namespace sipoc
