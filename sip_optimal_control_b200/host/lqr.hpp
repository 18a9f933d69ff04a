// C++ host side of the B200 engine: the reference's lqr.hpp surface (same type and member
// names, same argument meaning, same error behaviour, same arena sizes) implemented over the
// C ABI of include/sipoc.h.  A translation unit written against the reference's
//   #include "sip_optimal_control/lqr.hpp"
// compiles against this header instead; LQR::factor / LQR::solve then run on the GPU.
//
// Reference interfaces mirrored (file:line in joaospinto/sip_optimal_control):
//   Topology            lqr.hpp:5-22,    lqr.cpp:12-48    aggregate, reserve / free / mem_assign / num_bytes
//   Dimensions          lqr.hpp:24-64,   lqr.cpp:50-180   aggregate, the same three allocation modes
//   LQR::FactorStatus   lqr.hpp:68-74
//   LQR::Input / Output lqr.hpp:76-106,  lqr.cpp:182-212
//   LQR::Workspace      lqr.hpp:109-187, lqr.cpp:214-471  the reference's public fields and byte counts
//   LQR                 lqr.hpp:189-199, lqr.cpp:635-871
// Topology, Dimensions, Output and Workspace keep the reference's three allocation modes:
// reserve / free (new[] / delete[]), mem_assign (carve a caller arena) and num_bytes (size
// it; identical values, tests in host_tests.cpp).  The kept factorization itself lives on
// the device: the host arrays of Workspace (W, K, V, ...) exist with the reference's sizes so
// that arenas sized for the reference fit, but LQR does not populate them; the engine handle
// and its pinned staging hang off Workspace::device, created on first use and released by
// free() / release_device() (an arena user calls release_device()).
// The classic classes solve ONE problem per call (batch of one through the host-buffer entry
// points, like a maintainer's drop-in shim would); BatchedLQR exposes the same operations on
// a batch of problems resident on the device.
#pragma once

#include <cstdint>

struct sipoc_engine;

namespace sip::optimal_control {

struct Topology {
  int num_edges = 0;
  int root = 0;
  const int *edge_parents = nullptr;
  const int *edge_children = nullptr;

  int num_nodes() const;

  void reserve(int num_edges);
  void free();
  int mem_assign(int num_edges, unsigned char *mem_ptr);
  static constexpr int num_bytes(int num_edges) {
    return 2 * num_edges * static_cast<int>(sizeof(int));  // parents, children
  }

  void set_chain();
  void set_tree(int root, const int *edge_parents, const int *edge_children);
};

struct Dimensions {
  // State and node-constraint dimensions are indexed by node, control and edge-constraint
  // dimensions by edge.  A null constraint array means "all zero".
  int theta_dim = 0;
  const int *state_dims = nullptr;
  const int *control_dims = nullptr;
  const int *node_c_dims = nullptr;
  const int *node_g_dims = nullptr;
  const int *edge_c_dims = nullptr;
  const int *edge_g_dims = nullptr;

  void reserve(int num_edges);
  void free();
  int mem_assign(int num_edges, unsigned char *mem_ptr);
  static constexpr int num_bytes(int num_edges) {
    // three per-node and three per-edge int tables
    return (3 * (num_edges + 1) + 3 * num_edges) * static_cast<int>(sizeof(int));
  }

  void set_uniform(int num_edges, int state_dim, int control_dim, int node_c_dim,
                   int node_g_dim, int edge_c_dim, int edge_g_dim, int theta_dim = 0);

  int get_schur_dim() const;
  int get_state_dim(int node) const;
  int get_control_dim(int edge) const;
  int get_node_c_dim(int node) const;
  int get_node_g_dim(int node) const;
  int get_edge_c_dim(int edge) const;
  int get_edge_g_dim(int edge) const;
  int max_state_dim(int num_nodes) const;
  int max_control_dim(int num_edges) const;
  int max_node_c_dim(int num_nodes) const;
  int max_node_g_dim(int num_nodes) const;
  int max_edge_c_dim(int num_edges) const;
  int max_edge_g_dim(int num_edges) const;
  int get_stagewise_x_dim(int num_edges) const;
  int get_x_dim(int num_edges) const;
  int get_y_dim(int num_edges) const;
  int get_z_dim(int num_edges) const;
  int get_stagewise_kkt_dim(int num_edges) const;
};

class LQR {
 public:
  enum class FactorStatus {
    SUCCESS = 0,
    INVALID_DELTA = 1,
    F_FACTORIZATION_FAILURE = 2,
    G_FACTORIZATION_FAILURE = 3,
    INVALID_TOPOLOGY = 4,
  };

  // Views of caller-owned memory, one pointer per node / edge, column-major blocks.
  struct Input {
    double **Q;
    double **M;
    double **R;
    double **q;
    double **r;
    double **A;
    double **B;
    double **c;
    double **delta;

    const Dimensions &dimensions;
    const Topology &topology;
  };

  struct Output {
    double **x;
    double **u;
    double **y;

    void reserve(int num_edges);
    void free();
    auto mem_assign(int num_edges, unsigned char *mem_ptr) -> int;
    static constexpr auto num_bytes(int num_edges) -> int {
      // x and y tables of num_edges + 1 pointers, u of num_edges
      return (2 * (num_edges + 1) + num_edges) * static_cast<int>(sizeof(double *));
    }
  };

  struct DeviceState;  // engine handle + pinned staging (lqr.cpp)

  struct Workspace {
    // Per edge / per node blocks of the reference's kept factorization.
    double **W;
    double **K;
    double **V;
    double **G_factor;
    double **F_factor;
    double **sqrt_delta;
    double **sqrt_delta_inv;
    double **k;
    double **v;
    // Single-edge scratch.
    double *G;
    double *g;
    double *H;
    double *h;
    double *F;
    double *f;
    // Compiled topology (CSR children, traversal orders); filled by compile_topology().
    int *child_offsets;
    int *child_edges;
    int *edge_parents;
    int *edge_children;
    int *preorder_nodes;
    int *postorder_nodes;
    int *node_marks;

    void reserve(int state_dim, int control_dim, int num_edges);
    void reserve(const Dimensions &dimensions, const Topology &topology);
    void free(int num_edges);

    auto mem_assign(const Dimensions &dimensions, const Topology &topology,
                    unsigned char *mem_ptr) -> int;

    // Uniform chain: per edge W n^2, K m n, G_factor m^2, k m; per node V n^2, F_factor n^2,
    // sqrt_delta, sqrt_delta_inv, v n each; one pointer per block; scratch G, g, H, h, F, f;
    // seven int tables.
    static constexpr auto num_bytes(int state_dim, int control_dim, int num_edges) -> int {
      const int n = state_dim, m = control_dim, E = num_edges, N = num_edges + 1;
      const int dbl = static_cast<int>(sizeof(double)), ptr = static_cast<int>(sizeof(double *));
      const int per_edge = n * n + m * n + m * m + m;
      const int per_node = 2 * n * n + 3 * n;
      const int scratch = m * m + n + m * n + m + n * n + n;
      const int ints = (N + 1) + 3 * E + 3 * N;
      return (4 * E + 5 * N) * ptr + (E * per_edge + N * per_node + scratch) * dbl +
             ints * static_cast<int>(sizeof(int));
    }
    static auto num_bytes(const Dimensions &dimensions, const Topology &topology) -> int;

    // Not in the reference: the GPU engine behind this workspace.
    DeviceState *device = nullptr;
    void release_device();
  };

  LQR(const Input &data, Workspace &workspace);

  auto compile_topology() -> FactorStatus;
  FactorStatus factor_with_status();
  bool factor();
  void solve(Output &output);

 private:
  const Input &input_;
  Workspace &workspace_;
  FactorStatus traversal_status_;
};

// The engine of a workspace (created by LQR / CallbackProvider), or nullptr.
sipoc_engine *engine_of(const LQR::Workspace &workspace);

// The same operations on `batch` problems of one structure, device resident in the
// engine layout X[flat * batch_stride() + problem] (include/sipoc.h).
class BatchedLQR {
 public:
  BatchedLQR(const Dimensions &dimensions, const Topology &topology, int64_t batch,
             int device = -1);
  ~BatchedLQR();
  BatchedLQR(const BatchedLQR &) = delete;
  BatchedLQR &operator=(const BatchedLQR &) = delete;

  LQR::FactorStatus topology_status() const { return status_; }
  int64_t batch_stride() const;
  sipoc_engine *engine() const { return engine_; }

  // Device pointers; `status` is int[batch_stride()] with FactorStatus values.
  struct DeviceInput {
    const double *Q, *M, *R, *q, *r, *A, *B, *c, *delta;
  };
  struct DeviceOutput {
    double *x, *u, *y;
  };
  bool factor_with_status(const DeviceInput &in, int *status, void *stream = nullptr);
  bool solve(const DeviceInput &in, const DeviceOutput &out, void *stream = nullptr);
  bool factor_solve(const DeviceInput &in, const DeviceOutput &out, int *status,
                    void *stream = nullptr);
  // factor_solve, then the feedback policy u_e = K_e x_parent + k_e, y_i = V_i x_i + v_i of
  // every problem (sipoc_lqr_factor_solve_policy); a nullptr array is not computed.
  struct DevicePolicy {
    double *K, *k, *V, *v;
  };
  bool factor_solve_policy(const DeviceInput &in, const DeviceOutput &out,
                           const DevicePolicy &policy, int *status, void *stream = nullptr);

 private:
  sipoc_engine *engine_ = nullptr;
  LQR::FactorStatus status_ = LQR::FactorStatus::SUCCESS;
};

}  // namespace sip::optimal_control
