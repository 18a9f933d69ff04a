// See lqr.hpp.  Nothing here computes: the classes gather the caller's per-node /
// per-edge blocks into the flat arrays of the C ABI and forward the calls.
#include "lqr.hpp"

#include <algorithm>
#include <vector>

#include "../../include/sipoc.h"
#include "device_state.hpp"

namespace sip::optimal_control {

// ---- Topology (lqr.cpp:12-48) ------------------------------------------------------
// Plain aggregate, as in the reference: reserve() owns its two tables until free();
// mem_assign() points them into a caller arena of num_bytes(num_edges) bytes.
int Topology::num_nodes() const { return num_edges + 1; }

void Topology::reserve(int edges) {
  num_edges = edges;
  edge_parents = new int[std::max(edges, 1)]();
  edge_children = new int[std::max(edges, 1)]();
}

void Topology::free() {
  delete[] edge_parents;
  delete[] edge_children;
  edge_parents = edge_children = nullptr;
}

int Topology::mem_assign(int edges, unsigned char *mem_ptr) {
  int *tables = reinterpret_cast<int *>(mem_ptr);
  num_edges = edges;
  edge_parents = tables;
  edge_children = tables + edges;
  return num_bytes(edges);
}

void Topology::set_chain() {
  root = 0;
  int *parents = const_cast<int *>(edge_parents), *children = const_cast<int *>(edge_children);
  for (int e = 0; e < num_edges; ++e) {
    parents[e] = e;
    children[e] = e + 1;
  }
}

void Topology::set_tree(int new_root, const int *parents, const int *children) {
  root = new_root;
  std::copy(parents, parents + num_edges, const_cast<int *>(edge_parents));
  std::copy(children, children + num_edges, const_cast<int *>(edge_children));
}

// ---- Dimensions (lqr.cpp:50-180) -----------------------------------------------------
namespace {
// The six tables in declaration order with their lengths for E edges.
struct DimTables {
  const int **slot[6];
  int count[6];
  DimTables(Dimensions &d, int E)
      : slot{&d.state_dims,  &d.control_dims, &d.node_c_dims,
             &d.node_g_dims, &d.edge_c_dims,  &d.edge_g_dims},
        count{E + 1, E, E + 1, E + 1, E, E} {}
};
int largest(const int *v, int count) {
  int best = 0;
  for (int i = 0; v != nullptr && i < count; ++i) best = std::max(best, v[i]);
  return best;
}
}  // namespace

void Dimensions::reserve(int num_edges) {
  DimTables t(*this, num_edges);
  for (int i = 0; i < 6; ++i) *t.slot[i] = new int[std::max(t.count[i], 1)]();
}

void Dimensions::free() {
  DimTables t(*this, 0);
  for (int i = 0; i < 6; ++i) {
    delete[] *t.slot[i];
    *t.slot[i] = nullptr;
  }
}

int Dimensions::mem_assign(int num_edges, unsigned char *mem_ptr) {
  DimTables t(*this, num_edges);
  int *cursor = reinterpret_cast<int *>(mem_ptr);
  for (int i = 0; i < 6; ++i) {
    *t.slot[i] = cursor;
    cursor += t.count[i];
  }
  return num_bytes(num_edges);
}

void Dimensions::set_uniform(int num_edges, int state_dim, int control_dim, int node_c_dim,
                             int node_g_dim, int edge_c_dim, int edge_g_dim, int theta) {
  theta_dim = theta;
  DimTables t(*this, num_edges);
  const int value[6] = {state_dim, control_dim, node_c_dim, node_g_dim, edge_c_dim, edge_g_dim};
  for (int i = 0; i < 6; ++i)
    std::fill_n(const_cast<int *>(*t.slot[i]), t.count[i], value[i]);
}

int Dimensions::get_schur_dim() const { return theta_dim; }
int Dimensions::get_state_dim(int node) const { return state_dims[node]; }
int Dimensions::get_control_dim(int edge) const { return control_dims[edge]; }
// A null constraint-dimension array means "all zero" (lqr.cpp:98-112).
int Dimensions::get_node_c_dim(int node) const { return node_c_dims ? node_c_dims[node] : 0; }
int Dimensions::get_node_g_dim(int node) const { return node_g_dims ? node_g_dims[node] : 0; }
int Dimensions::get_edge_c_dim(int edge) const { return edge_c_dims ? edge_c_dims[edge] : 0; }
int Dimensions::get_edge_g_dim(int edge) const { return edge_g_dims ? edge_g_dims[edge] : 0; }
int Dimensions::max_state_dim(int num_nodes) const { return largest(state_dims, num_nodes); }
int Dimensions::max_control_dim(int num_edges) const { return largest(control_dims, num_edges); }
int Dimensions::max_node_c_dim(int num_nodes) const { return largest(node_c_dims, num_nodes); }
int Dimensions::max_node_g_dim(int num_nodes) const { return largest(node_g_dims, num_nodes); }
int Dimensions::max_edge_c_dim(int num_edges) const { return largest(edge_c_dims, num_edges); }
int Dimensions::max_edge_g_dim(int num_edges) const { return largest(edge_g_dims, num_edges); }

int Dimensions::get_stagewise_x_dim(int num_edges) const {
  int total = state_dims[num_edges];
  for (int e = 0; e < num_edges; ++e) total += state_dims[e] + control_dims[e];
  return total;
}
int Dimensions::get_x_dim(int num_edges) const { return get_stagewise_x_dim(num_edges) + theta_dim; }
int Dimensions::get_y_dim(int num_edges) const {
  int total = 0;
  for (int i = 0; i <= num_edges; ++i) total += state_dims[i] + get_node_c_dim(i);
  for (int e = 0; e < num_edges; ++e) total += get_edge_c_dim(e);
  return total;
}
int Dimensions::get_z_dim(int num_edges) const {
  int total = 0;
  for (int i = 0; i <= num_edges; ++i) total += get_node_g_dim(i);
  for (int e = 0; e < num_edges; ++e) total += get_edge_g_dim(e);
  return total;
}
int Dimensions::get_stagewise_kkt_dim(int num_edges) const {
  return get_stagewise_x_dim(num_edges) + get_y_dim(num_edges) + get_z_dim(num_edges);
}

// ---- LQR::Output (lqr.cpp:182-212) ---------------------------------------------------
void LQR::Output::reserve(int num_edges) {
  x = new double *[num_edges + 1]();
  u = new double *[std::max(num_edges, 1)]();
  y = new double *[num_edges + 1]();
}
void LQR::Output::free() {
  delete[] x;
  delete[] u;
  delete[] y;
  x = u = y = nullptr;
}
auto LQR::Output::mem_assign(int num_edges, unsigned char *mem_ptr) -> int {
  double **tables = reinterpret_cast<double **>(mem_ptr);
  x = tables;
  u = x + (num_edges + 1);
  y = u + num_edges;
  return num_bytes(num_edges);
}

// ---- LQR::Workspace (lqr.cpp:214-471) ------------------------------------------------
// One description of the workspace's blocks serves the allocation modes: walk_tables /
// walk_blocks visit every block in the reference's arena order (pointer tables, per-edge
// blocks, per-node blocks, single-edge scratch, topology ints) and hand it to a policy that
// carves it from an arena (mem_assign), allocates it (reserve) or releases it (free).
namespace {

template <class Policy>
void walk_tables(LQR::Workspace &w, int E, Policy &&pol) {
  const int N = E + 1;
  pol.table(w.W, E);
  pol.table(w.K, E);
  pol.table(w.V, N);
  pol.table(w.G_factor, E);
  pol.table(w.F_factor, N);
  pol.table(w.sqrt_delta, N);
  pol.table(w.sqrt_delta_inv, N);
  pol.table(w.k, E);
  pol.table(w.v, N);
}

template <class Policy>
void walk_blocks(LQR::Workspace &w, const Dimensions &d, int E, Policy &&pol) {
  const int N = E + 1;
  const int nmax = d.max_state_dim(N), mmax = d.max_control_dim(E);
  for (int e = 0; e < E; ++e) {
    const int m = d.get_control_dim(e);
    pol.block(w.W[e], nmax * nmax);  // W of an edge is sized for the largest state
    pol.block(w.K[e], m * nmax);
    pol.block(w.G_factor[e], m * m);
    pol.block(w.k[e], m);
  }
  for (int i = 0; i < N; ++i) {
    const int n = d.get_state_dim(i);
    pol.block(w.V[i], n * n);
    pol.block(w.F_factor[i], n * n);
    pol.block(w.sqrt_delta[i], n);
    pol.block(w.sqrt_delta_inv[i], n);
    pol.block(w.v[i], n);
  }
  pol.block(w.G, mmax * mmax);
  pol.block(w.g, nmax);
  pol.block(w.H, mmax * nmax);
  pol.block(w.h, mmax);
  pol.block(w.F, nmax * nmax);
  pol.block(w.f, nmax);
  pol.ints(w.child_offsets, N + 1);
  pol.ints(w.child_edges, E);
  pol.ints(w.edge_parents, E);
  pol.ints(w.edge_children, E);
  pol.ints(w.preorder_nodes, N);
  pol.ints(w.postorder_nodes, N);
  pol.ints(w.node_marks, N);
}

struct HeapAlloc {
  void table(double **&t, int count) { t = new double *[std::max(count, 1)](); }
  void block(double *&b, int count) { b = new double[std::max(count, 1)](); }
  void ints(int *&b, int count) { b = new int[std::max(count, 1)](); }
};
struct HeapRelease {
  void table(double **&t, int) {
    delete[] t;
    t = nullptr;
  }
  void block(double *&b, int) {
    delete[] b;
    b = nullptr;
  }
  void ints(int *&b, int) {
    delete[] b;
    b = nullptr;
  }
};
struct ArenaCarve {
  unsigned char *cursor;
  template <class T>
  T *take(int count) {
    T *p = reinterpret_cast<T *>(cursor);
    cursor += static_cast<size_t>(count) * sizeof(T);
    return p;
  }
  void table(double **&t, int count) { t = take<double *>(count); }
  void block(double *&b, int count) { b = take<double>(count); }
  void ints(int *&b, int count) { b = take<int>(count); }
};

}  // namespace

void LQR::Workspace::reserve(int state_dim, int control_dim, int num_edges) {
  Dimensions d;
  d.reserve(num_edges);
  d.set_uniform(num_edges, state_dim, control_dim, 0, 0, 0, 0);
  Topology t;
  t.reserve(num_edges);
  t.set_chain();
  reserve(d, t);
  t.free();
  d.free();
}

void LQR::Workspace::reserve(const Dimensions &dimensions, const Topology &topology) {
  walk_tables(*this, topology.num_edges, HeapAlloc{});
  walk_blocks(*this, dimensions, topology.num_edges, HeapAlloc{});
}

void LQR::Workspace::free(int num_edges) {
  release_device();
  if (W == nullptr) return;
  // The blocks only need their pointers, not their sizes: a dimension-free description.
  const std::vector<int> ones(static_cast<size_t>(num_edges) + 1, 1);
  Dimensions d{0, ones.data(), ones.data(), nullptr, nullptr, nullptr, nullptr};
  walk_blocks(*this, d, num_edges, HeapRelease{});
  walk_tables(*this, num_edges, HeapRelease{});
}

auto LQR::Workspace::mem_assign(const Dimensions &dimensions, const Topology &topology,
                                unsigned char *mem_ptr) -> int {
  ArenaCarve carve{mem_ptr};
  walk_tables(*this, topology.num_edges, carve);
  walk_blocks(*this, dimensions, topology.num_edges, carve);
  return static_cast<int>(carve.cursor - mem_ptr);
}

auto LQR::Workspace::num_bytes(const Dimensions &dimensions, const Topology &topology) -> int {
  // (walk_blocks needs the pointer tables to exist, so the arena is measured here, not walked.)
  const int E = topology.num_edges, N = E + 1;
  const int nmax = dimensions.max_state_dim(N), mmax = dimensions.max_control_dim(E);
  int64_t doubles = 0;
  for (int e = 0; e < E; ++e) {
    const int m = dimensions.get_control_dim(e);
    doubles += nmax * nmax + m * nmax + m * m + m;
  }
  for (int i = 0; i < N; ++i) {
    const int n = dimensions.get_state_dim(i);
    doubles += 2 * n * n + 3 * n;
  }
  doubles += mmax * mmax + nmax + mmax * nmax + mmax + nmax * nmax + nmax;
  const int64_t pointers = 4 * E + 5 * N, ints = (N + 1) + 3 * E + 3 * N;
  return static_cast<int>(pointers * sizeof(double *) + doubles * sizeof(double) +
                          ints * sizeof(int));
}

void LQR::Workspace::release_device() {
  delete device;
  device = nullptr;
}

sipoc_engine *engine_of(const LQR::Workspace &workspace) {
  return workspace.device != nullptr ? workspace.device->engine : nullptr;
}

namespace {

sipoc_structure describe(const Dimensions &d, const Topology &t, int64_t batch, int device) {
  sipoc_structure s{};
  s.num_edges = t.num_edges;
  s.root = t.root;
  s.edge_parents = t.edge_parents;
  s.edge_children = t.edge_children;
  s.state_dims = d.state_dims;
  s.control_dims = d.control_dims;
  s.node_c_dims = d.node_c_dims;
  s.node_g_dims = d.node_g_dims;
  s.edge_c_dims = d.edge_c_dims;
  s.edge_g_dims = d.edge_g_dims;
  s.theta_dim = d.theta_dim;
  s.batch = batch;
  s.device = device;
  s.flags = 0;
  return s;
}

// Blocks of one array, in node / edge order, appended to `flat`.
void gather(double **table, int count, const std::vector<int> &elems, std::vector<double> &flat) {
  size_t o = 0;
  for (int i = 0; i < count; ++i) {
    if (elems[i] == 0) continue;
    std::copy(table[i], table[i] + elems[i], flat.begin() + o);
    o += elems[i];
  }
}
void scatter(const std::vector<double> &flat, double **table, int count,
             const std::vector<int> &elems) {
  size_t o = 0;
  for (int i = 0; i < count; ++i) {
    if (elems[i] == 0) continue;
    std::copy(flat.begin() + o, flat.begin() + o + elems[i], table[i]);
    o += elems[i];
  }
}

struct BlockSizes {
  std::vector<int> nn, n, nm, mm, m, a, b;
  BlockSizes(const Dimensions &d, const Topology &t) {
    const int E = t.num_edges;
    for (int i = 0; i <= E; ++i) {
      nn.push_back(d.state_dims[i] * d.state_dims[i]);
      n.push_back(d.state_dims[i]);
    }
    for (int e = 0; e < E; ++e) {
      const int np = d.state_dims[t.edge_parents[e]], nc = d.state_dims[t.edge_children[e]],
                mm_ = d.control_dims[e];
      nm.push_back(np * mm_);
      mm.push_back(mm_ * mm_);
      m.push_back(mm_);
      a.push_back(nc * np);
      b.push_back(nc * mm_);
    }
  }
};

}  // namespace

// ---- LQR (lqr.cpp:635-871) -------------------------------------------------------------
LQR::LQR(const Input &data, Workspace &workspace)
    : input_(data), workspace_(workspace), traversal_status_(compile_topology()) {}

auto LQR::compile_topology() -> FactorStatus {
  workspace_.release_device();
  auto *dev = new DeviceState();
  const sipoc_structure s = describe(input_.dimensions, input_.topology, 1, -1);
  const sipoc_error rc = sipoc_create(&s, &dev->engine);
  if (rc != SIPOC_OK) {
    dev->engine = nullptr;
    delete dev;
    // An invalid tree is latched and reported by every later factor (lqr.cpp:646-648).
    return FactorStatus::INVALID_TOPOLOGY;
  }
  workspace_.device = dev;
  sipoc_lqr_sizes z{};
  sipoc_lqr_get_sizes(dev->engine, &z);
  const int64_t sizes[9] = {z.Q, z.M, z.R, z.q, z.r, z.A, z.B, z.c, z.delta};
  for (int i = 0; i < 9; ++i) dev->in[i].assign(static_cast<size_t>(sizes[i]), 0.0);
  dev->out[0].assign(static_cast<size_t>(z.x), 0.0);
  dev->out[1].assign(static_cast<size_t>(z.u), 0.0);
  dev->out[2].assign(static_cast<size_t>(z.y), 0.0);
  // The compiled topology lands in the workspace's own tables, like the reference's
  // compile_topology_data (lqr.cpp:563-631); they must have been reserved / assigned.
  if (workspace_.child_offsets != nullptr) {
    const int E = input_.topology.num_edges;
    sipoc_get_topology(dev->engine, workspace_.child_offsets, workspace_.child_edges,
                       workspace_.preorder_nodes, workspace_.postorder_nodes);
    std::copy(input_.topology.edge_parents, input_.topology.edge_parents + E,
              workspace_.edge_parents);
    std::copy(input_.topology.edge_children, input_.topology.edge_children + E,
              workspace_.edge_children);
  }
  return FactorStatus::SUCCESS;
}

LQR::FactorStatus LQR::factor_with_status() {
  if (traversal_status_ != FactorStatus::SUCCESS) return traversal_status_;
  const Topology &t = input_.topology;
  const BlockSizes bs(input_.dimensions, t);
  const int N = t.num_nodes(), E = t.num_edges;
  auto &w = *workspace_.device;
  gather(input_.Q, N, bs.nn, w.in[0]);
  gather(input_.M, E, bs.nm, w.in[1]);
  gather(input_.R, E, bs.mm, w.in[2]);
  gather(input_.A, E, bs.a, w.in[5]);
  gather(input_.B, E, bs.b, w.in[6]);
  gather(input_.delta, N, bs.n, w.in[8]);
  const sipoc_lqr_input in{w.in[0].data(), w.in[1].data(), w.in[2].data(), nullptr, nullptr,
                           w.in[5].data(), w.in[6].data(), nullptr,        w.in[8].data()};
  int status = 0;
  if (sipoc_lqr_factor_host(w.engine, &in, &status) != SIPOC_OK)
    return FactorStatus::INVALID_TOPOLOGY;
  return static_cast<FactorStatus>(status);
}

bool LQR::factor() { return factor_with_status() == FactorStatus::SUCCESS; }

void LQR::solve(Output &output) {
  const Topology &t = input_.topology;
  const BlockSizes bs(input_.dimensions, t);
  const int N = t.num_nodes(), E = t.num_edges;
  if (workspace_.device == nullptr) return;
  auto &w = *workspace_.device;
  gather(input_.q, N, bs.n, w.in[3]);
  gather(input_.r, E, bs.m, w.in[4]);
  gather(input_.c, N, bs.n, w.in[7]);
  const sipoc_lqr_input in{nullptr, nullptr, nullptr, w.in[3].data(), w.in[4].data(),
                           nullptr, nullptr, w.in[7].data(), nullptr};
  const sipoc_lqr_output out{w.out[0].data(), w.out[1].data(), w.out[2].data()};
  if ((w.last_error = sipoc_lqr_solve_host(w.engine, &in, &out)) != SIPOC_OK) return;
  scatter(w.out[0], output.x, N, bs.n);
  scatter(w.out[1], output.u, E, bs.m);
  scatter(w.out[2], output.y, N, bs.n);
}

// ---- BatchedLQR --------------------------------------------------------------------------
BatchedLQR::BatchedLQR(const Dimensions &d, const Topology &t, int64_t batch, int device) {
  const sipoc_structure s = describe(d, t, batch, device);
  if (sipoc_create(&s, &engine_) != SIPOC_OK) {
    engine_ = nullptr;
    status_ = LQR::FactorStatus::INVALID_TOPOLOGY;
  }
}
BatchedLQR::~BatchedLQR() {
  if (engine_ != nullptr) sipoc_destroy(engine_);
}
int64_t BatchedLQR::batch_stride() const { return sipoc_batch_stride(engine_); }

namespace {
sipoc_lqr_input to_abi(const BatchedLQR::DeviceInput &i) {
  return sipoc_lqr_input{i.Q, i.M, i.R, i.q, i.r, i.A, i.B, i.c, i.delta};
}
}  // namespace

bool BatchedLQR::factor_with_status(const DeviceInput &in, int *status, void *stream) {
  const sipoc_lqr_input a = to_abi(in);
  return engine_ != nullptr && sipoc_lqr_factor(engine_, &a, status, stream) == SIPOC_OK;
}
bool BatchedLQR::solve(const DeviceInput &in, const DeviceOutput &out, void *stream) {
  const sipoc_lqr_input a = to_abi(in);
  const sipoc_lqr_output o{out.x, out.u, out.y};
  return engine_ != nullptr && sipoc_lqr_solve(engine_, &a, &o, stream) == SIPOC_OK;
}
bool BatchedLQR::factor_solve(const DeviceInput &in, const DeviceOutput &out, int *status,
                              void *stream) {
  const sipoc_lqr_input a = to_abi(in);
  const sipoc_lqr_output o{out.x, out.u, out.y};
  return engine_ != nullptr &&
         sipoc_lqr_factor_solve(engine_, &a, &o, status, stream) == SIPOC_OK;
}

bool BatchedLQR::factor_solve_policy(const DeviceInput &in, const DeviceOutput &out,
                                     const DevicePolicy &policy, int *status, void *stream) {
  const sipoc_lqr_input a = to_abi(in);
  const sipoc_lqr_output o{out.x, out.u, out.y};
  const sipoc_lqr_policy p{policy.K, policy.k, policy.V, policy.v};
  return engine_ != nullptr &&
         sipoc_lqr_factor_solve_policy(engine_, &a, &o, &p, status, stream) == SIPOC_OK;
}

}  // namespace sip::optimal_control
