// Whole-encoder entry points for the chem GIN stack (chem/model.py:255-290 with gnn_type="gin", JK="last",
// drop_ratio=0): ONE call enqueues graph preparation, the atom embedding and all L x (aggregate -> MLP ->
// BatchNorm[-> ReLU]) layers; a second call enqueues the whole backward.  This is what GNN.forward binds
// to, so a training step crosses the Python/C boundary twice instead of ~60 times, and the inter-layer
// BatchNorm + ReLU never makes a pass of its own: layer l only accumulates the batch statistics and layer
// l+1's gather applies scale/shift/ReLU while it loads the rows (pgnn_aggregate_fwd's in_scale/in_shift).
//
// Parameters arrive as a host array of device pointers in a fixed order (PGNN_CHEM_GIN_* below), gradients
// leave in ONE flat fp32 buffer with the library-defined layout of pgnn_chem_gin_grad_offsets, which is
// also the buffer the data-parallel all-reduce runs on.
#include "common.cuh"

#include <cstdlib>
#include <map>
#include <mutex>
#include <vector>

int pgnn_internal_edge_table_bwd2(const float* S, int Q, const float* g, int64_t ldg, int64_t g_off, int64_t n, int C, float* gT,
                                  int64_t ldt, float* gT2, int q_split, cudaStream_t st);
int pgnn_internal_aggregate_fwd(const float* x, int64_t ldx, const float* in_scale, const float* in_shift, int in_relu,
                                int64_t num_nodes, int64_t C, const int32_t* rowptr_t, const int32_t* nbr_t, int mode, const float* dinv,
                                const float* S, int64_t Q, const float* T, const float* T2, int q_split, int64_t edge_off, float* out,
                                int64_t ldo, cudaStream_t st, const PgnnBnFold* fold);

int pgnn_tma_gin_gather_gemm(const float* x, int64_t ldx, const float* in_scale, const float* in_shift, const PgnnBnFold* fold, int in_relu,
                             const int32_t* rowptr_t, const int32_t* nbr_t, const float* S, int Q, const float* T, const float* T2,
                             int q_split, float* aggr, int64_t lda, const float* W, const float* bias, int relu, float* z1, int64_t ldz,
                             int64_t M, int64_t N, int64_t K, unsigned int* tile_ctr, cudaStream_t st);
int pgnn_internal_chem_onehot(const int64_t* x, int64_t n, int rows1, int rows2, float* onehot, int64_t ld, cudaStream_t st);

int pgnn_tc_linear_fwd(const float*, int64_t, const float*, const float*, int64_t, int64_t, int64_t, int, float*, int64_t,
                       cudaStream_t, const PgnnGemmHooks*);
int pgnn_tc_linear_bwd_x(const float*, int64_t, const float*, int64_t, int64_t, int64_t, const float*, int64_t, float*, int64_t,
                         cudaStream_t, const PgnnGemmHooks*);
int pgnn_tc_linear_bwd_w(const float*, int64_t, const float*, int64_t, int64_t, int64_t, int64_t, float*, float*, cudaStream_t);
int pgnn_tc_linear_bwd_w_ws(const float* gy, int64_t ldgy, const float* x, int64_t ldx, int64_t M, int64_t N, int64_t K, float* gw,
                            float* gb, float* partials, int64_t partial_floats, cudaStream_t st);
int pgnn_tc_linear_bwd_w_ws2(const float* gy, int64_t ldgy, const float* x, int64_t ldx, int64_t M, int64_t N, int64_t K, float* gw,
                             float* gb, float* partials, int64_t partial_floats, cudaStream_t st, bool in_kernel_fold_ok);
int64_t pgnn_tc_wgrad_workspace_floats(int64_t M, int64_t N, int64_t K);
int pgnn_tc_linear_bwd_x_wt(const float* gy, int64_t ldgy, const float* wT, int64_t M, int64_t N, int64_t K, const float* relu_src,
                            int64_t ldr, float* gx, int64_t ldgx, cudaStream_t st, const PgnnGemmHooks* hooks);
int pgnn_internal_transpose_batch(int count, const float* const* in, float* const* out, const int* rows, const int* cols,
                                  cudaStream_t st);
int pgnn_internal_bn_apply_fold(const float* x, int64_t ldx, int64_t M, int64_t C, const PgnnBnFold& fold, int relu, float* y,
                                int64_t ldy, cudaStream_t st);
int pgnn_internal_bn_bwd_colsum(const float* gy, int64_t ldgy, const float* x, int64_t ldx, int64_t M, int64_t C, const float* gamma,
                                const float* beta, const float* save_mean, const float* save_invstd, int relu, float* gx,
                                int64_t ldgx, float* ggamma, float* gbeta, float* colsum_part, int* parts, void* workspace, cudaStream_t st);
int64_t pgnn_internal_bn_colsum_parts(int64_t M);
int pgnn_internal_fold_colsums(const float* const* part, const int* parts, float* const* out, int count, int64_t C, cudaStream_t st);

namespace {

// order of the parameter pointer table and of the flat gradient layout
enum { P_XEMB1 = 0, P_XEMB2 = 1, P_LAYER0 = 2 };
enum { L_W1 = 0, L_B1, L_W2, L_B2, L_ET1, L_ET2, L_GAMMA, L_BETA, L_COUNT };

constexpr int kAtomRows = 120, kChiralRows = 3;   // chem/model.py:9-10
constexpr int kOneHotLd = 124;                    // kAtomRows + kChiralRows padded to a multiple of 4

struct Carve {
  char* base;
  int64_t off = 0;
  explicit Carve(void* b) : base(reinterpret_cast<char*>(b)) {}
  template <typename T>
  T* take(int64_t count) {
    T* p = reinterpret_cast<T*>(base + off);
    off += align_up(count * (int64_t)sizeof(T), 256);
    return p;
  }
};

struct Ws {
  int32_t *rowptr_t, *rowptr_s, *nbr_t, *eid_t, *nbr_s, *eid_s;
  float *S, *h0, *scale, *shift, *mean, *invstd;  // scale/shift/mean/invstd: [L, D]
  float* onehot;                                   // [N, kOneHotLd]: atom-code one-hot rows (embedding gradient as a GEMM)
  double* bn_acc;                                  // [L][2][D] fp64 BatchNorm sums of the forward
  unsigned int* tile_ctr;                          // [L][tiles] arrival counters of the fused gather + GEMM1 kernel (zeroed per forward)
  int64_t tiles;
  float *aggr, *z1, *z2;                           // [L, N, D], [L, N, 2D], [L, N, D]
  float *gh, *gz2, *gz1, *gaggr;                   // backward temporaries
  float* wT;                                       // [L][2][2D*D]: mlp.0.weight^T, mlp.2.weight^T (dgrad B operands)
  float* wpart;                                    // split-K partial tiles of one wgrad
  float* bn_part;                                  // [L][bn_parts][D] row-block partials of the mlp.2.bias gradients
  int64_t bn_parts;
  int64_t wpart_floats;
  void* scratch;                                   // bucket / BatchNorm scratch
  int64_t scratch_bytes, total;
};

Ws carve(void* base, int64_t N, int64_t E, int64_t L, int64_t D) {
  Carve c(base);
  Ws w;
  const int64_t e1 = E > 0 ? E : 1;
  w.rowptr_t = c.take<int32_t>(N + 1);
  w.rowptr_s = c.take<int32_t>(N + 1);
  w.nbr_t = c.take<int32_t>(e1);
  w.eid_t = c.take<int32_t>(e1);
  w.nbr_s = c.take<int32_t>(e1);
  w.eid_s = c.take<int32_t>(e1);
  w.S = c.take<float>(N * 9);
  w.h0 = c.take<float>(N * D);
  w.onehot = c.take<float>(N * kOneHotLd);
  w.bn_acc = c.take<double>(L * 2 * D);
  w.tiles = ceil_div(N > 0 ? N : 1, 128);
  w.tile_ctr = c.take<unsigned int>(L * w.tiles);
  w.scale = c.take<float>(L * D);
  w.shift = c.take<float>(L * D);
  w.mean = c.take<float>(L * D);
  w.invstd = c.take<float>(L * D);
  w.aggr = c.take<float>(L * N * D);
  w.z1 = c.take<float>(L * N * 2 * D);
  w.z2 = c.take<float>(L * N * D);
  w.gh = c.take<float>(N * D);
  w.gz2 = c.take<float>(2 * N * D);       // two copies each: layer l's weight-gradient GEMMs (side stream) may still read
  w.gz1 = c.take<float>(2 * N * 2 * D);   // them while layer l-1's backward writes the other copy
  w.gaggr = c.take<float>(N * D);
  w.wT = c.take<float>(L * 4 * D * D);
  w.wpart_floats = pgnn_tc_wgrad_workspace_floats(N, 2 * D, D);  // both MLP weight gradients have 2D*D elements
  {
    const int64_t e = pgnn_tc_wgrad_workspace_floats(N, 123, D);  // the embedding tables' gradient as a GEMM
    if (e > w.wpart_floats) w.wpart_floats = e;
  }
  w.wpart = c.take<float>(w.wpart_floats);
  w.bn_parts = pgnn_internal_bn_colsum_parts(N);
  w.bn_part = c.take<float>(L * w.bn_parts * D);
  int64_t sb = pgnn_graph_prep_workspace_bytes(N, E);
  const int64_t bb = pgnn_bn_workspace_bytes(N > 0 ? N : 1, D);
  if (bb > sb) sb = bb;
  w.scratch_bytes = sb;
  w.scratch = c.take<char>(sb);
  w.total = c.off;
  return w;
}

// Weight-gradient GEMMs on a side stream.  Per layer the critical path of the backward is BatchNorm-bwd -> dgrad2 -> dgrad1 ->
// transpose gather -> (next layer); wgrad2 (needs gz2, z1) and wgrad1 (needs gz1, aggr) only feed the gradient buffer.  On
// their own stream they run under the next layer's BatchNorm sweeps and gathers (LSU / L2-bound kernels that leave the tensor
// pipe and most of shared memory idle) instead of in front of them.  Ordering is by events; gz2 / gz1 are double-buffered
// by layer parity so the main stream never overwrites an operand a pending wgrad still reads.  PGNN_WGRAD_STREAM=0 disables.
struct SideCtx {
  cudaStream_t side = nullptr;
  cudaEvent_t gz2_ready[2] = {}, gz1_ready[2] = {}, w2_done[2] = {}, w1_done[2] = {}, join = nullptr;
  bool ok = false;
};
SideCtx* side_ctx(cudaStream_t main_stream) {
  static std::mutex mu;
  static std::map<std::pair<int, cudaStream_t>, SideCtx*> all;
  static int enabled = -1;
  std::lock_guard<std::mutex> g(mu);
  if (enabled < 0) {
    const char* e = getenv("PGNN_WGRAD_STREAM");
    enabled = (e && e[0] == '0') ? 0 : 1;
  }
  // the per-kernel timing mode (pgnn_profile_enable) wants each kernel's own duration: no concurrent stream while it is on
  if (!enabled || g_pgnn_profile_on.load(std::memory_order_relaxed) != 0) return nullptr;
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess) return nullptr;
  auto key = std::make_pair(dev, main_stream);
  auto it = all.find(key);
  if (it != all.end()) return it->second->ok ? it->second : nullptr;
  SideCtx* c = new SideCtx();
  all[key] = c;
  bool ok = cudaStreamCreateWithFlags(&c->side, cudaStreamNonBlocking) == cudaSuccess;
  for (int i = 0; i < 2 && ok; ++i)
    ok = cudaEventCreateWithFlags(&c->gz2_ready[i], cudaEventDisableTiming) == cudaSuccess &&
         cudaEventCreateWithFlags(&c->gz1_ready[i], cudaEventDisableTiming) == cudaSuccess &&
         cudaEventCreateWithFlags(&c->w2_done[i], cudaEventDisableTiming) == cudaSuccess &&
         cudaEventCreateWithFlags(&c->w1_done[i], cudaEventDisableTiming) == cudaSuccess;
  ok = ok && cudaEventCreateWithFlags(&c->join, cudaEventDisableTiming) == cudaSuccess;
  if (!ok) cudaGetLastError();
  c->ok = ok;
  return ok ? c : nullptr;
}

// PGNN_EMBED_GEMM=0: embedding-table gradient through the vector-atomics kernel instead of the one-hot GEMM (development switch)
inline bool embed_gemm_enabled() {
  static int v = -1;
  if (v < 0) {
    const char* e = getenv("PGNN_EMBED_GEMM");
    v = (e && e[0] == '0') ? 0 : 1;
  }
  return v == 1;
}

#define TRY(call)                 \
  do {                            \
    int rc__ = (call);            \
    if (rc__ != PGNN_OK) return rc__; \
  } while (0)

}  // namespace

extern "C" {

int64_t pgnn_chem_gin_num_params(int64_t L) { return L < 1 ? PGNN_EINVAL : 2 + L_COUNT * L; }

int pgnn_chem_gin_grad_offsets(int64_t L, int64_t D, int64_t* offsets /*host [num_params + 1]*/) {
  PGNN_CHECK_ARG(L >= 1 && D > 0 && offsets);
  int64_t o = 0, i = 0;
  offsets[i++] = o; o += 120 * D;  // x_embedding1.weight
  offsets[i++] = o; o += 3 * D;    // x_embedding2.weight
  for (int64_t l = 0; l < L; ++l) {
    offsets[i++] = o; o += 2 * D * D;  // mlp.0.weight [2D, D]
    offsets[i++] = o; o += 2 * D;      // mlp.0.bias
    offsets[i++] = o; o += 2 * D * D;  // mlp.2.weight [D, 2D]
    offsets[i++] = o; o += D;          // mlp.2.bias
    offsets[i++] = o; o += 6 * D;      // edge_embedding1.weight
    offsets[i++] = o; o += 3 * D;      // edge_embedding2.weight
    offsets[i++] = o; o += D;          // batch_norms.l.weight
    offsets[i++] = o; o += D;          // batch_norms.l.bias
  }
  offsets[i] = o;
  return PGNN_OK;
}

int64_t pgnn_chem_gin_workspace_bytes(int64_t N, int64_t E, int64_t L, int64_t D) {
  if (N < 0 || E < 0 || L < 1 || D <= 0) return PGNN_EINVAL;
  return carve(nullptr, N, E, L, D).total;
}

// Development / test aid: byte offsets inside the workspace of the saved activations a test needs to reconstruct the
// ReLU decisions the encoder actually took: out[0] = z1 (post-ReLU hidden activations, [L][N][2D]), out[1] = z2 (pre-BatchNorm
// layer outputs, [L][N][D]), out[2] = BatchNorm batch mean [L][D], out[3] = invstd [L][D].
int pgnn_chem_gin_debug_layout(int64_t N, int64_t E, int64_t L, int64_t D, int64_t* out4) {
  PGNN_CHECK_ARG(N >= 0 && E >= 0 && L >= 1 && D > 0 && out4);
  char* base = reinterpret_cast<char*>(0x1000);  // carve() only does pointer arithmetic
  Ws w = carve(base, N, E, L, D);
  out4[0] = reinterpret_cast<char*>(w.z1) - base;
  out4[1] = reinterpret_cast<char*>(w.z2) - base;
  out4[2] = reinterpret_cast<char*>(w.mean) - base;
  out4[3] = reinterpret_cast<char*>(w.invstd) - base;
  return PGNN_OK;
}

int pgnn_chem_gin_forward(const void* const* params, void* const* bn_running_mean, void* const* bn_running_var,
                          void* const* bn_num_batches_tracked, const int64_t* x, const int64_t* edge_index,
                          const int64_t* edge_attr, int64_t N, int64_t E, int64_t L, int64_t D, int training, float momentum, float eps,
                          int precision, float* node_rep, int64_t ld_out, void* workspace, int64_t workspace_bytes, void* stream) {
  PGNN_CHECK_ARG(N >= 0 && E >= 0 && L >= 1 && D > 0 && D % 4 == 0 && params && bn_running_mean && bn_running_var && workspace);
  PGNN_CHECK_ARG(N == 0 || (x && node_rep));
  if (workspace_bytes < pgnn_chem_gin_workspace_bytes(N, E, L, D)) return PGNN_EWORKSPACE;
  if (N == 0) return PGNN_OK;
  if (training && N < 1) return PGNN_EINVAL;
  Ws w = carve(workspace, N, E, L, D);
  if (precision == 1) PGNN_CUDA(cudaMemsetAsync(w.tile_ctr, 0, sizeof(unsigned int) * L * w.tiles, as_stream(stream)));
  TRY(pgnn_graph_prep(edge_index, E, N, w.rowptr_t, w.nbr_t, w.eid_t, w.rowptr_s, w.nbr_s, w.eid_s, w.scratch, w.scratch_bytes, stream));
  TRY(pgnn_chem_edge_summary(edge_attr, w.rowptr_t, w.nbr_t, w.eid_t, N, PGNN_AGG_SUM, nullptr, w.S, stream));
  TRY(pgnn_chem_embed_fwd(x, (const float*)params[P_XEMB1], kAtomRows, (const float*)params[P_XEMB2], kChiralRows, N, D, w.h0, D, stream));
  if (training && precision == 1) TRY(pgnn_internal_chem_onehot(x, N, kAtomRows, kChiralRows, w.onehot, kOneHotLd, as_stream(stream)));
  const float* h = w.h0;            // input rows of the current layer (pre-affine)
  const float *in_scale = nullptr, *in_shift = nullptr;
  PgnnBnFold fold;                  // pending BatchNorm finalisation of the previous layer (folded into this layer's gather)
  bool have_fold = false;
  double* const bn_acc = w.bn_acc;  // [L][2][D] fp64 sums
  for (int64_t l = 0; l < L; ++l) {
    const void* const* p = params + P_LAYER0 + l * L_COUNT;
    float* aggr = w.aggr + l * N * D;
    float* z1 = w.z1 + l * N * 2 * D;
    float* z2 = w.z2 + l * N * D;
    const bool last = (l == L - 1);
    // gather + GEMM1.  Tensor path: ONE kernel (k_gin_gather_gemm): the column tiles of a row tile form a cluster that gathers the
    // tile's rows together, then runs the GEMM on them (`aggr` is stored once: the backward's weight-gradient GEMM reads it).
    int rc_f = PGNN_EUNSUPPORTED;
    if (precision == 1)
      rc_f = pgnn_tma_gin_gather_gemm(h, D, in_scale, in_shift, have_fold ? &fold : nullptr, in_scale != nullptr || have_fold, w.rowptr_t,
                                      w.nbr_t, w.S, 9, (const float*)p[L_ET1], (const float*)p[L_ET2], 6, aggr, D,
                                      (const float*)p[L_W1], (const float*)p[L_B1], 1, z1, 2 * D, N, 2 * D, D, w.tile_ctr + l * w.tiles, as_stream(stream));
    if (rc_f == PGNN_EUNSUPPORTED) {
      TRY(pgnn_internal_aggregate_fwd(h, D, in_scale, in_shift, in_scale != nullptr || have_fold, N, D, w.rowptr_t, w.nbr_t, PGNN_AGG_SUM,
                                      nullptr, w.S, 9, (const float*)p[L_ET1], (const float*)p[L_ET2], 6, 0, aggr, D, as_stream(stream),
                                      have_fold ? &fold : nullptr));
      TRY(pgnn_linear_fwd(aggr, D, (const float*)p[L_W1], (const float*)p[L_B1], N, 2 * D, D, 1, z1, 2 * D, precision, stream));
    } else if (rc_f != PGNN_OK) {
      return rc_f;
    }
    have_fold = false;
    // GEMM2; on the tensor path its epilogue also accumulates the BatchNorm batch statistics of z2 (fp64 atomics)
    bool stats_fused = false;
    double* acc = bn_acc + l * 2 * D;
    if (training && precision == 1) {
      PGNN_CUDA(cudaMemsetAsync(acc, 0, sizeof(double) * 2 * D, as_stream(stream)));
      PgnnGemmHooks hk;
      hk.stats = acc;
      const int rc = pgnn_tc_linear_fwd(z1, 2 * D, (const float*)p[L_W2], (const float*)p[L_B2], N, D, 2 * D, 0, z2, D, as_stream(stream), &hk);
      if (rc == PGNN_OK) stats_fused = true;
      else if (rc != PGNN_EUNSUPPORTED) return rc;
    }
    if (!stats_fused)
      TRY(pgnn_linear_fwd(z1, 2 * D, (const float*)p[L_W2], (const float*)p[L_B2], N, D, 2 * D, 0, z2, D, precision, stream));
    if (training && stats_fused) {
      // no finalize launch: the consumer (next layer's gather, or the final apply) derives scale/shift from the sums
      fold = PgnnBnFold{};
      fold.acc = acc; fold.gamma = (const float*)p[L_GAMMA]; fold.beta = (const float*)p[L_BETA];
      fold.running_mean = (float*)bn_running_mean[l]; fold.running_var = (float*)bn_running_var[l];
      fold.nbt = bn_num_batches_tracked ? (int64_t*)bn_num_batches_tracked[l] : nullptr;
      fold.save_mean = w.mean + l * D; fold.save_invstd = w.invstd + l * D;
      fold.momentum = momentum; fold.eps = eps; fold.set_rows((int)N);
      if (last) {
        TRY(pgnn_internal_bn_apply_fold(z2, D, N, D, fold, 0, node_rep, ld_out, as_stream(stream)));
      } else {
        have_fold = true;
      }
      h = z2;
      in_scale = in_shift = nullptr;
    } else if (training) {
      // statistics only for inner layers (applied on load by the next gather); the last layer materialises node_rep
      TRY(pgnn_bn_fwd_train(z2, D, N, D, (const float*)p[L_GAMMA], (const float*)p[L_BETA], (float*)bn_running_mean[l],
                            (float*)bn_running_var[l], bn_num_batches_tracked ? (int64_t*)bn_num_batches_tracked[l] : nullptr, momentum,
                            eps, 0, last ? node_rep : nullptr, ld_out, w.mean + l * D, w.invstd + l * D, w.scale + l * D,
                            w.shift + l * D, w.scratch, w.scratch_bytes, stream));
      h = z2;
      in_scale = w.scale + l * D;
      in_shift = w.shift + l * D;
    } else {
      // eval: plain BN(+ReLU) pass with the running statistics, ping-ponging between two spare buffers
      float* y = last ? node_rep : ((l & 1) ? w.gz2 : w.gaggr);
      TRY(pgnn_bn_fwd_eval(z2, D, N, D, (const float*)p[L_GAMMA], (const float*)p[L_BETA], (const float*)bn_running_mean[l],
                           (const float*)bn_running_var[l], eps, !last, y, last ? ld_out : D, stream));
      h = y;
      in_scale = in_shift = nullptr;
    }
  }
  return PGNN_OK;
}

int pgnn_chem_gin_backward(const void* const* params, const float* g_node_rep, int64_t ldg, const int64_t* x, int64_t N, int64_t E,
                           int64_t L, int64_t D, int precision, float* grads, void* workspace, int64_t workspace_bytes,
                           void* stream) {
  PGNN_CHECK_ARG(N >= 0 && E >= 0 && L >= 1 && D > 0 && D % 4 == 0 && params && grads && workspace);
  if (workspace_bytes < pgnn_chem_gin_workspace_bytes(N, E, L, D)) return PGNN_EWORKSPACE;
  int64_t off[2 + L_COUNT * 64 + 1];
  PGNN_CHECK_ARG(L <= 64);
  pgnn_chem_gin_grad_offsets(L, D, off);
  cudaStream_t st = as_stream(stream);
  if (N == 0) {
    PGNN_CUDA(cudaMemsetAsync(grads, 0, sizeof(float) * off[2 + L_COUNT * L], st));
    return PGNN_OK;
  }
  PGNN_CHECK_ARG(g_node_rep && x);
  Ws w = carve(workspace, N, E, L, D);
  // transposed copies of the 2L MLP weights: with them every dgrad has both operands reduction-contiguous and runs on
  // the TMA-staged GEMM (dense_tma.cu) instead of the cp.async one
  bool have_wT = false;
  if (precision == 1 && 2 * L <= 32) {
    const float* in[32];
    float* out[32];
    int rows[32], cols[32];
    for (int64_t l = 0; l < L; ++l) {
      const void* const* p = params + P_LAYER0 + l * L_COUNT;
      in[2 * l] = (const float*)p[L_W1];     out[2 * l] = w.wT + (2 * l) * 2 * D * D;     rows[2 * l] = (int)(2 * D); cols[2 * l] = (int)D;
      in[2 * l + 1] = (const float*)p[L_W2]; out[2 * l + 1] = w.wT + (2 * l + 1) * 2 * D * D; rows[2 * l + 1] = (int)D; cols[2 * l + 1] = (int)(2 * D);
    }
    const int rc = pgnn_internal_transpose_batch((int)(2 * L), in, out, rows, cols, st);
    if (rc == PGNN_OK) have_wT = true;
    else if (rc != PGNN_EUNSUPPORTED) return rc;
  }
  const float* gy = g_node_rep;
  int64_t ldgy = ldg;
  SideCtx* sc = precision == 1 ? side_ctx(st) : nullptr;
  cudaStream_t wst = sc ? sc->side : st;   // the stream of the weight-gradient GEMMs
  std::vector<const float*> b2_part;   // mlp.2.bias gradients: row-block partials, folded in block order after the loop
  std::vector<int> b2_parts;
  std::vector<float*> b2_out;
  for (int64_t l = L - 1; l >= 0; --l) {
    const void* const* p = params + P_LAYER0 + l * L_COUNT;
    const int64_t* o = off + P_LAYER0 + l * L_COUNT;
    const float* aggr = w.aggr + l * N * D;
    const float* z1 = w.z1 + l * N * 2 * D;
    const float* z2 = w.z2 + l * N * D;
    const bool last = (l == L - 1);
    const int par = (int)(l & 1);
    float* gz2 = w.gz2 + (sc ? par * N * D : 0);
    float* gz1 = w.gz1 + (sc ? par * N * 2 * D : 0);
    // BatchNorm (+ReLU mask recomputed from z2) backward; the same pass leaves colsum(gz2) = gradient of mlp.2.bias
    if (sc) PGNN_CUDA(cudaStreamWaitEvent(st, sc->w2_done[par], 0));  // layer l+2's wgrad2 has finished reading this copy
    float* b2p = w.bn_part + l * w.bn_parts * D;
    int b2n = 0;
    TRY(pgnn_internal_bn_bwd_colsum(gy, ldgy, z2, D, N, D, (const float*)p[L_GAMMA], (const float*)p[L_BETA], w.mean + l * D,
                                    w.invstd + l * D, !last, gz2, D, grads + o[L_GAMMA], grads + o[L_BETA], b2p, &b2n, w.scratch, st));
    b2_part.push_back(b2p);
    b2_parts.push_back(b2n);
    b2_out.push_back(grads + o[L_B2]);
    // MLP backward.  On the tensor path the dgrad epilogues carry the column reductions that would otherwise be
    // passes of their own: colsum(gz1) = gradient of mlp.0.bias, and S^T gaggr = gradient of the two bond tables.
    bool fused = false;
    if (precision == 1) {
      if (sc) {
        PGNN_CUDA(cudaEventRecord(sc->gz2_ready[par], st));
        PGNN_CUDA(cudaStreamWaitEvent(wst, sc->gz2_ready[par], 0));
      }
      int rc = pgnn_tc_linear_bwd_w_ws2(gz2, D, z1, 2 * D, N, D, 2 * D, grads + o[L_W2], nullptr, w.wpart, w.wpart_floats, wst, sc == nullptr);
      if (rc == PGNN_OK) {
        if (sc) {
          PGNN_CUDA(cudaEventRecord(sc->w2_done[par], wst));
          PGNN_CUDA(cudaStreamWaitEvent(st, sc->w1_done[par], 0));  // layer l+2's wgrad1 has finished reading gz1[par]
        }
        PGNN_CUDA(cudaMemsetAsync(grads + o[L_B1], 0, sizeof(float) * 2 * D, st));
        PgnnGemmHooks h1;
        h1.colsum = grads + o[L_B1];
        rc = have_wT ? pgnn_tc_linear_bwd_x_wt(gz2, D, w.wT + (2 * l + 1) * 2 * D * D, N, D, 2 * D, z1, 2 * D, gz1, 2 * D, st, &h1)
                     : PGNN_EUNSUPPORTED;
        if (rc == PGNN_EUNSUPPORTED)
          rc = pgnn_tc_linear_bwd_x(gz2, D, (const float*)p[L_W2], N, D, 2 * D, z1, 2 * D, gz1, 2 * D, st, &h1);
        if (rc != PGNN_OK) return rc;
        if (sc) {
          PGNN_CUDA(cudaEventRecord(sc->gz1_ready[par], st));
          PGNN_CUDA(cudaStreamWaitEvent(wst, sc->gz1_ready[par], 0));
        }
        rc = pgnn_tc_linear_bwd_w_ws2(gz1, 2 * D, aggr, D, N, 2 * D, D, grads + o[L_W1], nullptr, w.wpart, w.wpart_floats, wst, sc == nullptr);
        if (rc != PGNN_OK) return rc;
        if (sc) PGNN_CUDA(cudaEventRecord(sc->w1_done[par], wst));
        PGNN_CUDA(cudaMemsetAsync(grads + o[L_ET1], 0, sizeof(float) * 9 * D, st));  // the two tables are adjacent in the layout
        PgnnGemmHooks h2;
        h2.S = w.S; h2.Q = 9; h2.gT = grads + o[L_ET1]; h2.gT2 = grads + o[L_ET2]; h2.q_split = 6; h2.ldt = D;
        rc = have_wT ? pgnn_tc_linear_bwd_x_wt(gz1, 2 * D, w.wT + (2 * l) * 2 * D * D, N, 2 * D, D, nullptr, 0, w.gaggr, D, st, &h2)
                     : PGNN_EUNSUPPORTED;
        if (rc == PGNN_EUNSUPPORTED)
          rc = pgnn_tc_linear_bwd_x(gz1, 2 * D, (const float*)p[L_W1], N, 2 * D, D, nullptr, 0, w.gaggr, D, st, &h2);
        if (rc != PGNN_OK) return rc;
        fused = true;
      } else if (rc != PGNN_EUNSUPPORTED) {
        return rc;
      }
    }
    if (!fused) {
      if (sc) {  // an unsupported shape on the tensor path: everything on the caller's stream from here on
        PGNN_CUDA(cudaEventRecord(sc->join, wst));
        PGNN_CUDA(cudaStreamWaitEvent(st, sc->join, 0));
      }
      TRY(pgnn_linear_bwd_w(gz2, D, z1, 2 * D, N, D, 2 * D, grads + o[L_W2], nullptr, precision, stream));
      TRY(pgnn_linear_bwd_x(gz2, D, (const float*)p[L_W2], N, D, 2 * D, z1, 2 * D, gz1, 2 * D, precision, stream));
      TRY(pgnn_linear_bwd_w(gz1, 2 * D, aggr, D, N, 2 * D, D, grads + o[L_W1], grads + o[L_B1], precision, stream));
      TRY(pgnn_linear_bwd_x(gz1, 2 * D, (const float*)p[L_W1], N, 2 * D, D, nullptr, 0, w.gaggr, D, precision, stream));
      // bond tables: gT = S^T gaggr, rows 0..5 -> edge_embedding1, 6..8 -> edge_embedding2
      PGNN_CUDA(cudaMemsetAsync(grads + o[L_ET1], 0, sizeof(float) * 9 * D, st));
      TRY(pgnn_internal_edge_table_bwd2(w.S, 9, w.gaggr, D, 0, N, (int)D, grads + o[L_ET1], D, grads + o[L_ET2], 6, st));
    }
    // transpose-graph gather: gradient w.r.t. this layer's input rows
    TRY(pgnn_aggregate_bwd(w.gaggr, D, N, D, w.rowptr_s, w.nbr_s, PGNN_AGG_SUM, nullptr, w.rowptr_t, w.gh, D, stream));
    gy = w.gh;
    ldgy = D;
  }
  if (sc) {  // the side stream's last wgrad (and its use of the split-K workspace) before the embedding GEMM and before returning
    PGNN_CUDA(cudaEventRecord(sc->join, wst));
    PGNN_CUDA(cudaStreamWaitEvent(st, sc->join, 0));
  }
  TRY(pgnn_internal_fold_colsums(b2_part.data(), b2_parts.data(), b2_out.data(), (int)b2_out.size(), D, st));
  // embedding tables: [120 + 3, D] = onehot^T . gh as a split-K weight-gradient GEMM (the two tables are adjacent in the flat
  // layout); the vector-atomics kernel remains the fallback (FFMA precision, TMA unavailable)
  int rc_e = PGNN_EUNSUPPORTED;
  if (precision == 1 && embed_gemm_enabled() && off[P_XEMB2] == off[P_XEMB1] + (int64_t)kAtomRows * D)
    rc_e = pgnn_tc_linear_bwd_w_ws(w.onehot, kOneHotLd, w.gh, D, N, kAtomRows + kChiralRows, D, grads + off[P_XEMB1], nullptr, w.wpart,
                                   w.wpart_floats, st);
  if (rc_e == PGNN_EUNSUPPORTED)
    rc_e = pgnn_chem_embed_bwd(x, w.gh, D, N, D, grads + off[P_XEMB1], kAtomRows, grads + off[P_XEMB2], kChiralRows, stream);
  return rc_e;
}

}  // extern "C"
