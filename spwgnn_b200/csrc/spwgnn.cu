// spwgnn.cu -- C ABI (include/spwgnn.h) and launch sequences of the SPWGNN B200 hot path.
// Build: nvcc -gencode arch=compute_100a,code=sm_100a -lineinfo -O3 --shared -Xcompiler -fPIC
#include "../../include/spwgnn.h"
#include "spw_common.cuh"
#include "spw_edges.cuh"
#include "spw_kernels.cuh"
#include "spw_tc.cuh"
#include "spw_rows_tc.cuh"
#include "spw_pipe_tc.cuh"
#include "spw_csl.cuh"
#include "spw_csl_kernels.cuh"
#include "spw_csl_wgrad.cuh"
#include "spw_small.cuh"
#include "spw_small_grad.cuh"
#include "spw_obj_grad.cuh"
#include "spw_rel_grad.cuh"
#include "spw_input_grad.cuh"

#include <stdarg.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <atomic>
#include <map>
#include <mutex>
#include <utility>
#include <string>
#include <vector>

using namespace spw;

// Tensor-core (tcgen05) kernels replace their FFMA counterparts in the GPU build; the host emulator
// build (tools/cuemu, test infrastructure) always uses the FFMA kernels.
#ifdef SPW_EMU
#define SPW_USE_TC 0
#elif !defined(SPW_USE_TC)
#define SPW_USE_TC 1
#endif

namespace {

// ---- launch accounting / per-kernel CUDA-event timing (bench.py: gpu_launches, roofline) -------
namespace prof {
std::atomic<long long> launches{0};
bool enabled = false;
#ifndef SPW_EMU
struct Rec { const char* name; cudaEvent_t a, b; };
std::vector<Rec> recs;
#endif
struct Scope {
  cudaStream_t st; bool on;
#ifndef SPW_EMU
  cudaEvent_t b;
#endif
  Scope(const char* name, cudaStream_t s) : st(s), on(enabled) {
    launches.fetch_add(1, std::memory_order_relaxed);
#ifndef SPW_EMU
    if (on) {
      Rec r; r.name = name;
      cudaEventCreate(&r.a); cudaEventCreate(&r.b);
      cudaEventRecord(r.a, st);
      b = r.b;
      recs.push_back(r);
    }
#else
    (void)name;
#endif
  }
  ~Scope() {
#ifndef SPW_EMU
    if (on) cudaEventRecord(b, st);
#endif
  }
};
}  // namespace prof
#define SPW_KLAUNCH(name, kern, grid, block, smem, st, ...) \
  do { prof::Scope _scope(name, st); SPW_LAUNCH(kern, grid, block, smem, st, __VA_ARGS__); } while (0)
// programmatic dependent launch (spw_common.cuh): only for kernels that call pdl_trigger() / pdl_wait()
#define SPW_KLAUNCH_PDL(name, kern, grid, block, smem, st, ...) \
  do { prof::Scope _scope(name, st); SPW_LAUNCH_PDL(kern, grid, block, smem, st, __VA_ARGS__); } while (0)

thread_local char g_err[512] = "";

int fail(int code, const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
  return code;
}

bool aligned16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15u) == 0; }

int check_launch(const char* what) {
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) return fail(SPW_ERR_LAUNCH, "%s: %s", what, cudaGetErrorString(e));
  return SPW_OK;
}

int num_sms() {       // SM count of the CURRENT device (cached per device id)
  static int sms[64] = {0};
  int dev = 0;
  cudaGetDevice(&dev);
  if (dev < 0 || dev >= 64) dev = 0;
  if (sms[dev] == 0) {
    int v = 0;
    cudaDeviceGetAttribute(&v, cudaDevAttrMultiProcessorCount, dev);
    sms[dev] = v > 0 ? v : 148;
  }
  return sms[dev];
}

// development switch: SPW_CSL=0 in the environment selects the round-1 data path (row-major activations)
bool use_csl() {
  static int v = -1;
  if (v < 0) { const char* e = getenv("SPW_CSL"); v = (e && e[0] == '0') ? 0 : 1; }
#if SPW_USE_TC
  return v != 0;
#else
  return false;
#endif
}

// development switch: SPW_PIPE=0 in the environment selects the round-1 (unpipelined) edge-step kernels
bool use_pipe() {
  static int v = -1;
  if (v < 0) { const char* e = getenv("SPW_PIPE"); v = (e && e[0] == '0') ? 0 : 1; }
  return v != 0;
}

constexpr int kMaxCtas = 160;
constexpr int kTN = 64;         // node-tile rows of k_linear (two CTAs per SM)   // upper bound on persistent-grid size used to size partial buffers

// ---- packed weight buffer -----------------------------------------------------------------------
enum PackId {
  P_RM1, P_RM2, P_RM3, P_W1A, P_W1B, P_W1C, P_W2, P_W3, P_V1A, P_V1B, P_V1C, P_V2P, P_OM1,
  P_RM1T, P_RM2T, P_RM3T, P_W1AT, P_W1BT, P_W1CT, P_W2T, P_W3T, P_V1AT, P_V1BT, P_V1CT, P_V2PT, P_OM1T,
  P_COUNT
};
struct PackShape { int Kp, ldw; };
// forward matrices [in][out]; transposed ones [out][in]
const PackShape kPackShape[P_COUNT] = {
    {152, 160}, {152, 160}, {152, 160}, {152, 160}, {100, 160}, {100, 160}, {152, 160}, {152, 128},
    {100, 128}, {100, 128}, {100, 128}, {100, 128}, {100, 128},
    {152, 160}, {152, 160}, {152, 160}, {152, 160}, {152, 128}, {152, 128}, {152, 160}, {100, 160},
    {100, 128}, {100, 128}, {100, 128}, {100, 128}, {100, 128}};

size_t align_up(size_t x, size_t a) { return (x + a - 1) / a * a; }

// ---- tensor-core B operands of the generic rows kernel (tc::k_rows_tc): hi at tcp[id], lo right behind it ----
enum TcId {
  T_OM1, T_RM1, T_RM2, T_RM3, T_W1A, T_W1B, T_W1C, T_W3, T_V1A, T_V1BC, T_V2P,
  T_V2PT, T_V1AT, T_V1BT, T_V1CT, T_W3T, T_W1BT, T_W1CT, T_OM1T, T_COUNT
};
struct TcShape { int ks, NB; };   // k-steps of 8 rows, MMA N
const TcShape kTcShape[T_COUNT] = {
    {13, 112}, {19, 160}, {19, 160}, {19, 160}, {19, 160}, {13, 160}, {13, 160}, {19, 112}, {13, 112}, {25, 112}, {13, 112},
    {13, 112}, {13, 112}, {13, 112}, {13, 112}, {13, 160}, {19, 112}, {19, 112}, {13, 112}};
inline size_t tc_floats(int id) { return (size_t)kTcShape[id].ks * 8 * kTcShape[id].NB; }

struct Layout {
  size_t pack[P_COUNT];
  size_t tcp[T_COUNT];
  size_t tcp2;                   // CTA-pair operands of the eight 150x150 relation-encoder matrices: 8 x (hi halves | lo halves)
  size_t QV;                     // q.V1a + c1, constant over the steps
  size_t Q1, Q, degf, A, PF, PL, W2hi, W2lo, W2Thi, W2Tlo, ENCT;   // ENCT: 4 x (hi, lo) transposed encoder operands
  size_t P, S, R, H2S, G, U;     // per-step arrays (training: 5 slots; inference: fewer)
  int slotsP, slotsSR, slotsN;   // number of step slots for P / (S,R) / (H2S,G,U)
  // backward
  size_t EB;                     // sign bits of the relation-encoder activations X0, X1, X2, C: 4 x [E][8] words
  size_t dU, dG, T, dS, dR, dH2S, DP, dQ, dQ1, dA, DH1, M2, M1, EX0, EX1, EX2, EC, GB, partE, partM, part0, partN;
  size_t total;   // floats
};

constexpr size_t kPartNodeElems = 160 * 160;   // >= (16*TA)*(16*TB) for every node-level wgrad config

Layout make_layout(int64_t n, int64_t E, int training) {
  Layout L;
  size_t off = 0;
  auto take = [&](size_t floats) { size_t o = off; off = align_up(off + floats, 64); return o; };
  for (int i = 0; i < P_COUNT; ++i) L.pack[i] = take((size_t)kPackShape[i].Kp * kPackShape[i].ldw);
  const size_t nt = (size_t)((E + kTME - 1) / kTME) + 1;
  L.W2hi = take(24320);
  L.W2lo = take(24320);
  L.W2Thi = take(24320);
  L.W2Tlo = take(24320);
  L.ENCT = take((size_t)8 * 24320);
  for (int i = 0; i < T_COUNT; ++i) L.tcp[i] = take(2 * tc_floats(i));
  L.tcp2 = take((size_t)8 * 4 * 19 * 8 * 80);
  L.Q1 = take(n * kDP);
  L.Q = take(n * kDP);
  L.QV = take(n * kDP);
  L.degf = take(n);
  L.A = take((size_t)E * kDEP + 8);
  L.PF = take(nt * kDEP);
  L.PL = take(nt * kDEP);
  L.slotsP = training ? 5 : 2;
  L.slotsSR = training ? 5 : 1;
  L.slotsN = training ? 5 : 1;
  L.P = take((size_t)L.slotsP * n * kDP);
  L.S = take((size_t)L.slotsSR * n * kDEP);
  L.R = take((size_t)L.slotsSR * n * kDEP);
  L.H2S = take((size_t)L.slotsN * n * kDEP);
  L.G = take((size_t)L.slotsN * n * kDP);
  L.U = take((size_t)L.slotsN * n * kDP);
  if (training) {
    L.dU = take((size_t)5 * n * kDP);
    L.dG = take((size_t)5 * n * kDP);
    L.T = take((size_t)4 * n * kDP);
    L.dS = take((size_t)4 * n * kDEP);
    L.dR = take((size_t)4 * n * kDEP);
    L.dH2S = take((size_t)n * kDEP);
    L.DP = take((size_t)n * kDP);
    L.dQ = take((size_t)n * kDP);
    L.dQ1 = take((size_t)n * kDP);
    L.dA = take((size_t)E * kDEP + 8);
    L.DH1 = take((size_t)E * kDEP + 8);
    L.M2 = take((size_t)SPW_N_STEPS * E * 8);      // relu bits of h2, 8 words per edge and step
    L.M1 = take((size_t)SPW_N_STEPS * E * 8);      // relu bits of h1 (tensor-core data-gradient epilogue)
    L.EX0 = take((size_t)E * kDEP + 8);            // relation-encoder activations kept for the backward pass
    L.EX1 = take((size_t)E * kDEP + 8);
    L.GB = take((size_t)E * kDEP + 8);             // second gradient buffer of the layer-by-layer encoder backward
    L.EX2 = take((size_t)E * kDEP + 8);
    L.EC = take((size_t)E * kDEP + 8);
    L.EB = take((size_t)4 * E * 8);
    L.partE = take((size_t)kMaxCtas * 2 * 160 * 128);
    L.partM = take((size_t)kMaxCtas * 4 * 160 * 160);
    L.part0 = take((size_t)2 * kMaxCtas * 3 * kDEP);
    L.partN = take((size_t)2 * kMaxCtas * kPartNodeElems);
  } else {
    L.dU = L.dG = L.T = L.dS = L.dR = L.dH2S = L.DP = L.dQ = L.dQ1 = L.dA = L.DH1 = L.M2 = L.M1 = L.EX0 = L.EX1 = L.EX2 = L.EC = L.GB = 0; L.EB = 0;
    L.partE = L.partM = L.part0 = L.partN = 0;
  }
  L.total = off;
  return L;
}

int check_params(const SpwParams* w, const char* what) {
  if (!w) return fail(SPW_ERR_BAD_ARG, "%s: null parameter struct", what);
  const float* const* p = reinterpret_cast<const float* const*>(w);
  for (int i = 0; i < 22; ++i)
    if (!p[i] || !aligned16(p[i])) return fail(SPW_ERR_BAD_ARG, "%s: tensor %d null or not 16-byte aligned", what, i);
  return SPW_OK;
}

int check_graph(const SpwGraph* g) {
  if (!g) return fail(SPW_ERR_BAD_ARG, "null graph");
  if (g->n_towers < 0 || g->n_nodes < 0 || g->n_edges < 0) return fail(SPW_ERR_BAD_ARG, "negative graph size");
  if (g->n_nodes > 0 && (!g->node_off || !g->in_off || !g->out_off)) return fail(SPW_ERR_BAD_ARG, "null graph offsets");
  if (g->n_edges > 0 && (!g->in_snd || !g->in_rcv || !g->out_pos)) return fail(SPW_ERR_BAD_ARG, "null graph edge arrays");
  return SPW_OK;
}

// opt-in dynamic shared memory of a kernel: set once per (device, kernel, size) -- a small training step is ~140 launches and
// the attribute call costs about as much as a launch
template <class K>
void set_smem(K kern, size_t bytes) {
#ifndef SPW_EMU
  static std::mutex mu;
  static std::map<std::pair<int, const void*>, size_t> done;
  int dev = 0;
  cudaGetDevice(&dev);
  const std::pair<int, const void*> key(dev, reinterpret_cast<const void*>(kern));
  std::lock_guard<std::mutex> lock(mu);
  auto it = done.find(key);
  if (it != done.end() && it->second >= bytes) return;
  done[key] = bytes;
#endif
  cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes);
}

// ---- launch helpers -----------------------------------------------------------------------------
int grid_for(int64_t items, int per_block) {
  int64_t b = (items + per_block - 1) / per_block;
  if (b < 1) b = 1;
  const int64_t cap = (int64_t)num_sms() * 8;
  return (int)(b < cap ? b : cap);
}

LinSeg seg(const float* X, int ldx, int K, const float* W) {
  LinSeg s; s.X = X; s.W = W; s.ldx = ldx; s.K = K; s.Kp = (K + 3) / 4 * 4; return s;
}

struct LinOpt {
  const float* bias = nullptr; const float* rowscale = nullptr; const float* addend = nullptr; int ld_add = 0;
  int act = 0; const float* mulsrc = nullptr; int ld_mul = 0; int mulmode = 0; int accumulate = 0;
  float post_scale = 1.f; uint32_t drop_thresh = 0; uint32_t drop_seed = 0; float drop_inv_keep = 1.f;
  int drop_stride = 128;         // dropout element index = row * drop_stride + column
  int ones_col = -1;             // tensor-core kernel only: Y[row][ones_col] = 1
  const char* tag = nullptr;     // profile name of the launch (default: the kernel's)
  const uint32_t* bits_in = nullptr;   // tensor-core kernel only: mulmode 3 multiplies by these mask bits ([M][8] words)
  uint32_t* bits_out = nullptr;        // tensor-core kernel only: sign bits of the result
};

// Y[M][ldy] (N valid columns) from up to 3 (X, W) segments; wide = 150-column output (CN = 5)
void launch_linear(cudaStream_t st, int M, int N, bool wide, int nseg, const LinSeg* segs, float* Y, int ldy,
                   const LinOpt& o) {
  if (M <= 0) return;
  LinArgs a;
  memset(&a, 0, sizeof(a));
  a.M = M; a.nseg = nseg; a.N = N;
  size_t xfloats = 0;
  for (int s = 0; s < nseg; ++s) { a.seg[s] = segs[s]; xfloats += (size_t)kTN * segs[s].Kp; }
  a.bias = o.bias; a.rowscale = o.rowscale; a.addend = o.addend; a.ld_add = o.ld_add; a.act = o.act;
  a.mulsrc = o.mulsrc; a.ld_mul = o.ld_mul; a.mulmode = o.mulmode; a.Y = Y; a.ldy = ldy; a.accumulate = o.accumulate;
  a.post_scale = o.post_scale; a.drop_thresh = o.drop_thresh; a.drop_seed = o.drop_seed; a.drop_inv_keep = o.drop_inv_keep;
  // rows per tile: the candidate that minimises (rounds x rows) for a grid of two CTAs per SM (wave quantisation)
  const int cap = 2 * num_sms();
  int best_tm = 64;
  long best_cost = -1;
  for (int tm = 64; tm >= 32; tm -= 8) {
    const long nt = (M + tm - 1) / tm;
    const long rounds = (nt + cap - 1) / cap;
    const long cost = rounds * (tm + 6);          // +6: per-tile fixed overhead in row units
    if (best_cost < 0 || cost < best_cost) { best_cost = cost; best_tm = tm; }
  }
  const int ntiles = (M + best_tm - 1) / best_tm;
  const int grid = ntiles < cap ? ntiles : cap;
  size_t xf = 0;
  for (int s = 0; s < nseg; ++s) xf += (size_t)best_tm * segs[s].Kp;
  const size_t smem = (xf + 2 * kKT * (wide ? kLdwE : kLdwP)) * sizeof(float);
#define SPW_LIN_CASE(TMV)                                                                                   \
  case TMV:                                                                                                 \
    if (wide) { auto kern = k_linear<5, TMV>; set_smem(kern, smem); SPW_KLAUNCH("k_linear<5>", kern, dim3(grid), dim3(kThreads), smem, st, a); } \
    else { auto kern = k_linear<4, TMV>; set_smem(kern, smem); SPW_KLAUNCH("k_linear<4>", kern, dim3(grid), dim3(kThreads), smem, st, a); }      \
    break;
  switch (best_tm) {
    SPW_LIN_CASE(64)
    SPW_LIN_CASE(56)
    SPW_LIN_CASE(48)
    SPW_LIN_CASE(40)
    SPW_LIN_CASE(32)
  }
#undef SPW_LIN_CASE
}

// ---- one fused linear layer on rows: tensor cores (tc::k_rows_tc) in the GPU build, FFMA (k_linear) in the emulator ----
struct RowsSeg { const float* X; int ldx; int K; };
struct LinId { int tc; int pk0, pk1; };     // B operand of the tensor-core kernel; packed FFMA matrices of the segments

#if SPW_USE_TC
tc::RowsTcArgs make_rows_args(const float* Bhi, const float* Blo, int M, int N, int nseg, const RowsSeg* sg, float* Y, int ldy,
                              const LinOpt& o) {
  tc::RowsTcArgs a;
  memset(&a, 0, sizeof(a));
  a.M = M; a.nseg = nseg; a.N = N;
  int ktot = 0;
  for (int s = 0; s < nseg; ++s) { a.X[s] = sg[s].X; a.ldx[s] = sg[s].ldx; a.K[s] = sg[s].K; ktot += sg[s].K; }
  a.ks = (ktot + 7) / 8;
  a.Bhi = Bhi; a.Blo = Blo;
  a.bias = o.bias; a.rowscale = o.rowscale; a.addend = o.addend; a.ld_add = o.ld_add; a.act = o.act;
  a.mulsrc = o.mulsrc; a.ld_mul = o.ld_mul; a.mulmode = o.mulmode; a.Y = Y; a.ldy = ldy; a.accumulate = o.accumulate;
  a.post_scale = o.post_scale; a.drop_thresh = o.drop_thresh; a.drop_seed = o.drop_seed; a.drop_inv_keep = o.drop_inv_keep;
  a.drop_stride = o.drop_stride; a.ones_col = o.ones_col; a.poison = Y; a.bits_in = o.bits_in; a.bits_out = o.bits_out;
  return a;
}

void launch_rows_tc_raw(cudaStream_t st, const float* Bhi, const float* Blo, int NB, int M, int N, int nseg, const RowsSeg* sg,
                        float* Y, int ldy, const LinOpt& o) {
  if (M <= 0) return;
  const tc::RowsTcArgs a = make_rows_args(Bhi, Blo, M, N, nseg, sg, Y, ldy, o);
  const int ntiles = (M + kTM - 1) / kTM;
  const int grid = ntiles < num_sms() ? ntiles : num_sms();
  // 512 threads: with one CTA per SM (shared and tensor memory are full) more warps mean less serial work per warp
  // between the slab barriers (measured: 256 -> 512 threads = -15 % per launch, relation encoder and node layers alike)
  if (NB == 160) {
    auto kern = tc::k_rows_tc<160, 512>; set_smem(kern, tc::rows_tc_smem<160>(19));
    SPW_KLAUNCH(o.tag ? o.tag : "k_rows_tc<160>", kern, dim3(grid), dim3(512), tc::rows_tc_smem<160>(a.ks), st, a);
  } else {
    auto kern = tc::k_rows_tc<112, 512>; set_smem(kern, tc::rows_tc_smem<112>(25));
    SPW_KLAUNCH(o.tag ? o.tag : "k_rows_tc<112>", kern, dim3(grid), dim3(512), tc::rows_tc_smem<112>(a.ks), st, a);
  }
}

void launch_rows_tc(cudaStream_t st, float* ws, const Layout& L, int id, int M, int N, int nseg, const RowsSeg* sg, float* Y,
                    int ldy, const LinOpt& o) {
  launch_rows_tc_raw(st, ws + L.tcp[id], ws + L.tcp[id] + tc_floats(id), kTcShape[id].NB, M, N, nseg, sg, Y, ldy, o);
}
#endif

void run_linear(cudaStream_t st, float* ws, const Layout& L, LinId id, int M, int N, int nseg, const RowsSeg* sg, float* Y,
                int ldy, const LinOpt& o) {
#if SPW_USE_TC
  launch_rows_tc(st, ws, L, id.tc, M, N, nseg, sg, Y, ldy, o);
#else
  LinSeg s[2];
  for (int i = 0; i < nseg; ++i) s[i] = seg(sg[i].X, sg[i].ldx, sg[i].K, ws + L.pack[i == 0 ? id.pk0 : id.pk1]);
  launch_linear(st, M, N, N > 128, nseg, s, Y, ldy, o);
#endif
}

// dW[Kin][N] (+ bias row) = X^T dY over M rows, reduced in fixed order into the Keras-layout gradient
struct WgOut { float* dW; int dst_ld, dst_row0, dst_col0; float* db; int db_off; };

// While a list is installed here (backward_csl), launch_reduce only records its job; flush_reduces launches them all at once.
thread_local std::vector<RedArgs>* t_deferred_reduces = nullptr;

void launch_reduce(cudaStream_t st, const float* part, int nparts, int part_stride, int src_ld, int TA, int TB, int Kin,
                   int N, const WgOut& out) {
  RedArgs r;
  r.part = part; r.nparts = nparts; r.part_stride = part_stride; r.src_ld = src_ld; r.TA = TA; r.TB = TB; r.Kin = Kin; r.N = N;
  r.dW = out.dW; r.dst_ld = out.dst_ld; r.dst_row0 = out.dst_row0; r.dst_col0 = out.dst_col0;
  r.db = out.db; r.db_off = out.db_off;
  if (t_deferred_reduces) { t_deferred_reduces->push_back(r); return; }
  SPW_KLAUNCH_PDL("k_reduce_parts", k_reduce_parts, dim3(grid_for((int64_t)(Kin + 1) * N, 32)), dim3(256), 0, st, r);
}

#ifndef SPW_EMU
void flush_reduces(cudaStream_t st, const std::vector<RedArgs>& jobs) {
  for (size_t i0 = 0; i0 < jobs.size(); i0 += kMaxRedJobs) {
    RedJobs rj;
    memset(&rj, 0, sizeof(rj));
    const int nj = (int)(jobs.size() - i0 < (size_t)kMaxRedJobs ? jobs.size() - i0 : (size_t)kMaxRedJobs);
    int64_t most = 1;
    for (int i = 0; i < nj; ++i) {
      rj.j[i] = jobs[i0 + i];
      const int64_t t = (int64_t)(rj.j[i].Kin + 1) * rj.j[i].N;
      if (t > most) most = t;
    }
    SPW_KLAUNCH_PDL("k_reduce_parts", k_reduce_multi, dim3(grid_for(most, 32), nj), dim3(256), 0, st, rj);
  }
}
#endif

constexpr int kTW = 64;   // rows per tile of the node-level weight-gradient kernel

void launch_wgrad(cudaStream_t st, int M, const float* X, int ldx, int Kin, int xmod, const float* rowscale, int rsmod,
                  const float* dY, int ldy, int N, float* part, const WgOut& out) {
  WgArgs a;
  a.M = M; a.X = X; a.ldx = ldx; a.Kin = Kin; a.xmod = xmod; a.rowscale = rowscale; a.rsmod = rsmod; a.dY = dY; a.ldy = ldy; a.N = N;
  a.part = part;
#if SPW_USE_TC
  if (Kin >= 8 && N >= 8 && (ldx & 3) == 0 && (ldy & 3) == 0 && Kin <= 150 && N <= 160) {   // tensor cores
    tc::WgradRowsArgs t;
    t.M = M; t.X = X; t.ldx = ldx; t.Kx = Kin; t.xmod = xmod; t.rowscale = rowscale; t.rsmod = rsmod; t.dY = dY; t.ldy = ldy; t.Ny = N;
    t.NB = N <= 112 ? 112 : 160; t.part = part; t.poison = part;
    const int tt = (M + kTM - 1) / kTM;
    int tgrid = tt < num_sms() ? tt : num_sms();
    if (tgrid > kMaxCtas) tgrid = kMaxCtas;
    if (Kin + 1 <= 128 && t.NB == 112) {           // one M-tile and a narrow B operand: 64-row chunks fit
      auto kern = tc::k_wgrad_rows_tc<64>; set_smem(kern, tc::wgrad_rows_smem(64, 112));
      SPW_KLAUNCH("k_wgrad_rows_tc", kern, dim3(tgrid), dim3(tc::kWgThreads), tc::wgrad_rows_smem(64, 112), st, t);
    } else {
      auto kern = tc::k_wgrad_rows_tc<32>; set_smem(kern, tc::wgrad_rows_smem(32, 160));
      SPW_KLAUNCH("k_wgrad_rows_tc", kern, dim3(tgrid), dim3(tc::kWgThreads), tc::wgrad_rows_smem(32, t.NB), st, t);
    }
    launch_reduce(st, part, tgrid, (int)tc::kWgPartFloats, 0, -1, Kin + 1 > 128 ? Kin + 1 - 128 : 0, Kin, N, out);
    return;
  }
#endif
  const int ntiles = (M + kTW - 1) / kTW;
  const bool wa = Kin + 1 > 112, wb = N > 112;
  const int LX = wa ? 160 : 112, LY = wb ? 160 : 112;
  const int per_sm = (wa || wb) ? 1 : 2;
  int grid = ntiles < per_sm * num_sms() ? ntiles : per_sm * num_sms();
  if (grid < 1) grid = 1;
  if (grid > kMaxCtas * 2) grid = kMaxCtas * 2;
  const size_t smem = (size_t)kTW * (LX + LY) * sizeof(float);
  if (wa && wb) { auto k = k_wgrad<10, 10, kTW, 1>; set_smem(k, smem); SPW_KLAUNCH("k_wgrad", k, dim3(grid), dim3(kThreads), smem, st, a); }
  else if (wa) { auto k = k_wgrad<10, 7, kTW, 1>; set_smem(k, smem); SPW_KLAUNCH("k_wgrad", k, dim3(grid), dim3(kThreads), smem, st, a); }
  else if (wb) { auto k = k_wgrad<7, 10, kTW, 1>; set_smem(k, smem); SPW_KLAUNCH("k_wgrad", k, dim3(grid), dim3(kThreads), smem, st, a); }
  else { auto k = k_wgrad<7, 7, kTW, 2>; set_smem(k, smem); SPW_KLAUNCH("k_wgrad", k, dim3(grid), dim3(kThreads), smem, st, a); }
  launch_reduce(st, part, grid, LX * LY, 0, wa ? 10 : 7, wb ? 10 : 7, Kin, N, out);
}

void pack_weights(cudaStream_t st, const SpwParams* w, float* ws, const Layout& L, bool with_transposes) {
  PackArgs pa;
  memset(&pa, 0, sizeof(pa));
  int n = 0;
  auto add = [&](int id, const float* src, int src_ld, int row0, int col0, int K, int N, int transpose) {
    PackDesc& d = pa.d[n++];
    d.src = src; d.src_ld = src_ld; d.row0 = row0; d.col0 = col0; d.K = K; d.N = N; d.transpose = transpose;
    d.dst = ws + L.pack[id]; d.Kp = kPackShape[id].Kp; d.ldw = kPackShape[id].ldw;
  };
  add(P_RM1, w->rm_w[1], 150, 0, 0, 150, 150, 0);
  add(P_RM2, w->rm_w[2], 150, 0, 0, 150, 150, 0);
  add(P_RM3, w->rm_w[3], 150, 0, 0, 150, 150, 0);
  add(P_W1A, w->rmp_w[0], 150, 0, 0, 150, 150, 0);     // Networks.py:86 concat order: [rel_enc | sender | receiver]
  add(P_W1B, w->rmp_w[0], 150, 150, 0, 100, 150, 0);
  add(P_W1C, w->rmp_w[0], 150, 250, 0, 100, 150, 0);
  add(P_W2, w->rmp_w[1], 150, 0, 0, 150, 150, 0);
  add(P_W3, w->rmp_w[2], 100, 0, 0, 150, 100, 0);
  add(P_V1A, w->omp_w[0], 100, 0, 0, 100, 100, 0);     // Networks.py:89 concat order: [obj_enc | effect | prop]
  add(P_V1B, w->omp_w[0], 100, 100, 0, 100, 100, 0);
  add(P_V1C, w->omp_w[0], 100, 200, 0, 100, 100, 0);
  add(P_V2P, w->omp_w[1], 101, 0, 1, 100, 100, 0);     // channels 1..100 (Networks.py:80)
  add(P_OM1, w->om_w[1], 100, 0, 0, 100, 100, 0);
  if (with_transposes) {
    // transposed: dst[k][n] = src[row0 + n][col0 + k];  K = #cols of the source block, N = #rows
    add(P_RM1T, w->rm_w[1], 150, 0, 0, 150, 150, 1);
    add(P_RM2T, w->rm_w[2], 150, 0, 0, 150, 150, 1);
    add(P_RM3T, w->rm_w[3], 150, 0, 0, 150, 150, 1);
    add(P_W1AT, w->rmp_w[0], 150, 0, 0, 150, 150, 1);
    add(P_W1BT, w->rmp_w[0], 150, 150, 0, 150, 100, 1);
    add(P_W1CT, w->rmp_w[0], 150, 250, 0, 150, 100, 1);
    add(P_W2T, w->rmp_w[1], 150, 0, 0, 150, 150, 1);
    add(P_W3T, w->rmp_w[2], 100, 0, 0, 100, 150, 1);
    add(P_V1AT, w->omp_w[0], 100, 0, 0, 100, 100, 1);
    add(P_V1BT, w->omp_w[0], 100, 100, 0, 100, 100, 1);
    add(P_V1CT, w->omp_w[0], 100, 200, 0, 100, 100, 1);
    add(P_V2PT, w->omp_w[1], 101, 0, 1, 100, 100, 1);
    add(P_OM1T, w->om_w[1], 100, 0, 0, 100, 100, 1);
  }
  pa.n = n;
  SPW_KLAUNCH("k_pack_weights", k_pack_weights, dim3(24, n), dim3(256), 0, st, pa);
}

#if SPW_USE_TC
void pack_tc(cudaStream_t st, const SpwParams* w, float* ws, const Layout& L, bool with_transposes) {
  tc::PackTcArgs pa;
  memset(&pa, 0, sizeof(pa));
  int n = 0;
  auto add = [&](int id, const float* src, int ld, int row0, int col0, int K, int N, int transpose) {
    tc::PackTcDesc& d = pa.d[n++];
    d.src = src; d.ld = ld; d.row0 = row0; d.col0 = col0; d.K = K; d.N = N; d.transpose = transpose;
    d.hi = ws + L.tcp[id]; d.lo = d.hi + tc_floats(id); d.NB = kTcShape[id].NB; d.k_off = 0; d.k_lim = 8 * kTcShape[id].ks;
  };
  add(T_OM1, w->om_w[1], 100, 0, 0, 100, 100, 0);
  add(T_RM1, w->rm_w[1], 150, 0, 0, 150, 150, 0);
  add(T_RM2, w->rm_w[2], 150, 0, 0, 150, 150, 0);
  add(T_RM3, w->rm_w[3], 150, 0, 0, 150, 150, 0);
  add(T_W1A, w->rmp_w[0], 150, 0, 0, 150, 150, 0);      // Networks.py:86 concat order: [rel_enc | sender | receiver]
  add(T_W1B, w->rmp_w[0], 150, 150, 0, 100, 150, 0);
  add(T_W1C, w->rmp_w[0], 150, 250, 0, 100, 150, 0);
  add(T_W3, w->rmp_w[2], 100, 0, 0, 150, 100, 0);
  add(T_V1A, w->omp_w[0], 100, 0, 0, 100, 100, 0);      // Networks.py:89 concat order: [obj_enc | effect | prop]
  add(T_V1BC, w->omp_w[0], 100, 100, 0, 200, 100, 0);   // rows [V1b ; V1c] are consecutive: one K = 200 operand for [g | p]
  add(T_V2P, w->omp_w[1], 101, 0, 1, 100, 100, 0);      // channels 1..100 (Networks.py:80)
  if (with_transposes) {   // transposed: dst[k][n] = src[row0 + n][col0 + k];  K = #cols of the source block, N = #rows
    add(T_V2PT, w->omp_w[1], 101, 0, 1, 100, 100, 1);
    add(T_V1AT, w->omp_w[0], 100, 0, 0, 100, 100, 1);
    add(T_V1BT, w->omp_w[0], 100, 100, 0, 100, 100, 1);
    add(T_V1CT, w->omp_w[0], 100, 200, 0, 100, 100, 1);
    add(T_W3T, w->rmp_w[2], 100, 0, 0, 100, 150, 1);
    add(T_W1BT, w->rmp_w[0], 150, 150, 0, 150, 100, 1);
    add(T_W1CT, w->rmp_w[0], 150, 250, 0, 150, 100, 1);
    add(T_OM1T, w->om_w[1], 100, 0, 0, 100, 100, 1);
  }
  pa.n = n;
  SPW_KLAUNCH("k_pack_tc", tc::k_pack_tc, dim3(16, n), dim3(256), 0, st, pa);
}
#endif

#if SPW_USE_TC
constexpr size_t kPairFloats = (size_t)4 * 19 * 8 * 80;      // per matrix: hi half 0, hi half 1, lo half 0, lo half 1
// pair operand ids: 0..3 forward RM1, RM2, RM3, W1A;  4..7 transposed W1A, RM3, RM2, RM1 (the order the backward pass walks)
void pack_tc_pair(cudaStream_t st, const SpwParams* w, float* ws, const Layout& L, bool with_transposes) {
  tc::PackTcArgs pa;
  memset(&pa, 0, sizeof(pa));
  int n = 0;
  auto add = [&](int id, const float* src, int transpose) {
    for (int h = 0; h < 2; ++h) {
      tc::PackTcDesc& d = pa.d[n++];
      d.src = src; d.ld = 150; d.K = 150; d.N = h == 0 ? 80 : 70; d.transpose = transpose;
      d.row0 = transpose ? 80 * h : 0; d.col0 = transpose ? 0 : 80 * h;
      d.hi = ws + L.tcp2 + (size_t)id * kPairFloats + (size_t)h * tc::kB2Floats;
      d.lo = d.hi + 2 * tc::kB2Floats; d.NB = 80; d.k_off = 0; d.k_lim = 8 * tc::kKS;
    }
  };
  add(0, w->rm_w[1], 0); add(1, w->rm_w[2], 0); add(2, w->rm_w[3], 0); add(3, w->rmp_w[0], 0);
  if (with_transposes) { add(4, w->rmp_w[0], 1); add(5, w->rm_w[3], 1); add(6, w->rm_w[2], 1); add(7, w->rm_w[1], 1); }
  pa.n = n;
  SPW_KLAUNCH("k_pack_tc", tc::k_pack_tc, dim3(16, n), dim3(256), 0, st, pa);
}

// one 150 -> 150 layer on [E][152] rows with the CTA-pair kernel
void launch_rows_pair(cudaStream_t st, float* ws, const Layout& L, int pair_id, int M, const float* X, float* Y, const LinOpt& o) {
  if (M <= 0) return;
  RowsSeg sg = {X, kDEP, kDE};
  const float* base = ws + L.tcp2 + (size_t)pair_id * kPairFloats;
  tc::RowsTcArgs a = make_rows_args(base, base + 2 * tc::kB2Floats, M, kDE, 1, &sg, Y, kDEP, o);
  const int ntiles = (M + kTM - 1) / kTM, npairs = (ntiles + 1) / 2;
  const int nclusters = npairs < num_sms() / 2 ? npairs : num_sms() / 2;
  set_smem(tc::k_rows_pair, tc::kRowsPairSmem);
  SPW_KLAUNCH(o.tag ? o.tag : "k_rows_pair", tc::k_rows_pair, dim3(2 * nclusters), dim3(tc::kPairThreads), tc::kRowsPairSmem, st, a);
}
#endif


#if SPW_USE_TC
// ---- CSL data path (spw_csl.cuh) ------------------------------------------------------------------
// one pipelined linear layer: nks k-steps of the packed operand (Bhi, Blo), MMA N = NB, compile-time epilogue mask `epi`.
// Every (NB, k-steps per thread, epilogue) combination the network (and the unit tests) use is instantiated here; anything
// else is refused loudly.
#define SPW_LIN_TABLE(X)                                                                                                   \
  X(100, 100, 0u) X(100, 150, 0u) X(100, 200, 0u) X(150, 100, 0u) X(150, 150, 0u)                                         \
  X(100, 100, csl::EPI_BIAS | csl::EPI_RELU) X(100, 100, csl::EPI_BIAS | csl::EPI_RELU | csl::EPI_DROP) X(100, 100, csl::EPI_BIAS) \
  X(150, 150, csl::EPI_BIAS | csl::EPI_RELU | csl::EPI_ONES) X(150, 150, csl::EPI_BIAS | csl::EPI_RELU | csl::EPI_ONES | csl::EPI_BITS_OUT) \
  X(150, 150, csl::EPI_BIAS | csl::EPI_RELU | csl::EPI_ONES | csl::EPI_BITS_OUT | csl::EPI_DROP) X(150, 150, csl::EPI_BIAS) \
  X(100, 150, csl::EPI_BIAS | csl::EPI_ROWSCALE | csl::EPI_TANH) X(100, 200, csl::EPI_ADD | csl::EPI_RELU)                 \
  X(100, 100, csl::EPI_BIAS | csl::EPI_ADD | csl::EPI_TANH) X(100, 100, csl::EPI_MUL_POS)                                 \
  X(100, 100, csl::EPI_MUL_POS | csl::EPI_SCALE) X(100, 100, csl::EPI_MUL_POS | csl::EPI_SCALE | csl::EPI_ACC)            \
  X(100, 100, csl::EPI_MUL_TANH) X(100, 100, csl::EPI_ADD) X(100, 150, csl::EPI_ACC) X(100, 150, csl::EPI_ADD | csl::EPI_MUL_TANH) \
  X(150, 150, csl::EPI_MUL_BITS | csl::EPI_SCALE)

int launch_lin(cudaStream_t st, uint32_t epi, const csl::LinCArgs& a, const char* tag) {
  if (a.M <= 0) return SPW_OK;
  const int ntiles = (a.M + kTM - 1) / kTM;
  const int grid = ntiles < num_sms() ? ntiles : num_sms();
#define SPW_LIN_X(NV, KV, EPIV)                                                                                            \
  if (a.N == NV && a.K == KV && epi == (uint32_t)(EPIV)) {                                                                \
    auto kern = csl::k_lin<NV, KV, (uint32_t)(EPIV)>;                                                                     \
    const size_t sm = csl::lin_smem(NV <= 112 ? 112 : 160, (KV + 7) / 8); set_smem(kern, sm);                             \
    SPW_KLAUNCH_PDL(tag, kern, dim3(grid), dim3(csl::kThreadsC), sm, st, a);                                               \
    return SPW_OK;                                                                                                        \
  }
  SPW_LIN_TABLE(SPW_LIN_X)
#undef SPW_LIN_X
  return fail(SPW_ERR_UNSUPPORTED, "launch_lin(%s): no kernel instance for K = %d, N = %d, epilogue mask 0x%x", tag, a.K, a.N, epi);
}
#endif

size_t edge_fwd_smem() { return (size_t)(2 * (kTME * kDEP + 8) + 2 * kKT * kLdwE + 2 * kTME) * sizeof(float); }
size_t edge_bwd_smem() { return (size_t)(2 * (kTM * kDEP + 8) + 2 * kKT * kLdwE + kTM + 5 * kTM) * sizeof(float); }
size_t edge_encb_smem() { return (size_t)(5 * (kTMB * kDEP + 8) + 2 * kKT * kLdwE + 2 * kTMB) * sizeof(float); }

#if SPW_USE_TC
#include "spw_csl_path.inl"
#endif

}  // namespace

// =================================================================================================
extern "C" {

int spw_version(void) { return SPW_VERSION; }

long long spw_launch_count(void) { return prof::launches.load(); }

int spw_profile(int enable) {
  prof::enabled = enable != 0;
  return SPW_OK;
}

// "name launches total_ms\n" per kernel, after synchronising the recorded events; clears the log
int spw_profile_report(char* buf, size_t cap) {
  if (!buf || cap == 0) return fail(SPW_ERR_BAD_ARG, "spw_profile_report: null buffer");
  buf[0] = 0;
#ifndef SPW_EMU
  std::map<std::string, std::pair<long long, double>> acc;
  for (auto& r : prof::recs) {
    cudaEventSynchronize(r.b);
    float ms = 0.f;
    cudaEventElapsedTime(&ms, r.a, r.b);
    auto& e = acc[r.name];
    e.first += 1; e.second += ms;
    cudaEventDestroy(r.a); cudaEventDestroy(r.b);
  }
  prof::recs.clear();
  size_t off = 0;
  for (auto& kv : acc) {
    int w = snprintf(buf + off, cap - off, "%s %lld %.6f\n", kv.first.c_str(), kv.second.first, kv.second.second);
    if (w < 0 || (size_t)w >= cap - off) break;
    off += (size_t)w;
  }
#endif
  return SPW_OK;
}

// FP32 FFMA pipe peak: `iters` dependent-chain-free FMAs x 16 accumulators per thread; flops = 2*16*iters*threads
int spw_ffma_peak(float* out /*[grid*256]*/, int grid, int iters, void* stream) {
  if (!out || grid <= 0 || iters <= 0) return fail(SPW_ERR_BAD_ARG, "spw_ffma_peak: bad argument");
  SPW_KLAUNCH("k_ffma_peak", k_ffma_peak, dim3(grid), dim3(256), 0, (cudaStream_t)stream, out, iters);
  return check_launch("spw_ffma_peak");
}
const char* spw_last_error(void) { return g_err; }

// tcgen05 self test: D[128][160] = A[128][152] . W, W given as a Keras [K][N] matrix (ld = N); scratch holds the
// packed hi/lo B operands (2 * 24320 floats); status: 1 ok, -1 the MMA never signalled its mbarrier
int spw_tc_selftest(const float* A, const float* W, int K, int N, float* D, float* scratch, int* status, void* stream) {
#ifdef SPW_EMU
  (void)A; (void)W; (void)K; (void)N; (void)D; (void)scratch; (void)status; (void)stream;
  return fail(SPW_ERR_UNSUPPORTED, "spw_tc_selftest: tensor-core path is not emulated");
#else
  if (!A || !W || !D || !scratch || !status || K > 152 || N > 160) return fail(SPW_ERR_BAD_ARG, "spw_tc_selftest: bad argument");
  cudaStream_t st = (cudaStream_t)stream;
  SPW_KLAUNCH("k_pack_umma", tc::k_pack_umma, dim3(48), dim3(256), 0, st, W, N, 0, 0, K, N, 0, (const float*)nullptr, scratch, scratch + tc::kBFloats);
  const size_t smem = (size_t)2 * tc::kBFloats * sizeof(float) + 64;
  set_smem(tc::k_tc_selftest, smem);
  SPW_KLAUNCH("k_tc_selftest", tc::k_tc_selftest, dim3(1), dim3(128), smem, st, A, scratch, scratch + tc::kBFloats, D, status);
  return check_launch("spw_tc_selftest");
#endif
}

// CTA-pair self test (tcgen05 cta_group::2): D[256][160] = A[256][152] . W, W a Keras [K][N] matrix (ld = N);
// scratch: 4 * 19 * 8 * 80 floats; status[2] (device ints, one per CTA): 1 ok, -1 the completion barrier timed out
int spw_tc2_selftest(const float* A, const float* W, int K, int N, float* D, float* scratch, int* status, void* stream) {
#if !SPW_USE_TC
  (void)A; (void)W; (void)K; (void)N; (void)D; (void)scratch; (void)status; (void)stream;
  return fail(SPW_ERR_UNSUPPORTED, "spw_tc2_selftest: tensor-core path is not emulated");
#else
  if (!A || !W || !D || !scratch || !status || K > 152 || N > 160 || K <= 0 || N <= 0) return fail(SPW_ERR_BAD_ARG, "spw_tc2_selftest: bad argument");
  cudaStream_t st = (cudaStream_t)stream;
  tc::PackTcArgs pa;
  memset(&pa, 0, sizeof(pa));
  float* hi = scratch; float* lo = scratch + 2 * tc::kB2Floats;
  for (int h = 0; h < 2; ++h) {
    tc::PackTcDesc& d = pa.d[h];
    d.src = W; d.ld = N; d.row0 = 0; d.col0 = 80 * h; d.K = K; d.N = N - 80 * h < 0 ? 0 : (N - 80 * h > 80 ? 80 : N - 80 * h);
    d.hi = hi + (size_t)h * tc::kB2Floats; d.lo = lo + (size_t)h * tc::kB2Floats; d.NB = 80; d.k_off = 0; d.k_lim = 8 * tc::kKS;
  }
  pa.n = 2;
  SPW_KLAUNCH("k_pack_tc", tc::k_pack_tc, dim3(16, 2), dim3(256), 0, st, pa);
  const size_t smem = (size_t)2 * tc::kB2Floats * sizeof(float) + 64;
  set_smem(tc::k_tc2_selftest, smem);
  SPW_KLAUNCH("k_tc2_selftest", tc::k_tc2_selftest, dim3(2), dim3(128), smem, st, A, (const float*)hi, (const float*)lo, D, status);
  return check_launch("spw_tc2_selftest");
#endif
}

// generic tensor-core linear layer (tc::k_rows_tc), exposed for unit tests:
//   Y[M][ldy] = post(act([X0 | X1].W + rowscale*bias + addend)), W Keras layout [K0 + K1][N] (ld = N); NB = 112 or 160;
//   scratch: 2 * ceil((K0 + K1) / 8) * 8 * NB floats
int spw_tc_linear(int M, const float* X0, int ldx0, int K0, const float* X1, int ldx1, int K1, const float* W, int N, int NB,
                  const float* bias, const float* rowscale, const float* addend, int ld_add, int act, const float* mulsrc,
                  int ld_mul, int mulmode, float* Y, int ldy, int accumulate, float post_scale, int ones_col, float* scratch,
                  void* stream) {
#if !SPW_USE_TC
  (void)M; (void)X0; (void)ldx0; (void)K0; (void)X1; (void)ldx1; (void)K1; (void)W; (void)N; (void)NB; (void)bias; (void)rowscale;
  (void)addend; (void)ld_add; (void)act; (void)mulsrc; (void)ld_mul; (void)mulmode; (void)Y; (void)ldy; (void)accumulate;
  (void)post_scale; (void)ones_col; (void)scratch; (void)stream;
  return fail(SPW_ERR_UNSUPPORTED, "spw_tc_linear: tensor-core path is not emulated");
#else
  if (M < 0 || !X0 || !W || !Y || !scratch || K0 <= 0 || K1 < 0 || N <= 0) return fail(SPW_ERR_BAD_ARG, "spw_tc_linear: bad argument");
  if (NB != 112 && NB != 160) return fail(SPW_ERR_UNSUPPORTED, "spw_tc_linear: NB must be 112 or 160");
  const int ks = (K0 + K1 + 7) / 8;
  if (N > NB || 16 * ks + NB > 512) return fail(SPW_ERR_UNSUPPORTED, "spw_tc_linear: K = %d, N = %d do not fit tensor memory", K0 + K1, N);
  if ((ldx0 & 3) || (K1 && ((ldx1 & 3) || (K0 & 3))) || (ldy & 3) || (addend && (ld_add & 3)) || (mulmode && (ld_mul & 3)))
    return fail(SPW_ERR_BAD_ARG, "spw_tc_linear: leading dimensions must be multiples of 4");
  cudaStream_t st = (cudaStream_t)stream;
  tc::PackTcArgs pa;
  memset(&pa, 0, sizeof(pa));
  tc::PackTcDesc& d = pa.d[0];
  d.src = W; d.ld = N; d.K = K0 + K1; d.N = N; d.hi = scratch; d.lo = scratch + (size_t)ks * 8 * NB; d.NB = NB; d.k_lim = 8 * ks;
  pa.n = 1;
  SPW_KLAUNCH("k_pack_tc", tc::k_pack_tc, dim3(16, 1), dim3(256), 0, st, pa);
  RowsSeg sg[2] = {{X0, ldx0, K0}, {X1, ldx1, K1}};
  LinOpt o;
  o.bias = bias; o.rowscale = rowscale; o.addend = addend; o.ld_add = ld_add; o.act = act; o.mulsrc = mulsrc; o.ld_mul = ld_mul;
  o.mulmode = mulmode; o.accumulate = accumulate; o.post_scale = post_scale; o.ones_col = ones_col;
  launch_rows_tc_raw(st, d.hi, d.lo, NB, M, N, K1 > 0 ? 2 : 1, sg, Y, ldy, o);
  return check_launch("spw_tc_linear");
#endif
}


// pipelined CSL linear layer (csl::k_lin), exposed for unit tests.  Arrays are column-slab major: element (row, c) of a view
// at p + ((col0 + c) >> 3) * slab + row * 8 + ((col0 + c) & 7).  W: Keras [K][N] (ld = N).  bits_in / bits_out: word-major sign
// bits [8][M][4 bytes].  scratch: 2 * ceil(K / 8) * 8 * NB floats.
int spw_csl_linear(int M, const float* X, long long x_slab, int x_col0, int K, const float* W, int N, int NB, const float* bias,
                   const float* rowscale, const float* addend, long long add_slab, int add_col0, int act, const float* mulsrc,
                   long long mul_slab, int mul_col0, int mulmode, const uint8_t* bits_in, uint8_t* bits_out, float* Y,
                   long long y_slab, int y_col0, int accumulate, float post_scale, int ones_col, int write_pad, float* scratch,
                   void* stream) {
#if !SPW_USE_TC
  (void)M; (void)X; (void)x_slab; (void)x_col0; (void)K; (void)W; (void)N; (void)NB; (void)bias; (void)rowscale; (void)addend;
  (void)add_slab; (void)add_col0; (void)act; (void)mulsrc; (void)mul_slab; (void)mul_col0; (void)mulmode; (void)bits_in;
  (void)bits_out; (void)Y; (void)y_slab; (void)y_col0; (void)accumulate; (void)post_scale; (void)ones_col; (void)write_pad;
  (void)scratch; (void)stream;
  return fail(SPW_ERR_UNSUPPORTED, "spw_csl_linear: tensor-core path is not emulated");
#else
  if (M < 0 || !X || !W || !Y || !scratch || K <= 0 || N <= 0) return fail(SPW_ERR_BAD_ARG, "spw_csl_linear: bad argument");
  if (NB != 112 && NB != 160) return fail(SPW_ERR_UNSUPPORTED, "spw_csl_linear: NB must be 112 or 160");
  const int nks = (K + 7) / 8;
  if (N > NB || 16 * nks + NB > 512) return fail(SPW_ERR_UNSUPPORTED, "spw_csl_linear: K = %d, N = %d do not fit tensor memory", K, N);
  if ((x_col0 & 3) || (y_col0 & 3) || (add_col0 & 3) || (mul_col0 & 3)) return fail(SPW_ERR_BAD_ARG, "spw_csl_linear: column offsets must be multiples of 4");
  cudaStream_t st = (cudaStream_t)stream;
  tc::PackTcArgs pa;
  memset(&pa, 0, sizeof(pa));
  tc::PackTcDesc& d = pa.d[0];
  d.src = W; d.ld = N; d.K = K; d.N = N; d.hi = scratch; d.lo = scratch + (size_t)nks * 8 * NB; d.NB = NB; d.k_lim = 8 * nks;
  pa.n = 1;
  SPW_KLAUNCH("k_pack_tc", tc::k_pack_tc, dim3(16, 1), dim3(256), 0, st, pa);
  csl::LinCArgs a;
  memset(&a, 0, sizeof(a));
  a.M = M; a.K = K; a.nks = nks; a.N = N;
  a.X = {const_cast<float*>(X), x_slab, x_col0};
  a.Bhi = d.hi; a.Blo = d.lo; a.bias = bias; a.rowscale = rowscale;
  a.addend = {const_cast<float*>(addend), add_slab, add_col0};
  a.mulsrc = {const_cast<float*>(mulsrc), mul_slab, mul_col0};
  a.bits_in = bits_in; a.bits_in_rows = M; a.bits_out = bits_out; a.bits_out_rows = M;
  a.Y = {Y, y_slab, y_col0}; a.post_scale = post_scale; a.ones_col = ones_col; a.write_pad = write_pad;
  a.drop_stride = 128; a.poison = Y;
  uint32_t epi = 0;
  if (bias) epi |= csl::EPI_BIAS;
  if (rowscale) epi |= csl::EPI_ROWSCALE;
  if (addend) epi |= csl::EPI_ADD;
  if (act == 1) epi |= csl::EPI_RELU;
  if (act == 2) epi |= csl::EPI_TANH;
  if (mulmode == 1) epi |= csl::EPI_MUL_POS;
  if (mulmode == 2) epi |= csl::EPI_MUL_TANH;
  if (mulmode == 3) epi |= csl::EPI_MUL_BITS;
  if (post_scale != 1.f) epi |= csl::EPI_SCALE;
  if (accumulate) epi |= csl::EPI_ACC;
  if (bits_out) epi |= csl::EPI_BITS_OUT;
  if (ones_col >= 0) epi |= csl::EPI_ONES;
  if (NB != (N <= 112 ? 112 : 160)) return fail(SPW_ERR_UNSUPPORTED, "spw_csl_linear: NB must be 112 for N <= 112, else 160");
  int rc = launch_lin(st, epi, a, "k_lin");
  if (rc != SPW_OK) return rc;
  return check_launch("spw_csl_linear");
#endif
}

int spw_edges_count(const double* pos_xy, const int32_t* node_off, int32_t n_towers, int32_t n_nodes,
                    int32_t max_nodes_per_tower, double thr, int fully_connected, int32_t* deg_out, int32_t* deg_in,
                    int32_t* edge_off, void* stream) {
  if (n_towers < 0 || n_nodes < 0) return fail(SPW_ERR_BAD_ARG, "spw_edges_count: negative size");
  if (max_nodes_per_tower > SPW_MAX_NODES)
    return fail(SPW_ERR_UNSUPPORTED, "spw_edges_count: %d blocks in a tower, limit is %d", max_nodes_per_tower, SPW_MAX_NODES);
  if (!edge_off || (n_towers > 0 && !node_off) || (n_nodes > 0 && (!pos_xy || !deg_out || !deg_in)))
    return fail(SPW_ERR_BAD_ARG, "spw_edges_count: null pointer");
  cudaStream_t st = (cudaStream_t)stream;
  if (n_towers == 0) { cudaMemsetAsync(edge_off, 0, sizeof(int32_t), st); return check_launch("spw_edges_count"); }
  SPW_KLAUNCH("k_edges_count", k_edges_count, dim3(n_towers), dim3(kMaxNodes), 0, st, pos_xy, node_off, thr, fully_connected, deg_out,
             deg_in, edge_off);
  SPW_KLAUNCH("k_scan_inplace", k_scan_inplace, dim3(1), dim3(1024), 0, st, edge_off, (int)n_towers);
  return check_launch("spw_edges_count");
}

int spw_edges_fill(const double* pos_xy, const int32_t* node_off, int32_t n_towers, int32_t n_nodes,
                   int32_t max_nodes_per_tower, double thr, int fully_connected, const int32_t* edge_off, int32_t* snd,
                   int32_t* rcv, int32_t* slot, int32_t* in_off, int32_t* in_snd, int32_t* in_rcv, int32_t* out_off,
                   int32_t* out_pos, void* stream) {
  if (n_towers < 0 || n_nodes < 0) return fail(SPW_ERR_BAD_ARG, "spw_edges_fill: negative size");
  if (max_nodes_per_tower > SPW_MAX_NODES)
    return fail(SPW_ERR_UNSUPPORTED, "spw_edges_fill: %d blocks in a tower, limit is %d", max_nodes_per_tower, SPW_MAX_NODES);
  if (!edge_off || !in_off || !out_off) return fail(SPW_ERR_BAD_ARG, "spw_edges_fill: null offsets");
  cudaStream_t st = (cudaStream_t)stream;
  if (n_towers == 0) {
    cudaMemsetAsync(in_off, 0, sizeof(int32_t), st);
    cudaMemsetAsync(out_off, 0, sizeof(int32_t), st);
    return check_launch("spw_edges_fill");
  }
  if (!pos_xy || !node_off || !in_snd || !in_rcv || !out_pos) return fail(SPW_ERR_BAD_ARG, "spw_edges_fill: null pointer");
  SPW_KLAUNCH("k_edges_fill", k_edges_fill, dim3(n_towers), dim3(kMaxNodes), 0, st, pos_xy, node_off, (int)n_towers, (int)n_nodes, thr,
             fully_connected, edge_off, snd, rcv, slot, in_off, in_snd, in_rcv, out_off, out_pos);
  return check_launch("spw_edges_fill");
}

int spw_sample_sizes(uint64_t seed, int32_t n_towers, int32_t n_lo, int32_t n_hi, int32_t* node_off, void* stream) {
  if (n_towers < 0 || n_lo < 1 || n_hi < n_lo) return fail(SPW_ERR_BAD_ARG, "spw_sample_sizes: bad size range");
  if (n_hi > SPW_MAX_NODES) return fail(SPW_ERR_UNSUPPORTED, "spw_sample_sizes: %d blocks in a tower, limit is %d", n_hi, SPW_MAX_NODES);
  if (!node_off) return fail(SPW_ERR_BAD_ARG, "spw_sample_sizes: null pointer");
  cudaStream_t st = (cudaStream_t)stream;
  SPW_KLAUNCH("k_sample_sizes", k_sample_sizes, dim3(grid_for(n_towers + 1, 256)), dim3(256), 0, st, seed, (int)n_towers, (int)n_lo, (int)n_hi, node_off);
  if (n_towers > 0) SPW_KLAUNCH("k_scan_inplace", k_scan_inplace, dim3(1), dim3(1024), 0, st, node_off, (int)n_towers);
  return check_launch("spw_sample_sizes");
}

int spw_sample_jenga(uint64_t seed, int32_t n_towers, const int32_t* node_off, double* raw, float* obj, double* pos,
                     int inference_glue, void* stream) {
  if (n_towers < 0) return fail(SPW_ERR_BAD_ARG, "spw_sample_jenga: negative size");
  if (n_towers == 0) return SPW_OK;
  if (!node_off || (!raw && !obj && !pos)) return fail(SPW_ERR_BAD_ARG, "spw_sample_jenga: null pointer");
  SPW_KLAUNCH("k_sample_jenga", k_sample_jenga, dim3((n_towers + 127) / 128), dim3(128), 0, (cudaStream_t)stream, seed, (int)n_towers, node_off, raw,
              obj, pos, inference_glue);
  return check_launch("spw_sample_jenga");
}

int spw_sample_tower(uint64_t seed, int32_t n_towers, const int32_t* node_off, double* raw, float* obj, double* pos,
                     int inference_glue, void* stream) {
  if (n_towers < 0) return fail(SPW_ERR_BAD_ARG, "spw_sample_tower: negative size");
  if (n_towers == 0) return SPW_OK;
  if (!node_off || (!raw && !obj && !pos)) return fail(SPW_ERR_BAD_ARG, "spw_sample_tower: null pointer");
  SPW_KLAUNCH("k_sample_tower", k_sample_tower, dim3((n_towers + 127) / 128), dim3(128), 0, (cudaStream_t)stream, seed, (int)n_towers, node_off, raw,
              obj, pos, inference_glue);
  return check_launch("spw_sample_tower");
}

int spw_candidates_remove(const double* raw, int32_t n_blocks, float* obj, double* pos, int inference_glue, void* stream) {
  if (n_blocks < 2 || n_blocks > SPW_MAX_NODES + 1) return fail(SPW_ERR_BAD_ARG, "spw_candidates_remove: %d blocks (need 2..%d)", n_blocks, SPW_MAX_NODES + 1);
  if (!raw || !obj || !pos) return fail(SPW_ERR_BAD_ARG, "spw_candidates_remove: null pointer");
  SPW_KLAUNCH("k_candidates_remove", k_candidates_remove, dim3(grid_for((int64_t)n_blocks * (n_blocks - 1), 256)), dim3(256), 0, (cudaStream_t)stream, raw,
              (int)n_blocks, obj, pos, inference_glue);
  return check_launch("spw_candidates_remove");
}

int spw_candidates_drop(const double* raw, int32_t n_blocks, const double* poses, int32_t n_poses, double width, float* obj, double* pos,
                        int inference_glue, void* stream) {
  if (n_blocks < 1 || n_blocks + 1 > SPW_MAX_NODES || n_poses < 0) return fail(SPW_ERR_BAD_ARG, "spw_candidates_drop: bad size");
  if (n_poses == 0) return SPW_OK;
  if (!raw || !poses || !obj || !pos) return fail(SPW_ERR_BAD_ARG, "spw_candidates_drop: null pointer");
  SPW_KLAUNCH("k_candidates_drop", k_candidates_drop, dim3(grid_for((int64_t)n_poses * (n_blocks + 1), 256)), dim3(256), 0, (cudaStream_t)stream, raw,
              (int)n_blocks, poses, (int)n_poses, width, obj, pos, inference_glue);
  return check_launch("spw_candidates_drop");
}

int spw_tower_sums(const float* probs, const int32_t* node_off, int32_t n_towers, double* sums, int32_t* argmin, void* stream) {
  if (n_towers < 0) return fail(SPW_ERR_BAD_ARG, "spw_tower_sums: negative size");
  if (n_towers == 0) return SPW_OK;
  if (!probs || !node_off || !sums) return fail(SPW_ERR_BAD_ARG, "spw_tower_sums: null pointer");
  cudaStream_t st = (cudaStream_t)stream;
  SPW_KLAUNCH("k_tower_sums", k_tower_sums, dim3(grid_for(n_towers, 256)), dim3(256), 0, st, probs, node_off, (int)n_towers, sums);
  if (argmin) SPW_KLAUNCH("k_argmin", k_argmin, dim3(1), dim3(256), 0, st, (const double*)sums, (int)n_towers, argmin);
  return check_launch("spw_tower_sums");
}

size_t spw_workspace_bytes(int32_t n_nodes, int32_t n_edges, int training) {
  if (n_nodes < 0 || n_edges < 0) return 0;
#if SPW_USE_TC
  if (use_csl()) return make_layout_c(n_nodes, n_edges, training).total * sizeof(float);
#endif
  return make_layout(n_nodes, n_edges, training).total * sizeof(float);
}

int spw_saved_state_layout(int32_t n_nodes, int32_t n_edges, int64_t* out) {
  if (n_nodes < 0 || n_edges < 0 || !out) return fail(SPW_ERR_BAD_ARG, "spw_saved_state_layout: bad argument");
#if SPW_USE_TC
  if (use_csl()) {
    const LayoutC L = make_layout_c(n_nodes, n_edges, 1);
    out[0] = L.bits_rows; out[1] = (int64_t)L.bits_floats * 4;
    out[2] = (int64_t)L.EB * 4; out[3] = (int64_t)L.M1 * 4; out[4] = (int64_t)L.M2 * 4;
    out[5] = (int64_t)L.U * 4; out[6] = (int64_t)L.Q * 4; out[7] = (int64_t)L.Q1 * 4;
    return SPW_OK;
  }
#endif
  return fail(SPW_ERR_UNSUPPORTED, "spw_saved_state_layout: column-slab path only");
}

// Every named array of the column-slab workspace (byte offsets), then the sizes a reader needs to index them; the order is
// the one of spw_workspace_layout_names.  Arrays a mode does not use (inference: the backward state) are 0.
static const char kWorkspaceLayoutNames[] =
    "W2hi,W2lo,W2Thi,W2Tlo,ENCT,degf,Q1,Q,QV,GP,U,S,R,H2S,PF,PL,X0,X1,X2,C,A,H1,EB,M1,M2,"
    "dU,dG,T,dS,dR,dH2S,DP,dQ,dQ1,dA,DH1,GB,partE,part0,partN,"
    "slots,slotsGP,bits_rows,bits_floats,edge_stride_floats,part_stride_floats,part0_stride_floats,total_bytes";

const char* spw_workspace_layout_names(void) { return kWorkspaceLayoutNames; }

int spw_workspace_layout(int32_t n_nodes, int32_t n_edges, int training, int64_t* out, int cap) {
  if (n_nodes < 0 || n_edges < 0 || !out) return fail(SPW_ERR_BAD_ARG, "spw_workspace_layout: bad argument");
#if SPW_USE_TC
  if (use_csl()) {
    const LayoutC L = make_layout_c(n_nodes, n_edges, training);
    const size_t offs[] = {L.W2hi, L.W2lo, L.W2Thi, L.W2Tlo, L.ENCT, L.degf, L.Q1, L.Q, L.QV, L.GP, L.U, L.S, L.R, L.H2S, L.PF, L.PL,
                           L.X0, L.X1, L.X2, L.C, L.A, L.H1, L.EB, L.M1, L.M2, L.dU, L.dG, L.T, L.dS, L.dR, L.dH2S, L.DP, L.dQ, L.dQ1,
                           L.dA, L.DH1, L.GB, L.partE, L.part0, L.partN};
    const int64_t sizes[] = {L.slots, L.slotsGP, L.bits_rows, L.bits_floats, (int64_t)kQ150 * n_edges * 4 + 64, (int64_t)L.part_stride,
                             (int64_t)L.part0_stride, (int64_t)L.total * 4};
    const int no = (int)(sizeof(offs) / sizeof(offs[0])), ns = (int)(sizeof(sizes) / sizeof(sizes[0]));
    if (cap < no + ns) return fail(SPW_ERR_BAD_ARG, "spw_workspace_layout: %d entries do not fit in %d", no + ns, cap);
    for (int i = 0; i < no; ++i) out[i] = (int64_t)offs[i] * 4;
    for (int i = 0; i < ns; ++i) out[no + i] = sizes[i];
    return no + ns;
  }
#endif
  (void)training; (void)cap;
  return fail(SPW_ERR_UNSUPPORTED, "spw_workspace_layout: column-slab path only");
}

int spw_forward(const SpwParams* w, const SpwGraph* g, const float* obj, float* logits, float* probs, void* workspace,
                size_t workspace_bytes, int training, float dropout_rate, uint64_t dropout_seed, void* stream) {
  int rc;
  if ((rc = check_params(w, "spw_forward")) != SPW_OK) return rc;
  if ((rc = check_graph(g)) != SPW_OK) return rc;
  const int n = g->n_nodes, E = g->n_edges;
  if (n == 0) return SPW_OK;
  if (!obj || !logits || !workspace) return fail(SPW_ERR_BAD_ARG, "spw_forward: null pointer");
  if (!aligned16(workspace)) return fail(SPW_ERR_BAD_ARG, "spw_forward: workspace not 16-byte aligned");
  if (dropout_rate < 0.f || dropout_rate >= 1.f) return fail(SPW_ERR_BAD_ARG, "spw_forward: dropout rate %g outside [0,1)", dropout_rate);
#if SPW_USE_TC
  if (use_csl())
    return forward_csl(w, g, obj, logits, probs, reinterpret_cast<float*>(workspace), workspace_bytes, training, dropout_rate, dropout_seed,
                       (cudaStream_t)stream);
#endif
  const bool drop = training && dropout_rate > 0.f;
  const uint32_t drop_thresh = drop ? (uint32_t)(dropout_rate * 16777216.0f) : 0u;
  const float inv_keep = drop ? 1.f / (1.f - dropout_rate) : 1.f;
  const uint32_t seed_c = (uint32_t)dropout_seed, seed_q = (uint32_t)(dropout_seed >> 32) ^ 0x5bd1e995u ^ (uint32_t)dropout_seed * 3u;
  const Layout L = make_layout(n, E, training);
  if (workspace_bytes < L.total * sizeof(float))
    return fail(SPW_ERR_WORKSPACE, "spw_forward: workspace %zu < %zu bytes", workspace_bytes, L.total * sizeof(float));
  cudaStream_t st = (cudaStream_t)stream;
  float* ws = reinterpret_cast<float*>(workspace);
  auto PK = [&](int id) { return ws + L.pack[id]; };
  const size_t nP = (size_t)n * kDP, nE = (size_t)n * kDEP;

#if SPW_USE_TC
  pack_tc(st, w, ws, L, training != 0);
  const bool use_pair = E >= 64 * kTM * 2;       // CTA-pair relation-encoder layers: worth it from a few tile pairs per cluster on
  if (use_pair) pack_tc_pair(st, w, ws, L, training != 0);
#else
  pack_weights(st, w, ws, L, training != 0);
#endif
#if SPW_USE_TC
  SPW_KLAUNCH("k_pack_umma", tc::k_pack_umma, dim3(48), dim3(256), 0, st, (const float*)w->rmp_w[1], 150, 0, 0, 150, 150, 0, (const float*)w->rmp_b[1], ws + L.W2hi, ws + L.W2lo);
  if (training) {   // B operands of the data gradients: [N = k_in][K = n_out] = W[k_in][n_out]
    SPW_KLAUNCH("k_pack_umma", tc::k_pack_umma, dim3(48), dim3(256), 0, st, (const float*)w->rmp_w[1], 150, 0, 0, 150, 150, 1, (const float*)nullptr, ws + L.W2Thi, ws + L.W2Tlo);
    const float* encw[4] = {w->rmp_w[0], w->rm_w[3], w->rm_w[2], w->rm_w[1]};       // W1a, RM3, RM2, RM1
    for (int i = 0; i < 4; ++i)
      SPW_KLAUNCH("k_pack_umma", tc::k_pack_umma, dim3(48), dim3(256), 0, st, encw[i], 150, 0, 0, 150, 150, 1, (const float*)nullptr,
                  ws + L.ENCT + (size_t)(2 * i) * 24320, ws + L.ENCT + (size_t)(2 * i + 1) * 24320);
  }
#endif
  SPW_KLAUNCH("k_deg_to_float", k_deg_to_float, dim3(grid_for(n, 256)), dim3(256), 0, st, g->in_off, n, ws + L.degf);

  // object encoder (Networks.py:47,76): q1 = relu(om0([y,w])), q = relu(om1(q1))
  SPW_KLAUNCH("k_obj_enc0", k_obj_enc0, dim3(grid_for((int64_t)n * kDP, 256)), dim3(256), 0, st, obj, n, w->om_w[0], w->om_b[0], ws + L.Q1);
  {
    RowsSeg s = {ws + L.Q1, kDP, kDP};
    LinOpt o; o.bias = w->om_b[1]; o.act = 1;
    o.drop_thresh = drop_thresh; o.drop_seed = seed_q; o.drop_inv_keep = inv_keep;      // Networks.py:78
    run_linear(st, ws, L, {T_OM1, P_OM1, 0}, n, kDP, 1, &s, ws + L.Q, kDP, o);
  }
  {   // the object-encoding part of omp layer 0 is the same in all five steps: qv = q.V1a + c1   (Networks.py:89)
    RowsSeg s = {ws + L.Q, kDP, kDP};
    LinOpt o; o.bias = w->omp_b[0];
    run_linear(st, ws, L, {T_V1A, P_V1A, 0}, n, kDP, 1, &s, ws + L.QV, kDP, o);
  }
  // relation encoder + A_e (Networks.py:46,75 and the c_e part of :86-87)
  const int etiles = (E + kTME - 1) / kTME;
  const int egrid = etiles < 2 * num_sms() ? etiles : 2 * num_sms();
#if SPW_USE_TC
  if (E > 0) {   // layer by layer on the tensor cores; training keeps X0, X1, X2, C for the backward pass, inference runs in place
    float* X0 = training ? ws + L.EX0 : ws + L.A;
    float* X1 = training ? ws + L.EX1 : ws + L.A;
    float* X2 = training ? ws + L.EX2 : ws + L.A;
    float* C = training ? ws + L.EC : ws + L.A;
    uint32_t* EB = training ? reinterpret_cast<uint32_t*>(ws + L.EB) : nullptr;     // sign bits of X0, X1, X2, C
    const size_t nb = (size_t)E * 8;
    SPW_KLAUNCH("k_edge_enc0", tc::k_edge_enc0, dim3(grid_for((int64_t)E * 40, 256)), dim3(256), 0, st, E, g->in_snd, g->in_rcv,
                obj, (const float*)w->rm_w[0], (const float*)w->rm_b[0], X0, EB);
    LinOpt o; o.act = 1; o.ones_col = kDE; o.tag = "k_rows_tc<160>:enc_fwd";
    RowsSeg s0 = {X0, kDEP, kDE}, s1 = {X1, kDEP, kDE}, s2 = {X2, kDEP, kDE}, s3 = {C, kDEP, kDE};
    o.bias = w->rm_b[1]; o.bits_out = EB ? EB + nb : nullptr;
    if (use_pair) launch_rows_pair(st, ws, L, 0, E, X0, X1, o); else
    launch_rows_tc(st, ws, L, T_RM1, E, kDE, 1, &s0, X1, kDEP, o);
    o.bias = w->rm_b[2]; o.bits_out = EB ? EB + 2 * nb : nullptr;
    if (use_pair) launch_rows_pair(st, ws, L, 1, E, X1, X2, o); else
    launch_rows_tc(st, ws, L, T_RM2, E, kDE, 1, &s1, X2, kDEP, o);
    o.bias = w->rm_b[3]; o.bits_out = EB ? EB + 3 * nb : nullptr;
    o.drop_thresh = drop_thresh; o.drop_seed = seed_c; o.drop_inv_keep = inv_keep; o.drop_stride = 160;   // Networks.py:77
    if (use_pair) launch_rows_pair(st, ws, L, 2, E, X2, C, o); else
    launch_rows_tc(st, ws, L, T_RM3, E, kDE, 1, &s2, C, kDEP, o);
    LinOpt oa; oa.bias = w->rmp_b[0]; oa.tag = "k_rows_tc<160>:enc_fwd";
    if (use_pair) launch_rows_pair(st, ws, L, 3, E, C, ws + L.A, oa); else
    launch_rows_tc(st, ws, L, T_W1A, E, kDE, 1, &s3, ws + L.A, kDEP, oa);
  }
#else
  if (E > 0) {
    EdgeEncArgs a;
    a.E = E; a.in_snd = g->in_snd; a.in_rcv = g->in_rcv; a.obj = obj; a.W0 = w->rm_w[0]; a.b0 = w->rm_b[0];
    a.RM1 = PK(P_RM1); a.RM2 = PK(P_RM2); a.RM3 = PK(P_RM3); a.b1 = w->rm_b[1]; a.b2 = w->rm_b[2]; a.b3 = w->rm_b[3];
    a.W1A = PK(P_W1A); a.bA = w->rmp_b[0]; a.A = ws + L.A;
    a.X1 = training ? ws + L.EX1 : nullptr; a.X2 = training ? ws + L.EX2 : nullptr; a.C = training ? ws + L.EC : nullptr;
    a.X0 = (training && SPW_USE_TC) ? ws + L.EX0 : nullptr;
    a.drop_thresh = drop_thresh; a.drop_seed = seed_c; a.drop_inv_keep = inv_keep;
    set_smem(k_edge_encode, edge_fwd_smem());
    SPW_KLAUNCH("k_edge_encode", k_edge_encode, dim3(egrid), dim3(kThreads), edge_fwd_smem(), st, a);
  }
#endif
  // nodes without in-edges keep an all-zero aggregate
  cudaMemsetAsync(ws + L.H2S, 0, (size_t)L.slotsN * nE * sizeof(float), st);
  cudaMemsetAsync(ws + L.P, 0, nP * sizeof(float), st);          // propagation input is zeros (main.py:68)
  cudaMemsetAsync(ws + L.S, 0, nE * sizeof(float), st);          // S^1 = R^1 = W1b.0 = 0
  cudaMemsetAsync(ws + L.R, 0, nE * sizeof(float), st);

  for (int l = 0; l < SPW_N_STEPS; ++l) {                        // Networks.py:83
    const float* Pin = ws + L.P + (size_t)(training ? l : (l & 1)) * nP;
    float* Pout = ws + L.P + (size_t)(training ? l + 1 : ((l + 1) & 1)) * nP;   // unused when l == 4
    float* S = ws + L.S + (size_t)(training ? l : 0) * nE;
    float* R = ws + L.R + (size_t)(training ? l : 0) * nE;
    float* H2S = ws + L.H2S + (size_t)(training ? l : 0) * nE;
    float* G = ws + L.G + (size_t)(training ? l : 0) * nP;
    float* U = ws + L.U + (size_t)(training ? l : 0) * nP;
    if (l > 0) {   // S = P.W1b, R = P.W1c   (sender / receiver parts of rmp layer 0, Networks.py:84-87)
      RowsSeg s = {Pin, kDP, kDP};
      LinOpt o;
      run_linear(st, ws, L, {T_W1B, P_W1B, 0}, n, kDE, 1, &s, S, kDEP, o);
      run_linear(st, ws, L, {T_W1C, P_W1C, 0}, n, kDE, 1, &s, R, kDEP, o);
    }
    if (E > 0) {
      if (!training && l > 0) cudaMemsetAsync(H2S, 0, nE * sizeof(float), st);
      EdgeStepArgs a;
      a.E = E; a.in_snd = g->in_snd; a.in_rcv = g->in_rcv; a.in_off = g->in_off; a.A = ws + L.A; a.S = S; a.R = R;
      a.W2 = PK(P_W2); a.b2 = w->rmp_b[1]; a.H2S = H2S; a.part_first = ws + L.PF; a.part_last = ws + L.PL;
      a.maskbits = training ? reinterpret_cast<uint32_t*>(ws + L.M2) + (size_t)l * E * 8 : nullptr;
#if SPW_USE_TC
      {
        tc::EdgeStepTcArgs t;
        t.E = E; t.in_snd = g->in_snd; t.in_rcv = g->in_rcv; t.in_off = g->in_off; t.A = ws + L.A; t.S = S; t.R = R;
        t.W2hi = ws + L.W2hi; t.W2lo = ws + L.W2lo; t.H2S = H2S; t.part_first = ws + L.PF;
        t.part_last = ws + L.PL; t.maskbits = a.maskbits;
        t.maskbits_h1 = training ? reinterpret_cast<uint32_t*>(ws + L.M1) + (size_t)l * E * 8 : nullptr;
        const int ttiles = (E + kTM - 1) / kTM;
        const int tgrid = ttiles < num_sms() ? ttiles : num_sms();
        if (use_pipe()) {
          set_smem(tc::k_edge_step_p, tc::kEdgeStepPSmem);
          SPW_KLAUNCH("k_edge_step_p", tc::k_edge_step_p, dim3(tgrid), dim3(tc::kPipeThreads), tc::kEdgeStepPSmem, st, t);
        } else {
          set_smem(tc::k_edge_step_tc, tc::kEdgeStepTcSmem);
          SPW_KLAUNCH("k_edge_step_tc", tc::k_edge_step_tc, dim3(tgrid), dim3(tc::kStThreads), tc::kEdgeStepTcSmem, st, t);
        }
        if (ttiles > 1)
          SPW_KLAUNCH("k_fix_boundaries", k_fix_boundaries, dim3(grid_for(ttiles - 1, 8)), dim3(256), 0, st, E, (int)kTM, g->in_rcv, ws + L.PF, ws + L.PL, H2S);
      }
#else
      set_smem(k_edge_step, edge_fwd_smem());
      SPW_KLAUNCH("k_edge_step", k_edge_step, dim3(egrid), dim3(kThreads), edge_fwd_smem(), st, a);
      if (etiles > 1)
        SPW_KLAUNCH("k_fix_boundaries", k_fix_boundaries, dim3(grid_for(etiles - 1, 8)), dim3(256), 0, st, E, (int)kTME, g->in_rcv, ws + L.PF, ws + L.PL, H2S);
#endif
    }
    {   // g = tanh(W3.sum h2 + deg.b3)   (Networks.py:87-88)
      RowsSeg s = {H2S, kDEP, kDE};
      LinOpt o; o.bias = w->rmp_b[2]; o.rowscale = ws + L.degf; o.act = 2;
      run_linear(st, ws, L, {T_W3, P_W3, 0}, n, kDP, 1, &s, G, kDP, o);
    }
    {   // u = relu(V1.[q, g, p] + c1) = relu(qv + [g | p].[V1b ; V1c])    (Networks.py:89-90, hidden layer of omp)
      RowsSeg s[2] = {{G, kDP, kDP}, {Pin, kDP, kDP}};
      LinOpt o; o.addend = ws + L.QV; o.ld_add = kDP; o.act = 1;
      run_linear(st, ws, L, {T_V1BC, P_V1B, P_V1C}, n, kDP, l == 0 ? 1 : 2, s, U, kDP, o);   // p^0 = 0: skip its segment
    }
    if (l < SPW_N_STEPS - 1) {   // p = tanh(z[1:] + p)   (Networks.py:80,91)
      RowsSeg s = {U, kDP, kDP};
      LinOpt o; o.bias = w->omp_b[1] + 1; o.addend = Pin; o.ld_add = kDP; o.act = 2;
      run_linear(st, ws, L, {T_V2P, P_V2P, 0}, n, kDP, 1, &s, Pout, kDP, o);
    } else {                     // head: channel 0 of the last z (Networks.py:93-96)
      SPW_KLAUNCH("k_logit", k_logit, dim3(grid_for(n, 8)), dim3(256), 0, st, U, n, w->omp_w[1], w->omp_b[1], logits, probs);
    }
  }
  return check_launch("spw_forward");
}

size_t spw_forward_towers_bytes(int32_t n_nodes, int32_t n_edges) {
  if (n_nodes < 0 || n_edges < 0) return 0;
  return (size_t)n_edges * kDEP * sizeof(float);        // A_e = c_e.W1a + b1, one 152-float row per edge
}

int spw_forward_towers(const SpwParams* w, const SpwGraph* g, int32_t max_nodes_per_tower, const float* obj, float* logits,
                       float* probs, void* workspace, size_t workspace_bytes, void* stream) {
  int rc;
  if ((rc = check_params(w, "spw_forward_towers")) != SPW_OK) return rc;
  if ((rc = check_graph(g)) != SPW_OK) return rc;
  if (max_nodes_per_tower < 0) return fail(SPW_ERR_BAD_ARG, "spw_forward_towers: negative max_nodes_per_tower");
  if (max_nodes_per_tower > SPW_SMALL_MAX_NODES)
    return fail(SPW_ERR_UNSUPPORTED, "spw_forward_towers: %d blocks in a tower, limit is %d", max_nodes_per_tower, SPW_SMALL_MAX_NODES);
  const int n = g->n_nodes, E = g->n_edges;
  if (n == 0 || g->n_towers == 0) return SPW_OK;
  if (!obj || !logits) return fail(SPW_ERR_BAD_ARG, "spw_forward_towers: null pointer");
  if (!aligned16(obj) || !aligned16(logits) || (probs && !aligned16(probs)))
    return fail(SPW_ERR_BAD_ARG, "spw_forward_towers: obj, logits or probs not 16-byte aligned");
  const size_t need = spw_forward_towers_bytes(n, E);
  if (workspace_bytes < need) return fail(SPW_ERR_WORKSPACE, "spw_forward_towers: workspace %zu < %zu bytes", workspace_bytes, need);
  if (need > 0 && (!workspace || !aligned16(workspace)))
    return fail(SPW_ERR_BAD_ARG, "spw_forward_towers: workspace null or not 16-byte aligned");
  TowerFwdArgs a;
  a.w = *w; a.node_off = g->node_off; a.in_off = g->in_off; a.in_snd = g->in_snd; a.in_rcv = g->in_rcv; a.obj = obj;
  a.logits = logits; a.probs = probs; a.A = reinterpret_cast<float*>(workspace); a.n_edges = E;
  a.max_nodes = max_nodes_per_tower > 0 ? max_nodes_per_tower : 1;
  const size_t smem = small_smem_bytes(a.max_nodes);
  set_smem(k_tower_forward, smem);
  SPW_KLAUNCH("k_tower_forward", k_tower_forward, dim3(g->n_towers), dim3(kSmallThreads), smem, (cudaStream_t)stream, a);
  return check_launch("spw_forward_towers");
}

size_t spw_backward_towers_bytes(int32_t n_nodes, int32_t n_edges) {
  if (n_nodes < 0 || n_edges < 0) return 0;
  return small_bwd_ws_floats(n_nodes, n_edges) * sizeof(float);   // A_e, d A_e, the node state of every step
}

int spw_backward_towers(const SpwParams* w, const SpwGraph* g, int32_t max_nodes_per_tower, const float* obj,
                        const float* dlogits, const float* dprobs, float* logits, float* dobj, float* drel,
                        void* workspace, size_t workspace_bytes, void* stream) {
  int rc;
  if ((rc = check_params(w, "spw_backward_towers")) != SPW_OK) return rc;
  if ((rc = check_graph(g)) != SPW_OK) return rc;
  if (max_nodes_per_tower < 0) return fail(SPW_ERR_BAD_ARG, "spw_backward_towers: negative max_nodes_per_tower");
  if (max_nodes_per_tower > SPW_SMALL_MAX_NODES)
    return fail(SPW_ERR_UNSUPPORTED, "spw_backward_towers: %d blocks in a tower, limit is %d", max_nodes_per_tower, SPW_SMALL_MAX_NODES);
  const int n = g->n_nodes, E = g->n_edges;
  if (n == 0 || g->n_towers == 0) return SPW_OK;
  if (!obj || !dobj) return fail(SPW_ERR_BAD_ARG, "spw_backward_towers: null pointer");
  if (!dlogits && !dprobs) return fail(SPW_ERR_BAD_ARG, "spw_backward_towers: null seed (dlogits and dprobs both null)");
  if (!aligned16(obj) || !aligned16(dobj) || (logits && !aligned16(logits)))
    return fail(SPW_ERR_BAD_ARG, "spw_backward_towers: obj, dobj or logits not 16-byte aligned");
  if (reinterpret_cast<uintptr_t>(drel) % sizeof(float) || reinterpret_cast<uintptr_t>(dlogits) % sizeof(float) ||
      reinterpret_cast<uintptr_t>(dprobs) % sizeof(float))
    return fail(SPW_ERR_BAD_ARG, "spw_backward_towers: dlogits, dprobs or drel not 4-byte aligned");
  const size_t need = spw_backward_towers_bytes(n, E);
  if (workspace_bytes < need) return fail(SPW_ERR_WORKSPACE, "spw_backward_towers: workspace %zu < %zu bytes", workspace_bytes, need);
  if (!workspace || !aligned16(workspace)) return fail(SPW_ERR_BAD_ARG, "spw_backward_towers: workspace null or not 16-byte aligned");
  float* ws = reinterpret_cast<float*>(workspace);
  TowerBwdArgs a;
  a.f.w = *w; a.f.node_off = g->node_off; a.f.in_off = g->in_off; a.f.in_snd = g->in_snd; a.f.in_rcv = g->in_rcv; a.f.obj = obj;
  a.f.logits = logits; a.f.probs = nullptr; a.f.A = ws; a.f.n_edges = E;
  a.f.max_nodes = max_nodes_per_tower > 0 ? max_nodes_per_tower : 1;
  a.out_off = g->out_off; a.out_pos = g->out_pos; a.dlogits = dlogits; a.dprobs = dprobs; a.dobj = dobj;
  a.drel = E > 0 ? drel : nullptr; a.dA = ws + (size_t)E * kDEP; a.ns = ws + (size_t)2 * E * kDEP;
  const size_t smem = small_bwd_smem_bytes(a.f.max_nodes);
  set_smem(k_tower_backward, smem);
  SPW_KLAUNCH("k_tower_backward", k_tower_backward, dim3(g->n_towers), dim3(kSmallThreads), smem, (cudaStream_t)stream, a);
  return check_launch("spw_backward_towers");
}

int spw_bce_grad(const float* logits, const float* target, int32_t n_nodes, double count, float* dlogits, double* stats,
                 void* stream) {
  if (n_nodes < 0 || count <= 0) return fail(SPW_ERR_BAD_ARG, "spw_bce_grad: bad size");
  if (n_nodes == 0) return SPW_OK;
  if (!logits || !target || !dlogits || !stats) return fail(SPW_ERR_BAD_ARG, "spw_bce_grad: null pointer");
  SPW_KLAUNCH("k_bce_grad", k_bce_grad, dim3(grid_for(n_nodes, 256)), dim3(256), 0, (cudaStream_t)stream, logits, target, (int)n_nodes,
             1.0 / count, dlogits, stats);
  return check_launch("spw_bce_grad");
}

}  // extern "C"

namespace {
// The backward pass of the row-major data path (round 1; the only one of the FFMA build).  grads == null (spw_backward_obj):
// no weight gradient is reduced; dobj != null: d obj [n][3] from the layer-0 gradients (k_obj_grad_c, spw_obj_grad.cuh);
// drel != null: d drel [E] with respect to the relation weights (k_rel_grad_step / k_rel_grad_enc, spw_rel_grad.cuh);
// ig != null: the gradients with respect to the dense relation tensors and the propagation input (spw_input_grad.cuh; dS / dR
// slot 0 take step 0's sender / receiver sums, and d prop is formed in place).
int backward_rows(const SpwParams* w, const SpwGraph* g, const float* obj, const float* dlogits, void* workspace,
                  size_t workspace_bytes, const SpwParams* grads, float dropout_rate, void* stream, float* dobj, float* drel,
                  const InputGradTarget* ig = nullptr) {
  const int n = g->n_nodes, E = g->n_edges;
  const float inv_keep = dropout_rate > 0.f ? 1.f / (1.f - dropout_rate) : 1.f;
  const Layout L = make_layout(n, E, 1);
  if (workspace_bytes < L.total * sizeof(float))
    return fail(SPW_ERR_WORKSPACE, "spw_backward: workspace %zu < %zu bytes", workspace_bytes, L.total * sizeof(float));
  cudaStream_t st = (cudaStream_t)stream;
  float* ws = reinterpret_cast<float*>(workspace);
  auto PK = [&](int id) { return ws + L.pack[id]; };
  const size_t nP = (size_t)n * kDP, nE = (size_t)n * kDEP;
  if (n == 0 && grads) {
    // no data: all gradients are zero
    static const int sizes[22] = {300, 22500, 22500, 22500, 150, 150, 150, 150, 200, 10000, 100, 100,
                                  52500, 22500, 15000, 150, 150, 100, 30000, 10100, 100, 101};
    float* const* p = reinterpret_cast<float* const*>(grads);
    for (int i = 0; i < 22; ++i) cudaMemsetAsync(p[i], 0, sizes[i] * sizeof(float), st);
    return check_launch("spw_backward");
  }
  if (!obj || !dlogits) return fail(SPW_ERR_BAD_ARG, "spw_backward: null pointer");
  const int etiles = (E + kTM - 1) / kTM;
  int egrid = etiles < num_sms() ? etiles : num_sms();
  if (egrid > kMaxCtas) egrid = kMaxCtas;         // the per-CTA partial buffers (partE) hold kMaxCtas entries
  float* partN = ws + L.partN;

  // head: dUpre^5 = dlogit (x) V2[:,0] * relu'
  float* dU5 = ws + L.dU + 4 * nP;
  const float* U5 = ws + L.U + 4 * nP;
  SPW_KLAUNCH("k_logit_bwd", k_logit_bwd, dim3(grid_for((int64_t)n * kDP, 256)), dim3(256), 0, st, dlogits, U5, n, w->omp_w[1], dU5);
  const InputGradScratch IS = input_grad_scratch(n, E);
  if (ig) {   // h2_0: the hidden state of the message of an all-zero relation column
    ZeroMessageArgs z;
    for (int i = 0; i < 4; ++i) { z.rm_w[i] = w->rm_w[i]; z.rm_b[i] = w->rm_b[i]; }
    z.w1a = w->rmp_w[0]; z.b1 = w->rmp_b[0]; z.w2 = w->rmp_w[1]; z.b2 = w->rmp_b[1]; z.h2_0 = ig->scratch + IS.H20;
    SPW_KLAUNCH_PDL("k_zero_message", k_zero_message, dim3(1), dim3(256), 0, st, z);
  }

  for (int l = SPW_N_STEPS - 1; l >= 0; --l) {   // step l+1 of the forward loop
    const float* Pin = ws + L.P + (size_t)l * nP;
    const float* S = ws + L.S + (size_t)l * nE;
    const float* R = ws + L.R + (size_t)l * nE;
    const float* G = ws + L.G + (size_t)l * nP;
    const float* U = ws + L.U + (size_t)l * nP;
    float* dU = ws + L.dU + (size_t)l * nP;
    float* dG = ws + L.dG + (size_t)l * nP;
    const float* Tl = l < 4 ? ws + L.T + (size_t)l * nP : nullptr;   // d(pre-tanh of p^{l+1})
    if (l < SPW_N_STEPS - 1) {   // dUpre = (T.V2p^T) * relu'(u)
      RowsSeg s = {Tl, kDP, kDP};
      LinOpt o; o.mulsrc = U; o.ld_mul = kDP; o.mulmode = 1;
      run_linear(st, ws, L, {T_V2PT, P_V2PT, 0}, n, kDP, 1, &s, dU, kDP, o);
    }
    {   // dq_pre += (dUpre.V1a^T) * relu'(q)
      RowsSeg s = {dU, kDP, kDP};
      LinOpt o; o.mulsrc = ws + L.Q; o.ld_mul = kDP; o.mulmode = 1; o.accumulate = l < SPW_N_STEPS - 1; o.post_scale = inv_keep;
      run_linear(st, ws, L, {T_V1AT, P_V1AT, 0}, n, kDP, 1, &s, ws + L.dQ, kDP, o);
    }
    {   // dg_pre = (dUpre.V1b^T) * (1 - g^2)
      RowsSeg s = {dU, kDP, kDP};
      LinOpt o; o.mulsrc = G; o.ld_mul = kDP; o.mulmode = 2;
      run_linear(st, ws, L, {T_V1BT, P_V1BT, 0}, n, kDP, 1, &s, dG, kDP, o);
    }
    if (l > 0 || ig) {   // DP = dUpre.V1c^T (+ residual T); step 0: the first term of d prop, in place
      RowsSeg s = {dU, kDP, kDP};
      LinOpt o; o.addend = Tl; o.ld_add = kDP;
      run_linear(st, ws, L, {T_V1CT, P_V1CT, 0}, n, kDP, 1, &s, l > 0 ? ws + L.DP : ig->dprop, kDP, o);
    }
    {   // d(sum h2) = dg_pre.W3^T
      RowsSeg s = {dG, kDP, kDP};
      LinOpt o;
      run_linear(st, ws, L, {T_W3T, P_W3T, 0}, n, kDE, 1, &s, ws + L.dH2S, kDEP, o);
    }
    if (E > 0) {
      EdgeStepBwdArgs a;
      a.E = E; a.in_snd = g->in_snd; a.in_rcv = g->in_rcv; a.A = ws + L.A; a.S = S; a.R = R;
      a.W2T = PK(P_W2T); a.dH2S = ws + L.dH2S; a.dA = ws + L.dA; a.DH1 = ws + L.DH1;
      a.maskbits = reinterpret_cast<const uint32_t*>(ws + L.M2) + (size_t)l * E * 8;
      a.partW2 = ws + L.partE; a.first = (l == SPW_N_STEPS - 1);
#if SPW_USE_TC
      {
        tc::WgradTcArgs wg;
        wg.M = E; wg.x_mode = 1; wg.X = ws + L.A; wg.S = S; wg.R = R; wg.in_snd = g->in_snd; wg.in_rcv = g->in_rcv;
        wg.y_mode = 1; wg.dY = ws + L.dH2S; wg.maskbits = a.maskbits; wg.part = ws + L.partE; wg.first = a.first;
        wg.poison = ws + L.partE;
        auto kwg = tc::k_wgrad_tc<1, 1>;
        set_smem(kwg, tc::kWgradTcSmem);
        SPW_KLAUNCH("k_wgrad_tc", kwg, dim3(egrid), dim3(tc::kWgThreads), tc::kWgradTcSmem, st, wg);
        tc::EdgeDgradTcArgs t;
        t.E = E; t.in_rcv = g->in_rcv; t.dH2S = ws + L.dH2S; t.Whi = ws + L.W2Thi; t.Wlo = ws + L.W2Tlo;
        t.maskbits = a.maskbits; t.maskbits_h1 = reinterpret_cast<const uint32_t*>(ws + L.M1) + (size_t)l * E * 8;
        t.act = nullptr; t.scale = 1.f; t.dA = ws + L.dA; t.DH1 = ws + L.DH1; t.first = a.first; t.poison = ws + L.dA;
        if (use_pipe()) {
          set_smem(tc::k_edge_dgrad_p, tc::kEdgeDgradPSmem);
          SPW_KLAUNCH("k_edge_dgrad_p", tc::k_edge_dgrad_p, dim3(egrid), dim3(tc::kPipeThreads), tc::kEdgeDgradPSmem, st, t);
        } else {
          set_smem(tc::k_edge_dgrad_tc, tc::kEdgeDgradTcSmem);
          SPW_KLAUNCH("k_edge_dgrad_tc", tc::k_edge_dgrad_tc, dim3(egrid), dim3(tc::kDgThreads), tc::kEdgeDgradTcSmem, st, t);
        }
      }
#else
      {
        auto kw = k_edge_step_bwd<true>;
        set_smem(kw, edge_bwd_smem());
        SPW_KLAUNCH("k_edge_step_bwd", kw, dim3(egrid), dim3(kThreads), edge_bwd_smem(), st, a);
      }
#endif
      if (drel) {   // this step's term of d drel, before the next step overwrites DH1 and dH2S
        RelGradStepArgs r;
        r.E = E; r.in_snd = g->in_snd; r.in_rcv = g->in_rcv; r.DH1 = ws + L.DH1; r.A = ws + L.A; r.e_ld = kDEP;
        r.S = l > 0 ? S : nullptr; r.R = l > 0 ? R : nullptr; r.s_ld = kDEP; r.dH2S = ws + L.dH2S; r.h_ld = kDEP;
        r.bits_h2 = reinterpret_cast<const uint8_t*>(a.maskbits); r.bits_rows = 0; r.dG = dG; r.g_ld = kDP;
        r.b2 = w->rmp_b[1]; r.b3 = w->rmp_b[2]; r.first = a.first; r.drel = drel;
        SPW_KLAUNCH_PDL("k_rel_grad_step", k_rel_grad_step<false>, dim3(grid_for(E, 256)), dim3(256), 0, st, r);
      }
    }
    if (ig) {   // this step's terms of d Rs, d Rr and of the inactive slots, before the next step overwrites DH1 and dH2S
      float* H2 = ig->scratch + IS.H2;
      if (E > 0) {
        H2RowsArgs h;
        h.E = E; h.in_snd = g->in_snd; h.in_rcv = g->in_rcv; h.A = ws + L.A; h.S = l > 0 ? S : nullptr; h.R = l > 0 ? R : nullptr;
        h.bits_h2 = reinterpret_cast<const uint32_t*>(ws + L.M2) + (size_t)l * E * 8; h.w2 = w->rmp_w[1]; h.b2 = w->rmp_b[1]; h.H2 = H2;
        SPW_KLAUNCH_PDL("k_h2_rows", k_h2_rows, dim3(grid_for((int64_t)E * kDEP, 256)), dim3(256), 0, st, h);
      }
      InputGradStepArgs a;
      a.T = g->n_towers; a.node_off = g->node_off; a.in_off = g->in_off; a.max_nodes = ig->max_nodes;
      a.DH1 = ws + L.DH1; a.H2 = H2; a.e_ld = kDEP; a.S = l > 0 ? S : nullptr; a.R = l > 0 ? R : nullptr; a.s_ld = kDEP;
      a.dH2S = ws + L.dH2S; a.h_ld = kDEP; a.dG = dG; a.g_ld = kDP; a.b3 = w->rmp_b[2]; a.h2_0 = ig->scratch + IS.H20;
      a.first = l == SPW_N_STEPS - 1; a.drs = ig->drs; a.drr = ig->drr; a.drr_free = ig->drr_free;
      const size_t sm = input_grad_step_smem(ig->max_nodes);
      set_smem(k_input_grad_step<false>, sm);
      SPW_KLAUNCH_PDL("k_input_grad_step", k_input_grad_step<false>, dim3(g->n_towers), dim3(256), sm, st, a);
    }
    if (l > 0 || ig) {
      float* dS = ws + L.dS + (size_t)(l > 0 ? l - 1 : 0) * nE;
      float* dR = ws + L.dR + (size_t)(l > 0 ? l - 1 : 0) * nE;
      if (E > 0) {
        SPW_KLAUNCH("k_gather_dsr", k_gather_dsr, dim3(grid_for(n, 8)), dim3(256), 0, st, n, g->in_off, g->out_off, g->out_pos,
                   ws + L.DH1, dS, dR);
      } else {
        cudaMemsetAsync(dS, 0, nE * sizeof(float), st);
        cudaMemsetAsync(dR, 0, nE * sizeof(float), st);
      }
      // T^{l} = (dS.W1b^T + dR.W1c^T + DP) * (1 - (p^l)^2)       (p^l = Pin of this step)
      //   two K = 150 products: the first one is added into DP, the second one finishes T
      RowsSeg s1 = {dS, kDEP, kDE}, s2 = {dR, kDEP, kDE};
      LinOpt o1; o1.accumulate = 1;
      if (l == 0) {   // d prop += dS^0.W1b^T + dR^0.W1c^T: the l > 0 expression below where 1 - (p^0)^2 = 1
        run_linear(st, ws, L, {T_W1BT, P_W1BT, 0}, n, kDP, 1, &s1, ig->dprop, kDP, o1);
        run_linear(st, ws, L, {T_W1CT, P_W1CT, 0}, n, kDP, 1, &s2, ig->dprop, kDP, o1);
        continue;
      }
      run_linear(st, ws, L, {T_W1BT, P_W1BT, 0}, n, kDP, 1, &s1, ws + L.DP, kDP, o1);
      LinOpt o; o.addend = ws + L.DP; o.ld_add = kDP; o.mulsrc = Pin; o.ld_mul = kDP; o.mulmode = 2;
      run_linear(st, ws, L, {T_W1CT, P_W1CT, 0}, n, kDP, 1, &s2, ws + L.T + (size_t)(l - 1) * nP, kDP, o);
    }
  }

  // ---- node-level weight gradients, each one contraction over all steps' rows -------------------
  const float* degf = ws + L.degf;
  if (grads) {
    // omp layer 0 = [V1a; V1b; V1c], bias c1
    launch_wgrad(st, 5 * n, ws + L.Q, kDP, kDP, n, nullptr, 0, ws + L.dU, kDP, kDP, partN, {grads->omp_w[0], 100, 0, 0, grads->omp_b[0], 0});
    launch_wgrad(st, 5 * n, ws + L.G, kDP, kDP, 0, nullptr, 0, ws + L.dU, kDP, kDP, partN, {grads->omp_w[0], 100, 100, 0, nullptr, 0});
    launch_wgrad(st, 5 * n, ws + L.P, kDP, kDP, 0, nullptr, 0, ws + L.dU, kDP, kDP, partN, {grads->omp_w[0], 100, 200, 0, nullptr, 0});
    // omp layer 1: channels 1..100 from T (steps 1..4), channel 0 from the head
    launch_wgrad(st, 4 * n, ws + L.U, kDP, kDP, 0, nullptr, 0, ws + L.T, kDP, kDP, partN, {grads->omp_w[1], 101, 0, 1, grads->omp_b[1], 1});
    launch_wgrad(st, n, U5, kDP, kDP, 0, nullptr, 0, dlogits, 1, 1, partN, {grads->omp_w[1], 101, 0, 0, grads->omp_b[1], 0});
    // rmp layer 2 (W3, b3 scaled by in-degree)
    launch_wgrad(st, 5 * n, ws + L.H2S, kDEP, kDE, 0, degf, n, ws + L.dG, kDP, kDP, partN, {grads->rmp_w[2], 100, 0, 0, grads->rmp_b[2], 0});
    // rmp layer 0 rows 150..349 (W1b, W1c): X = p^{l} for steps 2..5
    launch_wgrad(st, 4 * n, ws + L.P + nP, kDP, kDP, 0, nullptr, 0, ws + L.dS, kDEP, kDE, partN, {grads->rmp_w[0], 150, 150, 0, nullptr, 0});
    launch_wgrad(st, 4 * n, ws + L.P + nP, kDP, kDP, 0, nullptr, 0, ws + L.dR, kDEP, kDE, partN, {grads->rmp_w[0], 150, 250, 0, nullptr, 0});
    // object encoder
    launch_wgrad(st, n, ws + L.Q1, kDP, kDP, 0, nullptr, 0, ws + L.dQ, kDP, kDP, partN, {grads->om_w[1], 100, 0, 0, grads->om_b[1], 0});
  }
  {
    RowsSeg s = {ws + L.dQ, kDP, kDP};
    LinOpt o; o.mulsrc = ws + L.Q1; o.ld_mul = kDP; o.mulmode = 1;
    run_linear(st, ws, L, {T_OM1T, P_OM1T, 0}, n, kDP, 1, &s, ws + L.dQ1, kDP, o);
  }
  if (grads) launch_wgrad(st, n, obj + 1, 3, 2, 0, nullptr, 0, ws + L.dQ1, kDP, kDP, partN, {grads->om_w[0], 100, 0, 0, grads->om_b[0], 0});

  // ---- edge-level weight gradients --------------------------------------------------------------
  if (E > 0) {
    // rmp layer 1 (W2, b2) from the per-step kernel's per-CTA partials
#if SPW_USE_TC
    launch_reduce(st, ws + L.partE, egrid, (int)tc::kWgPartFloats, 0, -1, tc::kWgFeat1, kDE, kDE, {grads->rmp_w[1], 150, 0, 0, grads->rmp_b[1], 0});
#else
    if (grads) launch_reduce(st, ws + L.partE, egrid, 160 * 160, 0, 10, 10, kDE, kDE, {grads->rmp_w[1], 150, 0, 0, grads->rmp_b[1], 0});
#endif
#if SPW_USE_TC
    {   // relation-encoder backward, layer by layer on the tensor cores (activations X0, X1, X2, C saved by the forward pass)
      const float* acts[4] = {ws + L.EC, ws + L.EX2, ws + L.EX1, ws + L.EX0};       // layer inputs: C, X2, X1, X0
      float* gw[4] = {grads->rmp_w[0], grads->rm_w[3], grads->rm_w[2], grads->rm_w[1]};
      float* gb[4] = {grads->rmp_b[0], grads->rm_b[3], grads->rm_b[2], grads->rm_b[1]};
      const float* dY = ws + L.dA;
      float* gout[2] = {ws + L.DH1, ws + L.GB};
      auto kwg = tc::k_wgrad_tc<0, 0>;
      set_smem(kwg, tc::kWgradTcSmem);
      for (int i = 0; i < 4; ++i) {
        tc::WgradTcArgs wg;
        memset(&wg, 0, sizeof(wg));
        wg.M = E; wg.x_mode = 0; wg.X = acts[i]; wg.y_mode = 0; wg.dY = dY; wg.part = ws + L.partE; wg.first = 1; wg.poison = ws + L.partE;
        SPW_KLAUNCH("k_wgrad_tc", kwg, dim3(egrid), dim3(tc::kWgThreads), tc::kWgradTcSmem, st, wg);
        launch_reduce(st, ws + L.partE, egrid, (int)tc::kWgPartFloats, 0, -1, tc::kWgFeat1, kDE, kDE, {gw[i], 150, 0, 0, gb[i], 0});
        // data gradient of the layer: (dY . W^T) * relu'(layer input), times 1/keep through the dropout on c_e
        RowsSeg sg = {dY, kDEP, kDE};
        LinOpt o; o.mulmode = 3; o.post_scale = i == 0 ? inv_keep : 1.f;
        o.bits_in = reinterpret_cast<const uint32_t*>(ws + L.EB) + (size_t)(3 - i) * E * 8;     // bits of C, X2, X1, X0
        o.tag = "k_rows_tc<160>:enc_bwd";
        if (E >= 64 * kTM * 2) launch_rows_pair(st, ws, L, 4 + i, E, dY, gout[i & 1], o); else
        launch_rows_tc_raw(st, ws + L.ENCT + (size_t)(2 * i) * 24320, ws + L.ENCT + (size_t)(2 * i + 1) * 24320, 160, E, kDE, 1, &sg,
                           gout[i & 1], kDEP, o);
        dY = gout[i & 1];
      }
      const int g0grid = etiles < 2 * num_sms() ? etiles : 2 * num_sms();
      SPW_KLAUNCH("k_enc0_bwd", tc::k_enc0_bwd, dim3(g0grid), dim3(tc::kEnc0Threads), 0, st, E, g->in_snd, g->in_rcv, obj, dY, ws + L.part0);
      launch_reduce(st, ws + L.part0, g0grid, 3 * kDEP, kDEP, 0, 0, 2, kDE, {grads->rm_w[0], 150, 0, 0, grads->rm_b[0], 0});
    }
#else
    const int btiles = (E + kTMB - 1) / kTMB;
    const int bgrid = btiles < num_sms() ? btiles : num_sms();
    EdgeEncBwdArgs a;
    a.E = E; a.in_snd = g->in_snd; a.in_rcv = g->in_rcv; a.obj = obj; a.W0 = w->rm_w[0]; a.b0 = w->rm_b[0];
    a.RM1 = PK(P_RM1); a.RM2 = PK(P_RM2); a.RM3 = PK(P_RM3); a.b1 = w->rm_b[1]; a.b2 = w->rm_b[2]; a.b3 = w->rm_b[3];
    a.RM1T = PK(P_RM1T); a.RM2T = PK(P_RM2T); a.RM3T = PK(P_RM3T); a.W1AT = PK(P_W1AT); a.dA = ws + L.dA;
    a.X1 = ws + L.EX1; a.X2 = ws + L.EX2; a.C = ws + L.EC; a.inv_keep = inv_keep;
    a.partM = ws + L.partM; a.part0 = ws + L.part0; a.G0 = dobj || drel || ig ? ws + L.GB : nullptr;
    set_smem(k_edge_encode_bwd, edge_encb_smem());
    SPW_KLAUNCH("k_edge_encode_bwd", k_edge_encode_bwd, dim3(bgrid), dim3(kThreads), edge_encb_smem(), st, a);
    if (grads) {
      const int ps = 4 * 160 * 160;
      launch_reduce(st, ws + L.partM, bgrid, ps, 0, 10, 10, kDE, kDE, {grads->rmp_w[0], 150, 0, 0, grads->rmp_b[0], 0});
      launch_reduce(st, ws + L.partM + 160 * 160, bgrid, ps, 0, 10, 10, kDE, kDE, {grads->rm_w[3], 150, 0, 0, grads->rm_b[3], 0});
      launch_reduce(st, ws + L.partM + 2 * 160 * 160, bgrid, ps, 0, 10, 10, kDE, kDE, {grads->rm_w[2], 150, 0, 0, grads->rm_b[2], 0});
      launch_reduce(st, ws + L.partM + 3 * 160 * 160, bgrid, ps, 0, 10, 10, kDE, kDE, {grads->rm_w[1], 150, 0, 0, grads->rm_b[1], 0});
      // layer 0: part0 rows [w0 row 0 | w0 row 1 | b0], each kDEP long  ->  treat as Kin = 2 (+ bias row)
      launch_reduce(st, ws + L.part0, bgrid, 3 * kDEP, kDEP, 0, 0, 2, kDE, {grads->rm_w[0], 150, 0, 0, grads->rm_b[0], 0});
    }
#endif
  } else if (grads) {
    cudaMemsetAsync(grads->rmp_w[1], 0, 22500 * sizeof(float), st);
    cudaMemsetAsync(grads->rmp_b[1], 0, 150 * sizeof(float), st);
    cudaMemsetAsync(grads->rmp_w[0], 0, 150 * 150 * sizeof(float), st);   // rows 0..149 (rows 150.. written above)
    cudaMemsetAsync(grads->rmp_b[0], 0, 150 * sizeof(float), st);
    for (int i = 0; i < 4; ++i) {
      cudaMemsetAsync(grads->rm_w[i], 0, (i == 0 ? 300 : 22500) * sizeof(float), st);
      cudaMemsetAsync(grads->rm_b[i], 0, 150 * sizeof(float), st);
    }
  }
  if (dobj) {   // d obj from D_e (k_edge_encode_bwd's layer-0 gradient, in GB) and dQ1 (DESIGN.md section 2)
    ObjGradArgs a;
    a.n = n; a.in_off = g->in_off; a.out_off = g->out_off; a.out_pos = g->out_pos;
    a.G0 = ws + L.GB; a.g_ld = kDEP; a.dQ1 = ws + L.dQ1; a.q_ld = kDP;
    a.rm_w0 = w->rm_w[0]; a.om_w0 = w->om_w[0]; a.dobj = dobj;
    SPW_KLAUNCH_PDL("k_obj_grad_c", k_obj_grad_c<false>, dim3(grid_for(n, 256)), dim3(256), 0, st, a);
  }
  if (drel && E > 0) {   // the encoder term of d drel from D_e (in GB)
    RelGradEncArgs a;
    a.E = E; a.in_snd = g->in_snd; a.in_rcv = g->in_rcv; a.obj = obj; a.G0 = ws + L.GB; a.g_ld = kDEP;
    a.rm_w0 = w->rm_w[0]; a.drel = drel;
    SPW_KLAUNCH_PDL("k_rel_grad_enc", k_rel_grad_enc<false>, dim3(grid_for(E, 256)), dim3(256), 0, st, a);
  }
  if (ig && E > 0) {   // the encoder term of d Rs / d Rr from D_e (in GB)
    InputGradEncArgs a;
    a.T = g->n_towers; a.node_off = g->node_off; a.in_off = g->in_off; a.max_nodes = ig->max_nodes; a.obj = obj;
    a.G0 = ws + L.GB; a.g_ld = kDEP; a.rm_w0 = w->rm_w[0]; a.drs = ig->drs; a.drr = ig->drr;
    SPW_KLAUNCH_PDL("k_input_grad_enc", k_input_grad_enc<false>, dim3(g->n_towers), dim3(256), 0, st, a);
  }
  return check_launch(grads ? "spw_backward" : drel ? "spw_backward_rel" : ig ? "spw_backward_inputs" : "spw_backward_obj");
}
}  // namespace

extern "C" {

int spw_backward(const SpwParams* w, const SpwGraph* g, const float* obj, const float* dlogits, void* workspace,
                 size_t workspace_bytes, const SpwParams* grads, float dropout_rate, void* stream) {
  int rc;
  if ((rc = check_params(w, "spw_backward(weights)")) != SPW_OK) return rc;
  if ((rc = check_params(grads, "spw_backward(grads)")) != SPW_OK) return rc;
  if ((rc = check_graph(g)) != SPW_OK) return rc;
  if (!workspace || !aligned16(workspace)) return fail(SPW_ERR_BAD_ARG, "spw_backward: bad workspace");
  if (dropout_rate < 0.f || dropout_rate >= 1.f) return fail(SPW_ERR_BAD_ARG, "spw_backward: dropout rate %g outside [0,1)", dropout_rate);
#if SPW_USE_TC
  if (use_csl() && g->n_nodes > 0) {
    if (!obj || !dlogits) return fail(SPW_ERR_BAD_ARG, "spw_backward: null pointer");
    return backward_csl(w, g, obj, dlogits, reinterpret_cast<float*>(workspace), workspace_bytes, grads, dropout_rate, (cudaStream_t)stream);
  }
#endif
  return backward_rows(w, g, obj, dlogits, workspace, workspace_bytes, grads, dropout_rate, stream, nullptr, nullptr);
}

int spw_backward_obj(const SpwParams* w, const SpwGraph* g, const float* obj, const float* dlogits, void* workspace,
                     size_t workspace_bytes, float dropout_rate, float* dobj, void* stream) {
  int rc;
  if ((rc = check_params(w, "spw_backward_obj")) != SPW_OK) return rc;
  if ((rc = check_graph(g)) != SPW_OK) return rc;
  if (g->n_nodes == 0) return SPW_OK;
  if (!workspace || !aligned16(workspace)) return fail(SPW_ERR_BAD_ARG, "spw_backward_obj: workspace null or not 16-byte aligned");
  if (!obj || !dlogits || !dobj) return fail(SPW_ERR_BAD_ARG, "spw_backward_obj: null pointer");
  if (!aligned16(dobj)) return fail(SPW_ERR_BAD_ARG, "spw_backward_obj: dobj not 16-byte aligned");
  if (dropout_rate < 0.f || dropout_rate >= 1.f) return fail(SPW_ERR_BAD_ARG, "spw_backward_obj: dropout rate %g outside [0,1)", dropout_rate);
#if SPW_USE_TC
  if (!use_csl()) return fail(SPW_ERR_UNSUPPORTED, "spw_backward_obj: not implemented on the round-1 data path (SPW_CSL=0)");
  return backward_csl(w, g, obj, dlogits, reinterpret_cast<float*>(workspace), workspace_bytes, nullptr, dropout_rate, (cudaStream_t)stream, dobj);
#else
  return backward_rows(w, g, obj, dlogits, workspace, workspace_bytes, nullptr, dropout_rate, stream, dobj, nullptr);
#endif
}

int spw_backward_rel(const SpwParams* w, const SpwGraph* g, const float* obj, const float* dlogits, void* workspace,
                     size_t workspace_bytes, float dropout_rate, float* drel, float* dobj, void* stream) {
  int rc;
  if ((rc = check_params(w, "spw_backward_rel")) != SPW_OK) return rc;
  if ((rc = check_graph(g)) != SPW_OK) return rc;
  if (g->n_nodes == 0) return SPW_OK;
  if (!workspace || !aligned16(workspace)) return fail(SPW_ERR_BAD_ARG, "spw_backward_rel: workspace null or not 16-byte aligned");
  if (!obj || !dlogits || (!drel && g->n_edges > 0)) return fail(SPW_ERR_BAD_ARG, "spw_backward_rel: null pointer");
  if (reinterpret_cast<uintptr_t>(drel) % sizeof(float)) return fail(SPW_ERR_BAD_ARG, "spw_backward_rel: drel not 4-byte aligned");
  if (dobj && !aligned16(dobj)) return fail(SPW_ERR_BAD_ARG, "spw_backward_rel: dobj not 16-byte aligned");
  if (dropout_rate < 0.f || dropout_rate >= 1.f) return fail(SPW_ERR_BAD_ARG, "spw_backward_rel: dropout rate %g outside [0,1)", dropout_rate);
  if (g->n_edges == 0 && !dobj) return SPW_OK;
  float* dr = g->n_edges > 0 ? drel : nullptr;
#if SPW_USE_TC
  if (!use_csl()) return fail(SPW_ERR_UNSUPPORTED, "spw_backward_rel: not implemented on the round-1 data path (SPW_CSL=0)");
  return backward_csl(w, g, obj, dlogits, reinterpret_cast<float*>(workspace), workspace_bytes, nullptr, dropout_rate, (cudaStream_t)stream, dobj, dr);
#else
  return backward_rows(w, g, obj, dlogits, workspace, workspace_bytes, nullptr, dropout_rate, stream, dobj, dr);
#endif
}

size_t spw_backward_inputs_bytes(int32_t n_nodes, int32_t n_edges) {
  if (n_nodes < 0 || n_edges < 0) return 0;
  return input_grad_scratch(n_nodes, n_edges).total * sizeof(float);
}

int spw_backward_inputs(const SpwParams* w, const SpwGraph* g, int32_t max_nodes_per_tower, const float* obj, const float* dlogits,
                        void* workspace, size_t workspace_bytes, float dropout_rate, void* scratch, size_t scratch_bytes, float* drs,
                        float* drr, float* drr_free, float* dprop, float* dobj, void* stream) {
  int rc;
  if ((rc = check_params(w, "spw_backward_inputs")) != SPW_OK) return rc;
  if ((rc = check_graph(g)) != SPW_OK) return rc;
  if (max_nodes_per_tower < 0 || max_nodes_per_tower > SPW_MAX_NODES)
    return fail(SPW_ERR_BAD_ARG, "spw_backward_inputs: max_nodes_per_tower %d outside [0, %d]", max_nodes_per_tower, SPW_MAX_NODES);
  if (g->n_nodes == 0) return SPW_OK;
  if (!workspace || !aligned16(workspace)) return fail(SPW_ERR_BAD_ARG, "spw_backward_inputs: workspace null or not 16-byte aligned");
  if (!scratch || !aligned16(scratch)) return fail(SPW_ERR_BAD_ARG, "spw_backward_inputs: scratch null or not 16-byte aligned");
  if (!obj || !dlogits || !drr_free || !dprop || ((!drs || !drr) && g->n_edges > 0))
    return fail(SPW_ERR_BAD_ARG, "spw_backward_inputs: null pointer");
  if (reinterpret_cast<uintptr_t>(drs) % sizeof(float) || reinterpret_cast<uintptr_t>(drr) % sizeof(float) ||
      reinterpret_cast<uintptr_t>(drr_free) % sizeof(float))
    return fail(SPW_ERR_BAD_ARG, "spw_backward_inputs: drs, drr or drr_free not 4-byte aligned");
  if (!aligned16(dprop)) return fail(SPW_ERR_BAD_ARG, "spw_backward_inputs: dprop not 16-byte aligned");
  if (dobj && !aligned16(dobj)) return fail(SPW_ERR_BAD_ARG, "spw_backward_inputs: dobj not 16-byte aligned");
  if (dropout_rate < 0.f || dropout_rate >= 1.f) return fail(SPW_ERR_BAD_ARG, "spw_backward_inputs: dropout rate %g outside [0,1)", dropout_rate);
  const size_t need = spw_backward_inputs_bytes(g->n_nodes, g->n_edges);
  if (scratch_bytes < need) return fail(SPW_ERR_WORKSPACE, "spw_backward_inputs: scratch %zu < %zu bytes", scratch_bytes, need);
  InputGradTarget t;
  t.max_nodes = max_nodes_per_tower; t.scratch = reinterpret_cast<float*>(scratch);
  t.drs = drs; t.drr = drr; t.drr_free = drr_free; t.dprop = dprop;
#if SPW_USE_TC
  if (!use_csl()) return fail(SPW_ERR_UNSUPPORTED, "spw_backward_inputs: not implemented on the round-1 data path (SPW_CSL=0)");
  return backward_csl(w, g, obj, dlogits, reinterpret_cast<float*>(workspace), workspace_bytes, nullptr, dropout_rate, (cudaStream_t)stream, dobj,
                      nullptr, &t);
#else
  return backward_rows(w, g, obj, dlogits, workspace, workspace_bytes, nullptr, dropout_rate, stream, dobj, nullptr, &t);
#endif
}

}  // extern "C"
