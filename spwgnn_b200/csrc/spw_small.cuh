// spw_small.cuh -- inference of small towers: ONE CTA computes one tower's whole forward pass (Networks.py:58-96) in fp32 FFMA.
//
// The tiled path (spw_forward) runs ~47 launches of 128-row tensor-core tiles; a batch-1 predict (JengaBuilder.py:328-329,
// TowerCreator.py:430-431) fills a few dozen rows of each and pays every launch's fixed cost.  Here a tower of N_t <= 32 blocks
// (in-degree <= 31) is one CTA of one launch:
//   - node state (P, Q, QV, S, R, sum h2, G, U) lives in shared memory for the whole kernel;
//   - the per-edge A_e = c_e.W1a + b1 (DESIGN.md section 2) goes to the caller's workspace [E][152]: written once by the
//     relation encoder, read once per propagation step (it stays in L2);
//   - edges are processed in chunks of kSmallChunk rows in CSR (receiver-major) order, relative to the tower's first edge;
//   - weights are read directly from SpwParams in Keras layout (no pack launch).
// Every sum runs in a fixed order that depends on the tower's own data only: a tower's logits are the same bits whatever
// its position in the batch and whatever the other towers are.
//
// Plain CUDA (shared memory, __syncthreads, __ldg): the host emulator (tools/cuemu) compiles it unchanged.
#pragma once
#include "spw_common.cuh"

namespace spw {

constexpr int kSmallThreads = 256;          // 8 warps
constexpr int kSmallWarps = kSmallThreads / 32;
constexpr int kSmallChunk = 32;             // edge rows per chunk = 8 warps x 4 rows

struct TowerFwdArgs {
  SpwParams w;
  const int32_t* node_off;
  const int32_t* in_off;
  const int32_t* in_snd;
  const int32_t* in_rcv;
  const float* obj;
  float* logits;
  float* probs;                             // nullable
  float* A;                                 // workspace: [n_edges][kDEP]
  int n_edges;
  int max_nodes;                            // node capacity of the shared-memory carve-up
};

// shared-memory carve-up (floats) for `maxn` nodes; every array starts on a 16-byte boundary
struct SmallSmem {
  int QV, GP, U, S, R, H, XA, XB, Wst, ioff, total;
};
__host__ __device__ inline SmallSmem small_smem_layout(int maxn) {
  SmallSmem L;
  int off = 0;
  L.QV = off; off += maxn * kDP;            // q.V1a + c1
  L.GP = off; off += maxn * 2 * kDP;        // [g | p] per node (ld 200): K = 200 operand of omp layer 0
  L.U = off; off += maxn * kDP;             // omp hidden layer (and q1 at the start)
  L.S = off; off += maxn * kDEP;            // p.W1b
  L.R = off; off += maxn * kDEP;            // p.W1c
  L.H = off; off += maxn * kDEP;            // sum of h2 over the in-edges
  L.XA = off; off += kSmallChunk * kDEP;    // edge-chunk activations, ping-pong
  L.XB = off; off += kSmallChunk * kDEP;
  L.Wst = off; off += 2 * 32 * 32 * 5;      // weight k-tiles, 2 stages of 32 rows x 160 columns
  L.ioff = off; off += (maxn + 1 + 3) / 4 * 4;   // tower-local in_off (ints)
  L.total = off;
  return L;
}
inline size_t small_smem_bytes(int maxn) { return (size_t)small_smem_layout(maxn).total * sizeof(float); }

// Y[r][c] = epi(r, c, sum_k X[r][k] W[k][c]) for r < M, c < N.  X: shared, row-major, ldx % 4 == 0, 16-byte aligned;
// W: global, Keras layout [K][ldw].  W goes through shared memory in k-tiles of kSmallKT rows (Wst: 2 stages of
// kSmallKT x 32 C floats), the next tile held in registers while the current one is multiplied, so every warp shares one L2
// read of the weights and the L2 latency hides behind the FMAs.  Warp w owns rows [w R, w R + R), lane owns columns
// [lane C, lane C + C).  Each sum is one fmaf chain in increasing k, so the result does not depend on R or on which warp
// computes the row.  Every thread of the CTA must call it (barriers inside); it ends with a barrier before the epilogue.
constexpr int kSmallKT = 32;
// TRANS = false: tile element (kr, c) is W[(k0 + kr) ldw + c] (the product X.W); TRANS = true: it is W[c ldw + k0 + kr] (the
// product X.W^T of the backward pass, W still in Keras layout).  The transposed tile is read 8 k-rows x 4 columns per warp
// (32-byte segments) and staged with rows of 32 C + 4 floats, so neither the global reads nor the shared stores serialise.
template <int C, bool TRANS>
__device__ __forceinline__ int small_w_index(int idx, int& kr, int& c) {
  if (!TRANS) {
    kr = idx / (32 * C); c = idx - kr * 32 * C;
    return idx;
  }
  const int lo = idx & 31, hi = idx >> 5;
  kr = (lo & 7) + 8 * (hi & 3); c = (lo >> 3) + 4 * (hi >> 2);
  return kr * (32 * C + 4) + c;
}
template <int C, bool TRANS = false>
__device__ __forceinline__ void small_w_fetch(float (&pre)[kSmallKT * C / 8], const float* __restrict__ W, int ldw, int K, int N, int k0) {
#pragma unroll
  for (int i = 0; i < kSmallKT * C / 8; ++i) {
    int kr, c;
    small_w_index<C, TRANS>(threadIdx.x + kSmallThreads * i, kr, c);
    pre[i] = (k0 + kr < K && c < N) ? __ldg(TRANS ? W + (size_t)c * ldw + k0 + kr : W + (size_t)(k0 + kr) * ldw + c) : 0.f;
  }
}
template <int C, bool TRANS = false>
__device__ __forceinline__ void small_w_store(const float (&pre)[kSmallKT * C / 8], float* Ws) {
#pragma unroll
  for (int i = 0; i < kSmallKT * C / 8; ++i) {
    int kr, c;
    Ws[small_w_index<C, TRANS>(threadIdx.x + kSmallThreads * i, kr, c)] = pre[i];
  }
}
// staging floats of one k-tile (two are double-buffered in Wst)
template <int C, bool TRANS>
__host__ __device__ constexpr int small_w_tile() { return kSmallKT * (TRANS ? 32 * C + 4 : 32 * C); }

template <int R, int C, bool TRANS, class Epi>
__device__ __forceinline__ void small_gemm_r(const float* X, int ldx, int M, int K, const float* __restrict__ W, int ldw, int N,
                                             float* Wst, const Epi& epi) {
  constexpr int LDW = TRANS ? 32 * C + 4 : 32 * C, TILE = small_w_tile<C, TRANS>();
  static_assert((kSmallKT * 32 * C) % kSmallThreads == 0, "whole tile per thread");
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int r0 = warp * R;
  const bool active = r0 < M;
  float acc[R][C];
  bool rv[R];
#pragma unroll
  for (int i = 0; i < R; ++i) {
    rv[i] = r0 + i < M;
#pragma unroll
    for (int j = 0; j < C; ++j) acc[i][j] = 0.f;
  }
  const int ntile = (K + kSmallKT - 1) / kSmallKT;
  float pre[kSmallKT * C / 8];
  small_w_fetch<C, TRANS>(pre, W, ldw, K, N, 0);
  small_w_store<C, TRANS>(pre, Wst);
  __syncthreads();
  for (int t = 0; t < ntile; ++t) {
    if (t + 1 < ntile) small_w_fetch<C, TRANS>(pre, W, ldw, K, N, (t + 1) * kSmallKT);
    if (active) {
      const float* Ws = Wst + (t & 1) * TILE + lane * C;
      const int k0 = t * kSmallKT, rows = imin(kSmallKT, K - k0);
      int kk = 0;
      for (; kk + 4 <= rows; kk += 4) {
        float x[R][4];
#pragma unroll
        for (int i = 0; i < R; ++i) {
          float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
          if (rv[i]) v = *reinterpret_cast<const float4*>(X + (size_t)(r0 + i) * ldx + k0 + kk);
          x[i][0] = v.x; x[i][1] = v.y; x[i][2] = v.z; x[i][3] = v.w;
        }
#pragma unroll
        for (int q = 0; q < 4; ++q) {
          float wv[C];
#pragma unroll
          for (int j = 0; j < C; ++j) wv[j] = Ws[(kk + q) * LDW + j];
#pragma unroll
          for (int i = 0; i < R; ++i)
#pragma unroll
            for (int j = 0; j < C; ++j) acc[i][j] = fmaf(x[i][q], wv[j], acc[i][j]);
        }
      }
      for (; kk < rows; ++kk) {
#pragma unroll
        for (int i = 0; i < R; ++i) {
          const float xv = rv[i] ? X[(size_t)(r0 + i) * ldx + k0 + kk] : 0.f;
#pragma unroll
          for (int j = 0; j < C; ++j) acc[i][j] = fmaf(xv, Ws[kk * LDW + j], acc[i][j]);
        }
      }
    }
    if (t + 1 < ntile) small_w_store<C, TRANS>(pre, Wst + ((t + 1) & 1) * TILE);
    __syncthreads();
  }
  if (!active) return;
#pragma unroll
  for (int i = 0; i < R; ++i)
#pragma unroll
    for (int j = 0; j < C; ++j)
      if (rv[i] && lane * C + j < N) epi(r0 + i, lane * C + j, acc[i][j]);
}

// rows per warp from the row count (M <= 32): all 8 warps busy at 32 rows, no warp with idle rows below that
template <int C, class Epi>
__device__ __forceinline__ void small_gemm(const float* X, int ldx, int M, int K, const float* __restrict__ W, int ldw, int N,
                                           float* Wst, const Epi& epi) {
  if (M <= kSmallWarps) small_gemm_r<1, C, false>(X, ldx, M, K, W, ldw, N, Wst, epi);
  else if (M <= 2 * kSmallWarps) small_gemm_r<2, C, false>(X, ldx, M, K, W, ldw, N, Wst, epi);
  else small_gemm_r<4, C, false>(X, ldx, M, K, W, ldw, N, Wst, epi);
}
// Y = epi(X.W^T): the same product with W [N][ldw] in Keras layout read transposed (K = its row length used); Wst holds
// 2 small_w_tile<C, true>() floats
template <int C, class Epi>
__device__ __forceinline__ void small_gemm_t(const float* X, int ldx, int M, int K, const float* __restrict__ W, int ldw, int N,
                                             float* Wst, const Epi& epi) {
  if (M <= kSmallWarps) small_gemm_r<1, C, true>(X, ldx, M, K, W, ldw, N, Wst, epi);
  else if (M <= 2 * kSmallWarps) small_gemm_r<2, C, true>(X, ldx, M, K, W, ldw, N, Wst, epi);
  else small_gemm_r<4, C, true>(X, ldx, M, K, W, ldw, N, Wst, epi);
}

// Node state the backward pass (k_tower_backward, spw_small_grad.cuh) takes from the forward: per node, kNodeState floats
// at these offsets (step l of G / U at + kDP l, of P at + kDP (l - 1), of S / R at + 2 kDEP (l - 1); p^0 = S^0 = R^0 = 0 are
// not stored).
constexpr int kNsQ1 = 0, kNsQ = kDP, kNsG = 2 * kDP, kNsP = 7 * kDP, kNsU = 11 * kDP, kNsS = 16 * kDP, kNsZ = kNsS + 8 * kDEP;
constexpr int kNodeState = kNsZ + 4;

// 1 if tower [n0, n0 + nt) must not be computed: edges outside the tower or the edge arrays, offsets going backwards (a
// malformed graph must not index out of bounds).  eb, ee: its in-edge rows.  Every thread of the CTA calls it (barriers inside).
__device__ __forceinline__ int tower_malformed(const TowerFwdArgs& a, int n0, int nt, int eb, int ee, int* s_bad) {
  const int tid = threadIdx.x;
  if (tid == 0) *s_bad = (eb < 0 || ee > a.n_edges || ee < eb) ? 1 : 0;
  __syncthreads();
  if (!*s_bad) {
    for (int e = eb + tid; e < ee; e += kSmallThreads) {
      const int s = a.in_snd[e], r = a.in_rcv[e];
      if (s < n0 || s >= n0 + nt || r < n0 || r >= n0 + nt) *s_bad = 1;
    }
    for (int i = tid; i < nt; i += kSmallThreads)
      if (a.in_off[n0 + i] > a.in_off[n0 + i + 1]) *s_bad = 1;
  }
  __syncthreads();
  return *s_bad;
}

// The forward pass of tower [n0, n0 + nt) with in-edge rows [eb, eb + ne), in shared memory `sm` (small_smem_layout): the
// logit of each block goes to a.logits (and a.probs) when they are set.  save != null: the node state of kNodeState floats
// per block (kNs*) is also written there, for the backward pass; the arithmetic is the same either way.
__device__ __forceinline__ void tower_forward_body(const TowerFwdArgs& a, float* sm, int n0, int nt, int eb, int ne, float* save) {
  const int tid = threadIdx.x;
  const SmallSmem L = small_smem_layout(a.max_nodes);
  float* QV = sm + L.QV;
  float* GP = sm + L.GP;
  float* U = sm + L.U;
  float* S = sm + L.S;
  float* Rr = sm + L.R;
  float* H = sm + L.H;
  float* XA = sm + L.XA;
  float* XB = sm + L.XB;
  float* Wst = sm + L.Wst;
  int* ioff = reinterpret_cast<int*>(sm + L.ioff);
  const SpwParams& w = a.w;
  const float* obj = a.obj;

  // ---- object encoder (Networks.py:47,76): q1 = relu(om0([y, w])) -> U, p = 0 -----------------------------------------------
  for (int i = tid; i <= nt; i += kSmallThreads) ioff[i] = a.in_off[n0 + i] - eb;
  for (int idx = tid; idx < nt * kDP; idx += kSmallThreads) {
    const int i = idx / kDP, c = idx - i * kDP;
    const float y = __ldg(obj + 3 * (size_t)(n0 + i) + 1), wd = __ldg(obj + 3 * (size_t)(n0 + i) + 2);
    U[i * kDP + c] = relu_f(fmaf(wd, __ldg(w.om_w[0] + kDP + c), fmaf(y, __ldg(w.om_w[0] + c), __ldg(w.om_b[0] + c))));
  }
  for (int idx = tid; idx < nt * 2 * kDP; idx += kSmallThreads) GP[idx] = 0.f;
  __syncthreads();
  // q = relu(q1.om1 + b) -> the g half of GP (free until step 0 writes g)
  small_gemm<4>(U, kDP, nt, kDP, w.om_w[1], kDP, kDP,
                Wst, [&](int r, int c, float v) { GP[r * 2 * kDP + c] = relu_f(v + __ldg(w.om_b[1] + c)); });
  __syncthreads();
  if (save) {                                 // q1 (in U) and q (in the g half of GP), both complete at the barrier above
    for (int idx = tid; idx < nt * kDP; idx += kSmallThreads) {
      const int i = idx / kDP, c = idx - i * kDP;
      save[(size_t)i * kNodeState + kNsQ1 + c] = U[i * kDP + c];
      save[(size_t)i * kNodeState + kNsQ + c] = GP[i * 2 * kDP + c];
    }
  }
  // qv = q.V1a + c1: the object-encoding part of omp layer 0, the same in all five steps (Networks.py:89)
  small_gemm<4>(GP, 2 * kDP, nt, kDP, w.omp_w[0], kDP, kDP,
                Wst, [&](int r, int c, float v) { QV[r * kDP + c] = v + __ldg(w.omp_b[0] + c); });

  // ---- relation encoder + A_e (Networks.py:46,75 and the c_e part of :86-87), chunk by chunk ------------------------------------
  for (int c0 = 0; c0 < ne; c0 += kSmallChunk) {
    const int ch = imin(kSmallChunk, ne - c0);
    for (int idx = tid; idx < ch * kDE; idx += kSmallThreads) {
      const int r = idx / kDE, c = idx - r * kDE;
      const int e = eb + c0 + r;
      const int s = __ldg(a.in_snd + e), rc = __ldg(a.in_rcv + e);
      const float dx = __ldg(obj + 3 * (size_t)rc) - __ldg(obj + 3 * (size_t)s);
      const float dy = __ldg(obj + 3 * (size_t)rc + 1) - __ldg(obj + 3 * (size_t)s + 1);
      XA[r * kDEP + c] = relu_f(fmaf(dy, __ldg(w.rm_w[0] + kDE + c), fmaf(dx, __ldg(w.rm_w[0] + c), __ldg(w.rm_b[0] + c))));
    }
    __syncthreads();
    small_gemm<5>(XA, kDEP, ch, kDE, w.rm_w[1], kDE, kDE,
                  Wst, [&](int r, int c, float v) { XB[r * kDEP + c] = relu_f(v + __ldg(w.rm_b[1] + c)); });
    __syncthreads();
    small_gemm<5>(XB, kDEP, ch, kDE, w.rm_w[2], kDE, kDE,
                  Wst, [&](int r, int c, float v) { XA[r * kDEP + c] = relu_f(v + __ldg(w.rm_b[2] + c)); });
    __syncthreads();
    small_gemm<5>(XA, kDEP, ch, kDE, w.rm_w[3], kDE, kDE,
                  Wst, [&](int r, int c, float v) { XB[r * kDEP + c] = relu_f(v + __ldg(w.rm_b[3] + c)); });
    __syncthreads();
    float* Ach = a.A + (size_t)(eb + c0) * kDEP;
    small_gemm<5>(XB, kDEP, ch, kDE, w.rmp_w[0], kDE, kDE,
                  Wst, [&](int r, int c, float v) { Ach[(size_t)r * kDEP + c] = v + __ldg(w.rmp_b[0] + c); });
    // no barrier: the next chunk writes XA only, and the barrier after it orders this read of XB before the next write
  }

  // ---- five propagation steps (Networks.py:83-91) ---------------------------------------------------------------------------
  const float* V1bc = w.omp_w[0] + (size_t)kDP * kDP;       // rows [V1b ; V1c] of omp layer 0 are consecutive: K = 200
  for (int l = 0; l < SPW_N_STEPS; ++l) {
    if (l > 0) {   // S = p.W1b, R = p.W1c (sender / receiver parts of rmp layer 0); both 0 in step 0 (p = 0)
      small_gemm<5>(GP + kDP, 2 * kDP, nt, kDP, w.rmp_w[0] + (size_t)kDE * kDE, kDE, kDE,
                    Wst, [&](int r, int c, float v) { S[r * kDEP + c] = v; });
      small_gemm<5>(GP + kDP, 2 * kDP, nt, kDP, w.rmp_w[0] + (size_t)(kDE + kDP) * kDE, kDE, kDE,
                    Wst, [&](int r, int c, float v) { Rr[r * kDEP + c] = v; });
    }
    for (int idx = tid; idx < nt * kDEP; idx += kSmallThreads) H[idx] = 0.f;
    __syncthreads();
    for (int c0 = 0; c0 < ne; c0 += kSmallChunk) {
      const int ch = imin(kSmallChunk, ne - c0);
      // h1 = relu(A_e + S[sender] + R[receiver])
      for (int idx = tid; idx < ch * kDE; idx += kSmallThreads) {
        const int r = idx / kDE, c = idx - r * kDE;
        const int e = eb + c0 + r;
        float v = a.A[(size_t)e * kDEP + c];
        if (l > 0) v = v + S[(__ldg(a.in_snd + e) - n0) * kDEP + c] + Rr[(__ldg(a.in_rcv + e) - n0) * kDEP + c];
        XA[r * kDEP + c] = relu_f(v);
      }
      __syncthreads();
      // h2 = relu(h1.W2 + b2)
      small_gemm<5>(XA, kDEP, ch, kDE, w.rmp_w[1], kDE, kDE,
                    Wst, [&](int r, int c, float v) { XB[r * kDEP + c] = relu_f(v + __ldg(w.rmp_b[1] + c)); });
      __syncthreads();
      // receiver sums in CSR order: H[i] = (((H[i] + h2_first) + ...) + h2_last) over the in-edges of node i in this chunk
      for (int idx = tid; idx < nt * kDE; idx += kSmallThreads) {
        const int i = idx / kDE, c = idx - i * kDE;
        const int e0 = imax(ioff[i], c0), e1 = imin(ioff[i + 1], c0 + ch);
        if (e0 >= e1) continue;
        float h = H[i * kDEP + c];
        for (int e = e0; e < e1; ++e) h += XB[(e - c0) * kDEP + c];
        H[i * kDEP + c] = h;
      }
      __syncthreads();
    }
    // g = tanh(W3.sum h2 + deg.b3)   (Networks.py:87-88)
    small_gemm<4>(H, kDEP, nt, kDE, w.rmp_w[2], kDP, kDP, Wst, [&](int r, int c, float v) {
      GP[r * 2 * kDP + c] = tanhf(v + (float)(ioff[r + 1] - ioff[r]) * __ldg(w.rmp_b[2] + c));
    });
    __syncthreads();
    // u = relu(qv + [g | p].[V1b ; V1c])   (Networks.py:89-90); p = 0 in step 0: its half is skipped
    small_gemm<4>(GP, 2 * kDP, nt, l == 0 ? kDP : 2 * kDP, V1bc, kDP, kDP,
                  Wst, [&](int r, int c, float v) { U[r * kDP + c] = relu_f(QV[r * kDP + c] + v); });
    __syncthreads();
    if (save) {                  // g^l, p^l, u^l, S^l, R^l: read here, before the p update below writes p^{l+1}
      for (int idx = tid; idx < nt * kDP; idx += kSmallThreads) {
        const int i = idx / kDP, c = idx - i * kDP;
        float* sv = save + (size_t)i * kNodeState;
        sv[kNsG + l * kDP + c] = GP[i * 2 * kDP + c];
        sv[kNsU + l * kDP + c] = U[i * kDP + c];
        if (l > 0) sv[kNsP + (l - 1) * kDP + c] = GP[i * 2 * kDP + kDP + c];
      }
      if (l > 0)
        for (int idx = tid; idx < nt * kDE; idx += kSmallThreads) {
          const int i = idx / kDE, c = idx - i * kDE;
          float* sv = save + (size_t)i * kNodeState + kNsS + (l - 1) * 2 * kDEP;
          sv[c] = S[i * kDEP + c];
          sv[kDEP + c] = Rr[i * kDEP + c];
        }
    }
    if (l < SPW_N_STEPS - 1) {   // p = tanh(z[1:] + p)   (Networks.py:80,91); the update after the last step is dead
      small_gemm<4>(U, kDP, nt, kDP, w.omp_w[1] + 1, kDP + 1, kDP, Wst, [&](int r, int c, float v) {
        float* p = GP + r * 2 * kDP + kDP + c;
        *p = tanhf(v + __ldg(w.omp_b[1] + 1 + c) + *p);
      });
      __syncthreads();
    }
  }
  // ---- head (Networks.py:93-96), as k_logit_c: logit = U5 . V2[:, 0] + c2[0] ---------------------------------------------------
  for (int i = tid; i < nt; i += kSmallThreads) {
    float s = 0.f;
    for (int k = 0; k < kDP; ++k) s = fmaf(U[i * kDP + k], __ldg(w.omp_w[1] + (size_t)k * (kDP + 1)), s);
    const float z = s + __ldg(w.omp_b[1]);
    if (a.logits) a.logits[n0 + i] = z;
    if (save) save[(size_t)i * kNodeState + kNsZ] = z;
    if (a.probs) a.probs[n0 + i] = 1.f / (1.f + expf(-z));
  }
}

__global__ void __launch_bounds__(kSmallThreads) k_tower_forward(const TowerFwdArgs a) {
  SPW_DYN_SMEM(smem_raw);
  __shared__ int s_bad;
  const int tid = threadIdx.x;
  const int n0 = a.node_off[blockIdx.x], nt = a.node_off[blockIdx.x + 1] - n0;
  if (nt <= 0) return;
  const float qnan = nanf("");
  const int eb = nt > a.max_nodes ? 0 : a.in_off[n0], ee = nt > a.max_nodes ? 0 : a.in_off[n0 + nt];
  // larger than the caller declared, or malformed: this tower's rows are NaN, nothing else is written
  if (nt > a.max_nodes || tower_malformed(a, n0, nt, eb, ee, &s_bad)) {
    for (int i = tid; i < nt; i += kSmallThreads) {
      a.logits[n0 + i] = qnan;
      if (a.probs) a.probs[n0 + i] = qnan;
    }
    return;
  }
  tower_forward_body(a, reinterpret_cast<float*>(smem_raw), n0, nt, eb, ee - eb, nullptr);
}

}  // namespace spw
