// spw_small_grad.cuh -- the backward pass of the one-CTA-per-tower inference (spw_small.cuh): ONE CTA computes one tower's
// logits and their gradients with respect to the block features (as spw_backward_obj) and, optionally, the relation
// weights (as spw_backward_rel), in plain fp32 FFMA (DESIGN.md section 2, "The per-tower backward pass").
//
//   - forward: tower_forward_body, the very code of k_tower_forward, so the logits are its bits; it also leaves the node
//     state of every step (q1, q, g^l, p^l, u^l, S^l, R^l, the logit) in the workspace, and A_e as k_tower_forward does;
//   - seed: dlogit_i = dlogits[i] + dprobs[i] p_i (1 - p_i), p from the kernel's own logit (either pointer may be null);
//   - steps 5..1: the node-level products in shared memory; per 32-relation chunk in CSR order, h1 / h2 are recomputed from
//     A_e + S_s + R_r, G_e = relu'(h2) dSh2_r, DH1_e = (G_e.W2^T) relu'(h1) is added into dA_e (workspace) and into the
//     receiver (CSR order) and sender (out-CSR order) sums of the tower, and the step's term of drel is formed;
//   - encoder: the rm activations are recomputed chunk by chunk (their relu patterns kept as bytes), dA goes back through
//     W1a and rm layers 3..1 to D_e, and u_e = D_e.rm0^T; then dobj as k_obj_grad_c and the encoder term of drel.
// Every sum runs in a fixed order that depends on the tower alone (no atomics): a tower's logits, dobj and drel are the same
// bits at any position in any batch.  Nothing per edge and step is stored.
//
// Plain CUDA (shared memory, __syncthreads, __ldg): the host emulator (tools/cuemu) compiles it unchanged.
#pragma once
#include "spw_common.cuh"
#include "spw_small.cuh"

namespace spw {

struct TowerBwdArgs {
  TowerFwdArgs f;                           // f.logits nullable, f.probs null, f.A: workspace [n_edges][kDEP]
  const int32_t* out_off;
  const int32_t* out_pos;
  const float* dlogits;                     // nullable
  const float* dprobs;                      // nullable (not both)
  float* dobj;                              // [n][3]
  float* drel;                              // nullable: [n_edges], receiver-major rows
  float* dA;                                // workspace: [n_edges][kDEP] (d A_e, then u_e in columns 0, 1)
  float* ns;                                // workspace: [n][kNodeState]
};

// workspace floats: A, dA, node state
__host__ __device__ inline size_t small_bwd_ws_floats(int n, int E) { return (size_t)2 * E * kDEP + (size_t)n * kNodeState; }

constexpr int kSmallParts = kSmallThreads / kSmallChunk;   // partial sums per relation of the drel step term

// shared-memory carve-up (floats) of the backward phase for `maxn` nodes; every array starts on a 16-byte boundary
struct SmallBwdSmem {
  int dU, T, dUs, dG, dH, dS, dR, dl, dgb3, vv, XA, XB, M, part, Wst, ioff, ooff, total;
};
__host__ __device__ inline SmallBwdSmem small_bwd_smem_layout(int maxn) {
  SmallBwdSmem L;
  const int m4 = (maxn + 1 + 3) / 4 * 4;
  int off = 0;
  L.dU = off; off += maxn * kDP;            // d pre-relu of u^l (then dQ1)
  L.T = off; off += maxn * kDP;             // d pre-tanh of p^{l+1}, then d p^l while it is formed
  L.dUs = off; off += maxn * kDP;           // sum over the steps of dU
  L.dG = off; off += maxn * kDP;            // d pre-tanh of g^l (then dq)
  L.dH = off; off += maxn * kDEP;           // d sum h2
  L.dS = off; off += maxn * kDEP;           // sender sums of DH1
  L.dR = off; off += maxn * kDEP;           // receiver sums of DH1
  L.dl = off; off += m4;                    // dlogit
  L.dgb3 = off; off += m4;                  // <dG_i, b3>
  L.vv = off; off += 2 * m4;                // v_i = dQ1_i.om0^T
  L.XA = off; off += kSmallChunk * kDEP;    // edge-chunk rows, ping-pong
  L.XB = off; off += kSmallChunk * kDEP;
  L.M = off; off += kSmallChunk * kDEP;     // relu patterns of the 4 rm layers of a chunk, bytes [4][32][kDEP]
  L.part = off; off += kSmallThreads;       // drel partial sums [32][kSmallParts]
  L.Wst = off; off += 2 * small_w_tile<5, true>();
  L.ioff = off; off += m4;                  // tower-local in_off, out_off (ints)
  L.ooff = off; off += m4;
  L.total = off;
  return L;
}
inline size_t small_bwd_smem_bytes(int maxn) {
  const size_t f = small_smem_bytes(maxn), b = (size_t)small_bwd_smem_layout(maxn).total * sizeof(float);
  return f > b ? f : b;
}

__global__ void __launch_bounds__(kSmallThreads) k_tower_backward(const TowerBwdArgs a) {
  SPW_DYN_SMEM(smem_raw);
  __shared__ int s_bad;
  const int tid = threadIdx.x;
  const TowerFwdArgs& f = a.f;
  const int n0 = f.node_off[blockIdx.x], nt = f.node_off[blockIdx.x + 1] - n0;
  if (nt <= 0) return;
  const float qnan = nanf("");
  int eb = 0, ee = 0, bad = 0;
  if (nt > f.max_nodes) {                     // larger than the caller declared: NaN rows, and its relations' drel if in bounds
    bad = 1;
    eb = f.in_off[n0]; ee = f.in_off[n0 + nt];
    if (a.drel && eb >= 0 && ee <= f.n_edges)
      for (int e = eb + tid; e < ee; e += kSmallThreads) a.drel[e] = qnan;
  } else {
    eb = f.in_off[n0]; ee = f.in_off[n0 + nt];
    bad = tower_malformed(f, n0, nt, eb, ee, &s_bad);
    if (!bad) {                                // the out-CSR: the tower's out-edges are its in-edges, listed by sender
      __syncthreads();                         // every thread has read s_bad before it is reused
      const int ob = a.out_off[n0], oe = a.out_off[n0 + nt];
      if (tid == 0 && (ob < 0 || oe - ob != ee - eb || oe > f.n_edges)) s_bad = 1;
      __syncthreads();
      if (!s_bad) {
        for (int o = ob + tid; o < oe; o += kSmallThreads) {
          const int e = a.out_pos[o];
          if (e < eb || e >= ee) s_bad = 1;
        }
        for (int i = tid; i < nt; i += kSmallThreads)
          if (a.out_off[n0 + i] > a.out_off[n0 + i + 1]) s_bad = 1;
      }
      __syncthreads();
      bad = s_bad;
    }
  }
  if (bad) {
    for (int i = tid; i < nt; i += kSmallThreads) {
      if (f.logits) f.logits[n0 + i] = qnan;
      a.dobj[3 * (size_t)(n0 + i)] = qnan; a.dobj[3 * (size_t)(n0 + i) + 1] = qnan; a.dobj[3 * (size_t)(n0 + i) + 2] = qnan;
    }
    return;
  }
  const int ne = ee - eb;
  float* sm = reinterpret_cast<float*>(smem_raw);
  float* ns = a.ns + (size_t)n0 * kNodeState;
  tower_forward_body(f, sm, n0, nt, eb, ne, ns);
  __syncthreads();

  const SmallBwdSmem L = small_bwd_smem_layout(f.max_nodes);
  float* dU = sm + L.dU;
  float* T = sm + L.T;
  float* dUs = sm + L.dUs;
  float* dG = sm + L.dG;
  float* dH = sm + L.dH;
  float* dS = sm + L.dS;
  float* dR = sm + L.dR;
  float* dl = sm + L.dl;
  float* dgb3 = sm + L.dgb3;
  float* vv = sm + L.vv;
  float* XA = sm + L.XA;
  float* XB = sm + L.XB;
  uint8_t* M = reinterpret_cast<uint8_t*>(sm + L.M);
  float* part = sm + L.part;
  float* Wst = sm + L.Wst;
  int* ioff = reinterpret_cast<int*>(sm + L.ioff);
  int* ooff = reinterpret_cast<int*>(sm + L.ooff);
  const SpwParams& w = f.w;
  const float* obj = f.obj;
  const float* A = f.A;
  float* dA = a.dA;
  float* drel = a.drel;
  auto nsv = [&](int i, int off) -> float* { return ns + (size_t)i * kNodeState + off; };

  // ---- seed and head (Networks.py:93-96): dUpre^5 = dlogit V2[:, 0] relu'(u^5) ---------------------------------------------
  for (int i = tid; i <= nt; i += kSmallThreads) {
    ioff[i] = f.in_off[n0 + i] - eb;
    ooff[i] = a.out_off[n0 + i];
  }
  for (int i = tid; i < nt; i += kSmallThreads) {
    const float z = *nsv(i, kNsZ), p = 1.f / (1.f + expf(-z));
    const float g0 = a.dlogits ? a.dlogits[n0 + i] : 0.f, g1 = a.dprobs ? a.dprobs[n0 + i] : 0.f;
    dl[i] = fmaf(g1, p * (1.f - p), g0);
  }
  __syncthreads();
  for (int idx = tid; idx < nt * kDP; idx += kSmallThreads) {
    const int i = idx / kDP, c = idx - i * kDP;
    const float v = *nsv(i, kNsU + (SPW_N_STEPS - 1) * kDP + c) > 0.f ? dl[i] * __ldg(w.omp_w[1] + (size_t)c * (kDP + 1)) : 0.f;
    dU[idx] = v;
    dUs[idx] = v;
  }
  __syncthreads();

  // ---- five propagation steps in reverse (Networks.py:83-91) ----------------------------------------------------------------
  for (int l = SPW_N_STEPS - 1; l >= 0; --l) {
    if (l < SPW_N_STEPS - 1) {   // dUpre = (T^{l+1}.V2p^T) relu'(u^l)
      small_gemm_t<4>(T, kDP, nt, kDP, w.omp_w[1] + 1, kDP + 1, kDP, Wst, [&](int r, int c, float v) {
        const float d = *nsv(r, kNsU + l * kDP + c) > 0.f ? v : 0.f;
        dU[r * kDP + c] = d;
        dUs[r * kDP + c] += d;
      });
      __syncthreads();
    }
    // dG = (dUpre.V1b^T) (1 - g^2)
    small_gemm_t<4>(dU, kDP, nt, kDP, w.omp_w[0] + (size_t)kDP * kDP, kDP, kDP, Wst, [&](int r, int c, float v) {
      const float g = *nsv(r, kNsG + l * kDP + c);
      dG[r * kDP + c] = v * (1.f - g * g);
    });
    if (l > 0) {   // d p^l = dUpre.V1c^T + T^{l+1} (the residual p^{l+1} = tanh(z[1:] + p^l)), into T
      small_gemm_t<4>(dU, kDP, nt, kDP, w.omp_w[0] + (size_t)2 * kDP * kDP, kDP, kDP, Wst, [&](int r, int c, float v) {
        T[r * kDP + c] = l < SPW_N_STEPS - 1 ? v + T[r * kDP + c] : v;
      });
    }
    __syncthreads();
    if (drel)
      for (int i = tid; i < nt; i += kSmallThreads) {
        float s = 0.f;
        for (int c = 0; c < kDP; ++c) s = fmaf(dG[i * kDP + c], __ldg(w.rmp_b[2] + c), s);
        dgb3[i] = s;
      }
    // d sum h2 = dG.W3^T
    small_gemm_t<5>(dG, kDP, nt, kDP, w.rmp_w[2], kDP, kDE, Wst, [&](int r, int c, float v) { dH[r * kDEP + c] = v; });
    if (l > 0)
      for (int idx = tid; idx < nt * kDEP; idx += kSmallThreads) { dS[idx] = 0.f; dR[idx] = 0.f; }
    __syncthreads();
    for (int c0 = 0; c0 < ne; c0 += kSmallChunk) {
      const int ch = imin(kSmallChunk, ne - c0);
      // h1 = relu(A_e + S[sender] + R[receiver]), as the forward pass
      for (int idx = tid; idx < ch * kDE; idx += kSmallThreads) {
        const int r = idx / kDE, c = idx - r * kDE;
        const int e = eb + c0 + r;
        float v = A[(size_t)e * kDEP + c];
        if (l > 0) v = v + *nsv(__ldg(f.in_snd + e) - n0, kNsS + (l - 1) * 2 * kDEP + c) +
                       *nsv(__ldg(f.in_rcv + e) - n0, kNsS + (l - 1) * 2 * kDEP + kDEP + c);
        XA[r * kDEP + c] = relu_f(v);
      }
      __syncthreads();
      // h2 = relu(h1.W2 + b2), then G = relu'(h2) dSh2[receiver] in place
      small_gemm<5>(XA, kDEP, ch, kDE, w.rmp_w[1], kDE, kDE,
                    Wst, [&](int r, int c, float v) { XB[r * kDEP + c] = relu_f(v + __ldg(w.rmp_b[1] + c)); });
      __syncthreads();
      for (int idx = tid; idx < ch * kDE; idx += kSmallThreads) {
        const int r = idx / kDE, c = idx - r * kDE;
        const int rc = __ldg(f.in_rcv + eb + c0 + r) - n0;
        XB[r * kDEP + c] = XB[r * kDEP + c] > 0.f ? dH[rc * kDEP + c] : 0.f;
      }
      __syncthreads();
      // DH1 = (G.W2^T) relu'(h1), in place of h1
      small_gemm_t<5>(XB, kDEP, ch, kDE, w.rmp_w[1], kDE, kDE, Wst, [&](int r, int c, float v) {
        XA[r * kDEP + c] = XA[r * kDEP + c] > 0.f ? v : 0.f;
      });
      __syncthreads();
      // dA_e += DH1_e
      for (int idx = tid; idx < ch * kDE; idx += kSmallThreads) {
        const int r = idx / kDE, c = idx - r * kDE;
        float* d = dA + (size_t)(eb + c0 + r) * kDEP + c;
        *d = l == SPW_N_STEPS - 1 ? XA[r * kDEP + c] : *d + XA[r * kDEP + c];
      }
      if (l > 0) {   // receiver sums in CSR order, sender sums in out-CSR order (chunk by chunk: out-CSR rows ascend)
        for (int idx = tid; idx < nt * kDE; idx += kSmallThreads) {
          const int i = idx / kDE, c = idx - i * kDE;
          const int e0 = imax(ioff[i], c0), e1 = imin(ioff[i + 1], c0 + ch);
          if (e0 < e1) {
            float h = dR[i * kDEP + c];
            for (int e = e0; e < e1; ++e) h += XA[(e - c0) * kDEP + c];
            dR[i * kDEP + c] = h;
          }
          float h = dS[i * kDEP + c];
          for (int o = ooff[i]; o < ooff[i + 1]; ++o) {
            const int r = __ldg(a.out_pos + o) - eb - c0;
            if (r >= 0 && r < ch) h += XA[r * kDEP + c];
          }
          dS[i * kDEP + c] = h;
        }
      }
      if (drel) {    // this step's term: <DH1_e, A_e + 2 (S_s + R_r)> + <G_e, b2>, kSmallParts column-strided partial sums
        const int r = tid / kSmallParts, j = tid - r * kSmallParts;
        if (r < ch) {
          const int e = eb + c0 + r;
          const float* sp = l > 0 ? nsv(__ldg(f.in_snd + e) - n0, kNsS + (l - 1) * 2 * kDEP) : nullptr;
          const float* rp = l > 0 ? nsv(__ldg(f.in_rcv + e) - n0, kNsS + (l - 1) * 2 * kDEP + kDEP) : nullptr;
          float acc = 0.f;
          for (int c = j; c < kDE; c += kSmallParts) {
            float v = A[(size_t)e * kDEP + c];
            if (l > 0) v = fmaf(2.f, sp[c] + rp[c], v);
            acc = fmaf(XA[r * kDEP + c], v, acc);
          }
          for (int c = j; c < kDE; c += kSmallParts) acc = fmaf(XB[r * kDEP + c], __ldg(w.rmp_b[1] + c), acc);
          part[tid] = acc;
        }
      }
      __syncthreads();
      if (drel && tid < ch) {   // + <dG_r, b3>; written in step 5, added afterwards
        const int e = eb + c0 + tid;
        float acc = part[tid * kSmallParts];
        for (int j = 1; j < kSmallParts; ++j) acc += part[tid * kSmallParts + j];
        acc += dgb3[__ldg(f.in_rcv + e) - n0];
        drel[e] = l == SPW_N_STEPS - 1 ? acc : drel[e] + acc;
      }
      // no barrier: the next chunk writes XA only after its first barrier, which orders these reads of part and XA
    }
    if (l > 0) {   // T^l = (d p^l + dS.W1b^T + dR.W1c^T) (1 - (p^l)^2)
      __syncthreads();
      small_gemm_t<4>(dS, kDEP, nt, kDE, w.rmp_w[0] + (size_t)kDE * kDE, kDE, kDP, Wst,
                      [&](int r, int c, float v) { T[r * kDP + c] += v; });
      __syncthreads();
      small_gemm_t<4>(dR, kDEP, nt, kDE, w.rmp_w[0] + (size_t)(kDE + kDP) * kDE, kDE, kDP, Wst, [&](int r, int c, float v) {
        const float p = *nsv(r, kNsP + (l - 1) * kDP + c);
        T[r * kDP + c] = (T[r * kDP + c] + v) * (1.f - p * p);
      });
    }
    __syncthreads();
  }

  // ---- object encoder: dq = (sum_l dUpre^l . V1a^T) relu'(q), dQ1 = (dq.om1^T) relu'(q1), v_i = dQ1_i.om0^T ------------------
  small_gemm_t<4>(dUs, kDP, nt, kDP, w.omp_w[0], kDP, kDP, Wst, [&](int r, int c, float v) {
    dG[r * kDP + c] = *nsv(r, kNsQ + c) > 0.f ? v : 0.f;
  });
  __syncthreads();
  small_gemm_t<4>(dG, kDP, nt, kDP, w.om_w[1], kDP, kDP, Wst, [&](int r, int c, float v) {
    dU[r * kDP + c] = *nsv(r, kNsQ1 + c) > 0.f ? v : 0.f;
  });
  __syncthreads();
  for (int i = tid; i < nt; i += kSmallThreads) {
    float v0 = 0.f, v1 = 0.f;
    for (int c = 0; c < kDP; ++c) {
      v0 = fmaf(dU[i * kDP + c], __ldg(w.om_w[0] + c), v0);
      v1 = fmaf(dU[i * kDP + c], __ldg(w.om_w[0] + kDP + c), v1);
    }
    vv[2 * i] = v0; vv[2 * i + 1] = v1;
  }

  // ---- relation encoder (Networks.py:46,75), chunk by chunk: recompute X0..C, then dA back to D_e and u_e ---------------------
  const float* rmw[4] = {w.rm_w[1], w.rm_w[2], w.rm_w[3], w.rmp_w[0]};
  const float* rmb[3] = {w.rm_b[1], w.rm_b[2], w.rm_b[3]};
  for (int c0 = 0; c0 < ne; c0 += kSmallChunk) {
    const int ch = imin(kSmallChunk, ne - c0);
    for (int idx = tid; idx < ch * kDE; idx += kSmallThreads) {
      const int r = idx / kDE, c = idx - r * kDE;
      const int e = eb + c0 + r;
      const int s = __ldg(f.in_snd + e), rc = __ldg(f.in_rcv + e);
      const float dx = __ldg(obj + 3 * (size_t)rc) - __ldg(obj + 3 * (size_t)s);
      const float dy = __ldg(obj + 3 * (size_t)rc + 1) - __ldg(obj + 3 * (size_t)s + 1);
      const float x = relu_f(fmaf(dy, __ldg(w.rm_w[0] + kDE + c), fmaf(dx, __ldg(w.rm_w[0] + c), __ldg(w.rm_b[0] + c))));
      XA[r * kDEP + c] = x;
      M[r * kDEP + c] = x > 0.f;
    }
    __syncthreads();
#pragma unroll
    for (int k = 0; k < 3; ++k) {   // X1, X2, C (ping-pong XA -> XB -> XA -> XB) and their relu patterns
      float* X = k & 1 ? XB : XA;
      float* Y = k & 1 ? XA : XB;
      uint8_t* Mk = M + (k + 1) * kSmallChunk * kDEP;
      small_gemm<5>(X, kDEP, ch, kDE, rmw[k], kDE, kDE, Wst, [&](int r, int c, float v) {
        const float y = relu_f(v + __ldg(rmb[k] + c));
        Y[r * kDEP + c] = y;
        Mk[r * kDEP + c] = y > 0.f;
      });
      __syncthreads();
    }
    for (int idx = tid; idx < ch * kDE; idx += kSmallThreads) {   // C is in XB: dA -> XA
      const int r = idx / kDE, c = idx - r * kDE;
      XA[r * kDEP + c] = dA[(size_t)(eb + c0 + r) * kDEP + c];
    }
    __syncthreads();
#pragma unroll
    for (int k = 3; k >= 0; --k) {  // dA.W1a^T, then through rm layers 3, 2, 1 (XA -> XB -> XA -> XB -> XA), each product
      float* X = k & 1 ? XA : XB;   // masked by the relu pattern of its input
      float* Y = k & 1 ? XB : XA;
      const uint8_t* Mk = M + k * kSmallChunk * kDEP;
      small_gemm_t<5>(X, kDEP, ch, kDE, rmw[k], kDE, kDE, Wst, [&](int r, int c, float v) { Y[r * kDEP + c] = Mk[r * kDEP + c] ? v : 0.f; });
      __syncthreads();
    }
    // D_e is in XA; u_e = (D_e.rm0[0, :], D_e.rm0[1, :]) into dA_e columns 0, 1 (read for this chunk above)
    if (tid < ch) {
      const int e = eb + c0 + tid;
      float u0 = 0.f, u1 = 0.f;
      for (int c = 0; c < kDE; ++c) {
        u0 = fmaf(XA[tid * kDEP + c], __ldg(w.rm_w[0] + c), u0);
        u1 = fmaf(XA[tid * kDEP + c], __ldg(w.rm_w[0] + kDE + c), u1);
      }
      dA[(size_t)e * kDEP] = u0; dA[(size_t)e * kDEP + 1] = u1;
      if (drel) {   // + u_e . (obj[r, 0:2] - obj[s, 0:2]), as k_rel_grad_enc
        const int s = __ldg(f.in_snd + e), rc = __ldg(f.in_rcv + e);
        const float dx = __ldg(obj + 3 * (size_t)rc) - __ldg(obj + 3 * (size_t)s);
        const float dy = __ldg(obj + 3 * (size_t)rc + 1) - __ldg(obj + 3 * (size_t)s + 1);
        drel[e] += fmaf(u1, dy, u0 * dx);
      }
    }
    __syncthreads();
  }

  // ---- dobj, as k_obj_grad_c: in-edges in CSR order, out-edges in out-CSR order ----------------------------------------------
  for (int i = tid; i < nt; i += kSmallThreads) {
    float ix = 0.f, iy = 0.f, ox = 0.f, oy = 0.f;
    for (int e = eb + ioff[i]; e < eb + ioff[i + 1]; ++e) { ix += dA[(size_t)e * kDEP]; iy += dA[(size_t)e * kDEP + 1]; }
    for (int o = ooff[i]; o < ooff[i + 1]; ++o) {
      const size_t e = __ldg(a.out_pos + o);
      ox += dA[e * kDEP]; oy += dA[e * kDEP + 1];
    }
    a.dobj[3 * (size_t)(n0 + i)] = ix - ox;
    a.dobj[3 * (size_t)(n0 + i) + 1] = (iy - oy) + vv[2 * i];
    a.dobj[3 * (size_t)(n0 + i) + 2] = vv[2 * i + 1];
  }
}

}  // namespace spw
