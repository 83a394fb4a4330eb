// spw_input_grad.cuh -- gradient of sum_i dlogits[i]*logit[i] with respect to every input of the reference's model
// (spw_backward_inputs, DESIGN.md section 2): the dense relation tensors sender_relations / receiver_relations, the
// propagation input and the objects.  Notation of section 2; per step l (input state p^l, p^0 = 0) the backward pass holds
// S^l_j = W1b.p^l_j, R^l_j = W1c.p^l_j, DH1^l_e (gradient w.r.t. pre1_e), dSh2^l_j and dG^l_j (gradient w.r.t. the pre-tanh
// aggregate); h2^l_e is recomputed from the kept h1 (k_lin, or k_h2_rows in the FFMA build).  For relation column e of a tower
// and every block j of that tower:
//   dRs[j,e] = -u_e.(x_j, y_j) + sum_l <DH1^l_e, S^l_j>
//   dRr[j,e] = +u_e.(x_j, y_j) + sum_l ( <DH1^l_e, R^l_j> + <dSh2^l_j, h2^l_e> + <dG^l_j, b3> )
// and, for an inactive (all-zero) column, dRs = 0 and dRr[j] = sum_l ( <dSh2^l_j, h2_0> + <dG^l_j, b3> ), h2_0 being the hidden
// state of the message of a zero input (k_zero_message).
//   k_input_grad_step: one launch per step, right after that step's k_edge_dgrad_c (DH1 and dSh2 are overwritten by the next
//                      step); CTA = tower.  S, R, dSh2 of the tower's blocks are staged in shared memory ([column][block], so a
//                      warp's reads of consecutive blocks hit consecutive banks), DH1 and h2 are streamed; a thread owns one
//                      block and kEpt relations.  Step 0 (S = R = 0) gathers nothing for the S and R terms.
//   k_input_grad_enc:  the encoder term, after the last encoder data gradient (D_e in GB).
// Every value is one fixed-order chain (columns ascending; per column S term into dRs, R term then h2 term into dRr; then
// <dG, b3>; steps 5..1, then the encoder term) that depends on the tower alone, so reruns are bit-identical.
// Plain CUDA: the host emulator (tools/cuemu) compiles it unchanged.
#pragma once
#include "spw_common.cuh"
#include "spw_obj_grad.cuh"

namespace spw {

constexpr int kEpt = 4;   // relations per thread in k_input_grad_step: each staged S / R / dSh2 value feeds 3 kEpt fmas

struct InputGradStepArgs {
  int T;
  const int32_t* node_off; const int32_t* in_off;
  int max_nodes;                                        // row length of drs / drr, and the largest tower staged
  const float* DH1; const float* H2; long long e_ld;     // [E][150] of the step: column slab (e_ld = slab floats) or row-major
  const float* S; const float* R; long long s_ld;       // [n][150] of the step, or null in step 0 (p = 0)
  const float* dH2S; long long h_ld;                    // [n][150] d(sum h2) of the step
  const float* dG; long long g_ld;                      // [n][100] of the step
  const float* b3;                                      // rmp.b2 [100]
  const float* h2_0;                                    // [150] hidden state of the zero-input message
  int first;                                            // outputs are written (first processed step) or added to
  float* drs; float* drr;                               // [E][max_nodes]
  float* drr_free;                                      // [n]
};

__device__ __forceinline__ float f4c(const float4& v, int i) { return i == 0 ? v.x : i == 1 ? v.y : i == 2 ? v.z : v.w; }

inline size_t input_grad_step_smem(int max_nodes) { return (size_t)(3 * kDE * max_nodes + max_nodes + kDP + kDE) * sizeof(float); }

template <bool SLAB, bool HAS_SR>
__device__ __forceinline__ void input_grad_pairs(const InputGradStepArgs& a, const float* sS, const float* sR, const float* sH,
                                                 const float* sGb, int Nt, int e0, int e1) {
  const int ld = a.max_nodes;
  const int groups = (e1 - e0 + kEpt - 1) / kEpt;
  for (int p = threadIdx.x; p < groups * Nt; p += blockDim.x) {
    const int j = p % Nt, e = e0 + (p / Nt) * kEpt;
    long long ek[kEpt];
#pragma unroll
    for (int k = 0; k < kEpt; ++k) ek[k] = e + k < e1 ? e + k : e1 - 1;     // clamped: read, never written
    float as[kEpt], ar[kEpt];
#pragma unroll
    for (int k = 0; k < kEpt; ++k) { as[k] = 0.f; ar[k] = 0.f; }
#pragma unroll 1
    for (int q = 0; q < 38; ++q) {
      float4 d[kEpt], h[kEpt];
#pragma unroll
      for (int k = 0; k < kEpt; ++k) {
        d[k] = *reinterpret_cast<const float4*>(quad_ptr<SLAB>(a.DH1, a.e_ld, ek[k], q));
        h[k] = *reinterpret_cast<const float4*>(quad_ptr<SLAB>(a.H2, a.e_ld, ek[k], q));
      }
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        const int c = 4 * q + i;
        if (c >= kDE) break;                                                 // columns 150 (ones) and 151 (pad)
        const float hv = sH[c * ld + j];
        if (HAS_SR) {
          const float sv = sS[c * ld + j], rv = sR[c * ld + j];
#pragma unroll
          for (int k = 0; k < kEpt; ++k) {
            as[k] = fmaf(f4c(d[k], i), sv, as[k]);
            ar[k] = fmaf(f4c(d[k], i), rv, ar[k]);
            ar[k] = fmaf(f4c(h[k], i), hv, ar[k]);
          }
        } else {
#pragma unroll
          for (int k = 0; k < kEpt; ++k) ar[k] = fmaf(f4c(h[k], i), hv, ar[k]);
        }
      }
    }
#pragma unroll
    for (int k = 0; k < kEpt; ++k) {
      if (e + k >= e1) break;
      const long long o = (long long)(e + k) * ld + j;
      const float r = ar[k] + sGb[j];
      a.drs[o] = a.first ? as[k] : a.drs[o] + as[k];
      a.drr[o] = a.first ? r : a.drr[o] + r;
    }
  }
}

template <bool SLAB>
__global__ void __launch_bounds__(256) k_input_grad_step(InputGradStepArgs a) {
  SPW_DYN_SMEM(smem_raw);
  const int ld = a.max_nodes;
  float* sS = reinterpret_cast<float*>(smem_raw);
  float* sR = sS + kDE * ld;
  float* sH = sR + kDE * ld;
  float* sGb = sH + kDE * ld;                      // <dG_j, b3> per block
  float* sb3 = sGb + ld;
  float* sh0 = sb3 + kDP;
  pdl_trigger();
  for (int c = threadIdx.x; c < kDP; c += blockDim.x) sb3[c] = a.b3[c];     // a weight: written by no kernel of the pass
  pdl_wait();
  for (int c = threadIdx.x; c < kDE; c += blockDim.x) sh0[c] = a.h2_0[c];
  for (int t = blockIdx.x; t < a.T; t += gridDim.x) {
    const int n0 = a.node_off[t], Nt = a.node_off[t + 1] - n0;
    const int e0 = a.in_off[n0], e1 = a.in_off[n0 + Nt];
    if (Nt > ld) {                                 // a tower larger than declared: NaN rows, nothing else
      const float nan = NAN;
      for (long long i = threadIdx.x; i < (long long)(e1 - e0) * ld; i += blockDim.x) {
        a.drs[(long long)e0 * ld + i] = nan; a.drr[(long long)e0 * ld + i] = nan;
      }
      for (int j = threadIdx.x; j < Nt; j += blockDim.x) a.drr_free[n0 + j] = nan;
      continue;
    }
    __syncthreads();                               // the previous tower's pairs are done with the staged tables
    for (int i = threadIdx.x; i < 38 * Nt; i += blockDim.x) {
      const int q = i / Nt, j = i % Nt;
      const float4 h = *reinterpret_cast<const float4*>(quad_ptr<SLAB>(a.dH2S, a.h_ld, n0 + j, q));
      float4 s = make_float4(0.f, 0.f, 0.f, 0.f), r = s;
      if (a.S) {
        s = *reinterpret_cast<const float4*>(quad_ptr<SLAB>(a.S, a.s_ld, n0 + j, q));
        r = *reinterpret_cast<const float4*>(quad_ptr<SLAB>(a.R, a.s_ld, n0 + j, q));
      }
#pragma unroll
      for (int k = 0; k < 4; ++k) {
        const int c = 4 * q + k;
        if (c < kDE) { sS[c * ld + j] = f4c(s, k); sR[c * ld + j] = f4c(r, k); sH[c * ld + j] = f4c(h, k); }
      }
    }
    for (int j = threadIdx.x; j < Nt; j += blockDim.x) {     // <dG_j, b3>, and the inactive-slot value of block j
      float gb = 0.f;
#pragma unroll 5
      for (int q = 0; q < kDP / 4; ++q) {
        const float4 g = *reinterpret_cast<const float4*>(quad_ptr<SLAB>(a.dG, a.g_ld, n0 + j, q));
        gb = fmaf(g.x, sb3[4 * q], gb); gb = fmaf(g.y, sb3[4 * q + 1], gb);
        gb = fmaf(g.z, sb3[4 * q + 2], gb); gb = fmaf(g.w, sb3[4 * q + 3], gb);
      }
      sGb[j] = gb;
      float fr = 0.f;
#pragma unroll 2
      for (int q = 0; q < 38; ++q) {
        const float4 h = *reinterpret_cast<const float4*>(quad_ptr<SLAB>(a.dH2S, a.h_ld, n0 + j, q));
        fr = fmaf(h.x, sh0[4 * q], fr); fr = fmaf(h.y, sh0[4 * q + 1], fr);
        if (q < 37) { fr = fmaf(h.z, sh0[4 * q + 2], fr); fr = fmaf(h.w, sh0[4 * q + 3], fr); }
      }
      fr += gb;
      a.drr_free[n0 + j] = a.first ? fr : a.drr_free[n0 + j] + fr;
    }
    __syncthreads();
    if (a.S) input_grad_pairs<SLAB, true>(a, sS, sR, sH, sGb, Nt, e0, e1);
    else input_grad_pairs<SLAB, false>(a, sS, sR, sH, sGb, Nt, e0, e1);
    if (a.first && Nt < ld) {                      // columns j >= N_t of the tower's rows
      const int pad = ld - Nt;
      for (long long i = threadIdx.x; i < (long long)(e1 - e0) * pad; i += blockDim.x) {
        const long long o = (e0 + i / pad) * ld + Nt + i % pad;
        a.drs[o] = 0.f; a.drr[o] = 0.f;
      }
    }
  }
}

struct InputGradEncArgs {
  int T;
  const int32_t* node_off; const int32_t* in_off;
  int max_nodes;
  const float* obj;                     // [n][3]
  const float* G0; long long g_ld;      // D_e, as ObjGradArgs::G0
  const float* rm_w0;                   // [2][150] Keras layout
  float* drs; float* drr;               // [E][max_nodes], added to
};

// dRr[j,e] += u_e.(x_j, y_j), dRs[j,e] -= u_e.(x_j, y_j) for every block j of relation e's tower; CTA = tower, thread = relation
template <bool SLAB>
__global__ void __launch_bounds__(256) k_input_grad_enc(InputGradEncArgs a) {
  __shared__ float sw[2][kDEP];
  pdl_trigger();
  for (int c = threadIdx.x; c < kDEP; c += blockDim.x) {
    sw[0][c] = c < kDE ? a.rm_w0[c] : 0.f; sw[1][c] = c < kDE ? a.rm_w0[kDE + c] : 0.f;
  }
  __syncthreads();
  pdl_wait();
  for (int t = blockIdx.x; t < a.T; t += gridDim.x) {
    const int n0 = a.node_off[t], Nt = a.node_off[t + 1] - n0;
    if (Nt > a.max_nodes) continue;                // NaN rows already
    const int e0 = a.in_off[n0], e1 = a.in_off[n0 + Nt];
    for (int e = e0 + threadIdx.x; e < e1; e += blockDim.x) {
      const float2 u = edge_u<SLAB>(a.G0, a.g_ld, e, sw);
      float* rs = a.drs + (long long)e * a.max_nodes;
      float* rr = a.drr + (long long)e * a.max_nodes;
      for (int j = 0; j < Nt; ++j) {
        const float v = fmaf(u.y, a.obj[3 * (n0 + j) + 1], u.x * a.obj[3 * (n0 + j)]);
        rr[j] += v; rs[j] -= v;
      }
    }
  }
}

struct ZeroMessageArgs {
  const float* rm_w[4]; const float* rm_b[4];   // relation encoder (Keras layout)
  const float* w1a; const float* b1;            // rmp layer 0 rows 0..149 ([350][150]), bias
  const float* w2; const float* b2;             // rmp layer 1
  float* h2_0;                                  // [152]: columns 150, 151 = 0
};

// h2_0 = relu(W2.relu(W1a.rm(0) + b1) + b2): the hidden state of the message of an all-zero relation column (the dense model
// runs rm and rmp on every column, Networks.py:75,86-87).  One CTA; every output is one fixed-order chain (inputs ascending).
__global__ void __launch_bounds__(256) k_zero_message(ZeroMessageArgs a) {
  __shared__ float x[2][kDEP];
  pdl_trigger();
  pdl_wait();
  const int c = threadIdx.x;
  if (c < kDE) x[0][c] = fmaxf(a.rm_b[0][c], 0.f);                    // rm layer 0 of a zero input: relu(b0)
  __syncthreads();
  int cur = 0;
  for (int layer = 0; layer < 5; ++layer) {                            // rm layers 1..3, rmp layer 0 (W1a), rmp layer 1
    const float* W = layer < 3 ? a.rm_w[layer + 1] : layer == 3 ? a.w1a : a.w2;
    const float* b = layer < 3 ? a.rm_b[layer + 1] : layer == 3 ? a.b1 : a.b2;
    if (c < kDE) {
      float acc = 0.f;
      for (int k = 0; k < kDE; ++k) acc = fmaf(x[cur][k], W[k * kDE + c], acc);
      x[cur ^ 1][c] = fmaxf(acc + b[c], 0.f);
    }
    __syncthreads();
    cur ^= 1;
  }
  if (c < kDEP) a.h2_0[c] = c < kDE ? x[cur][c] : 0.f;
}

// column slab [25 quads][n][4] (slab = n * 4 floats) -> row-major dprop [n][100]; thread = (node, quad)
__global__ void __launch_bounds__(256) k_dprop_rows(const float* src, long long slab, int n, float* dprop) {
  pdl_trigger();
  pdl_wait();
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < (long long)n * (kDP / 4); i += (long long)gridDim.x * blockDim.x) {
    const long long node = i / (kDP / 4);
    const int q = (int)(i % (kDP / 4));
    *reinterpret_cast<float4*>(dprop + node * kDP + 4 * q) = *reinterpret_cast<const float4*>(src + q * slab + node * 4);
  }
}

struct H2RowsArgs {
  int E;
  const int32_t* in_snd; const int32_t* in_rcv;
  const float* A; const float* S; const float* R;        // [E][152], [n][152] (S = R = null: step 0)
  const uint32_t* bits_h2;                               // [E][8] words of the step
  const float* w2; const float* b2;                      // rmp layer 1, Keras layout
  float* H2;                                             // [E][152]
};

// FFMA build (the host emulator): h2_e = relu'(h2) * (h1_e.W2 + b2) with h1_e = relu(A_e + S_s + R_r), masked by the saved
// relu state of h2; thread = (relation, column).
__global__ void __launch_bounds__(256) k_h2_rows(H2RowsArgs a) {
  pdl_trigger();
  pdl_wait();
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < (long long)a.E * kDEP; i += (long long)gridDim.x * blockDim.x) {
    const long long e = i / kDEP;
    const int c = (int)(i % kDEP);
    float v = 0.f;
    if (c < kDE && ((a.bits_h2[e * 8 + (c >> 5)] >> (c & 31)) & 1u)) {
      const long long s = a.in_snd[e], r = a.in_rcv[e];
      float acc = 0.f;
      for (int k = 0; k < kDE; ++k) {
        float h1 = a.A[e * kDEP + k];
        if (a.S) h1 = (h1 + a.S[s * kDEP + k]) + a.R[r * kDEP + k];
        acc = fmaf(fmaxf(h1, 0.f), a.w2[k * kDE + c], acc);
      }
      v = acc + a.b2[c];
    }
    a.H2[e * kDEP + c] = v;
  }
}

// caller-provided scratch of spw_backward_inputs (floats; both builds): H2 [E][152] (column slab or row-major), h2_0 [152],
// the column-slab staging of dprop [26 quads][n][4]
struct InputGradScratch { size_t H2, H20, DP, total; };
inline InputGradScratch input_grad_scratch(int64_t n, int64_t E) {
  InputGradScratch s;
  size_t off = 0;
  auto take = [&](size_t floats) { size_t o = off; off = (off + floats + 63) / 64 * 64; return o; };
  s.H2 = take((size_t)38 * E * 4 + 64);
  s.H20 = take(kDEP);
  s.DP = take((size_t)26 * n * 4);
  s.total = off;
  return s;
}

// what backward_csl / backward_rows receive: the outputs of spw_backward_inputs and its scratch
struct InputGradTarget {
  int max_nodes;
  float* scratch;
  float* drs; float* drr; float* drr_free; float* dprop;
};

}  // namespace spw
