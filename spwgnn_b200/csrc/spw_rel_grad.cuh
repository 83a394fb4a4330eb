// spw_rel_grad.cuh -- gradient of sum_i dlogits[i]*logit[i] with respect to the relation weights (spw_backward_rel, DESIGN.md
// section 2).  Relation e = s -> r gets a weight w_e multiplying both of its one-hot entries; drel[e] = d/dw_e at w = 1:
//   drel[e] = u_e . dpos_e + sum over the steps of ( <DH1_e, A_e + 2 (S_s + R_r)> + <G_e, b2> + <dG_r, b3> )
// with, per step, DH1_e the gradient w.r.t. pre1_e = A_e + S_s + R_r (rmp layer 0), G_e = relu'(h2_e) * dSh2_r (the masked
// gathered gradient k_edge_dgrad_c forms), dG_r the gradient w.r.t. the pre-tanh aggregate, and u_e the layer-0 encoder
// gradient of k_obj_grad_c (edge_u, spw_obj_grad.cuh).  <DH1, pre1 + S + R> is evaluated as <DH1, A + 2 (S + R)> on the
// stored A, S, R (the message term <DH1, pre1> and the gather term <DH1, S + R> folded into one dot product).
//   k_rel_grad_step: one launch per step, right after that step's k_edge_dgrad_c (DH1 and dH2S are overwritten by the next
//                    step); thread = receiver-major relation row.  Step 0 (S = R = 0): S = R = null, nothing is gathered.
//   k_rel_grad_enc:  the encoder term, after the last encoder data gradient (D_e in GB).
// Every sum is one fixed-order chain per relation (columns ascending; DH1 term, G term, dG term; steps 5..1, then the encoder
// term), so reruns are bit-identical.  Only the 150 real columns of the relation rows are read.
// Plain CUDA: the host emulator (tools/cuemu) compiles it unchanged.
#pragma once
#include "spw_common.cuh"
#include "spw_obj_grad.cuh"

namespace spw {

struct RelGradStepArgs {
  int E;
  const int32_t* in_snd; const int32_t* in_rcv;
  const float* DH1; const float* A; long long e_ld;     // [E][150]: column slab (e_ld = slab floats) or row-major (e_ld = kDEP)
  const float* S; const float* R; long long s_ld;       // [n][150] of the step, or null in step 0 (p = 0)
  const float* dH2S; long long h_ld;                    // [n][150] d(sum h2) of the step
  const uint8_t* bits_h2; long long bits_rows;          // relu'(h2) of the step: byte slab [19][bits_rows] / words [E][8]
  const float* dG; long long g_ld;                      // [n][100] of the step
  const float* b2; const float* b3;                     // rmp.b1 [150], rmp.b2 [100]
  int first;                                            // drel is written (first processed step) or added to
  float* drel;                                          // [E]
};

// relu'(h2) bits of columns 4q .. 4q+3 of relation e, in bits 0..3
template <bool SLAB>
__device__ __forceinline__ uint32_t h2_nibble(const uint8_t* bits, long long bits_rows, long long e, int q) {
  if (SLAB) return (uint32_t)bits[(long long)(q >> 1) * bits_rows + e] >> (4 * (q & 1));
  return reinterpret_cast<const uint32_t*>(bits)[e * 8 + (q >> 3)] >> (4 * (q & 7));
}

template <bool SLAB>
__global__ void __launch_bounds__(256) k_rel_grad_step(RelGradStepArgs a) {
  __shared__ float sb2[kDEP];
  __shared__ float sb3[kDP];
  pdl_trigger();
  for (int c = threadIdx.x; c < kDEP; c += blockDim.x) {        // biases: written by no kernel of the pass
    sb2[c] = c < kDE ? a.b2[c] : 0.f;
    if (c < kDP) sb3[c] = a.b3[c];
  }
  __syncthreads();
  pdl_wait();
  for (long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x; e < a.E; e += (long long)gridDim.x * blockDim.x) {
    const long long s = a.in_snd[e], r = a.in_rcv[e];
    float acc = 0.f;
    // <DH1_e, A_e + 2 (S_s + R_r)>
#pragma unroll 2
    for (int q = 0; q < 37; ++q) {
      const float4 d = *reinterpret_cast<const float4*>(quad_ptr<SLAB>(a.DH1, a.e_ld, e, q));
      float4 v = *reinterpret_cast<const float4*>(quad_ptr<SLAB>(a.A, a.e_ld, e, q));
      if (a.S) {
        const float4 x = *reinterpret_cast<const float4*>(quad_ptr<SLAB>(a.S, a.s_ld, s, q));
        const float4 y = *reinterpret_cast<const float4*>(quad_ptr<SLAB>(a.R, a.s_ld, r, q));
        v.x = fmaf(2.f, x.x + y.x, v.x); v.y = fmaf(2.f, x.y + y.y, v.y);
        v.z = fmaf(2.f, x.z + y.z, v.z); v.w = fmaf(2.f, x.w + y.w, v.w);
      }
      acc = fmaf(d.x, v.x, acc); acc = fmaf(d.y, v.y, acc); acc = fmaf(d.z, v.z, acc); acc = fmaf(d.w, v.w, acc);
    }
    {   // columns 148, 149 (150: ones, 151: pad)
      const float2 d = *reinterpret_cast<const float2*>(quad_ptr<SLAB>(a.DH1, a.e_ld, e, 37));
      float2 v = *reinterpret_cast<const float2*>(quad_ptr<SLAB>(a.A, a.e_ld, e, 37));
      if (a.S) {
        const float2 x = *reinterpret_cast<const float2*>(quad_ptr<SLAB>(a.S, a.s_ld, s, 37));
        const float2 y = *reinterpret_cast<const float2*>(quad_ptr<SLAB>(a.R, a.s_ld, r, 37));
        v.x = fmaf(2.f, x.x + y.x, v.x); v.y = fmaf(2.f, x.y + y.y, v.y);
      }
      acc = fmaf(d.x, v.x, acc); acc = fmaf(d.y, v.y, acc);
    }
    // <relu'(h2_e) * dSh2_r, b2>
#pragma unroll 2
    for (int q = 0; q < 37; ++q) {
      const float4 h = *reinterpret_cast<const float4*>(quad_ptr<SLAB>(a.dH2S, a.h_ld, r, q));
      const uint32_t m = h2_nibble<SLAB>(a.bits_h2, a.bits_rows, e, q);
      acc = fmaf((m & 1u) ? h.x : 0.f, sb2[4 * q], acc); acc = fmaf((m & 2u) ? h.y : 0.f, sb2[4 * q + 1], acc);
      acc = fmaf((m & 4u) ? h.z : 0.f, sb2[4 * q + 2], acc); acc = fmaf((m & 8u) ? h.w : 0.f, sb2[4 * q + 3], acc);
    }
    {
      const float2 h = *reinterpret_cast<const float2*>(quad_ptr<SLAB>(a.dH2S, a.h_ld, r, 37));
      const uint32_t m = h2_nibble<SLAB>(a.bits_h2, a.bits_rows, e, 37);
      acc = fmaf((m & 1u) ? h.x : 0.f, sb2[148], acc); acc = fmaf((m & 2u) ? h.y : 0.f, sb2[149], acc);
    }
    // <dG_r, b3>
#pragma unroll 5
    for (int q = 0; q < kDP / 4; ++q) {
      const float4 g = *reinterpret_cast<const float4*>(quad_ptr<SLAB>(a.dG, a.g_ld, r, q));
      acc = fmaf(g.x, sb3[4 * q], acc); acc = fmaf(g.y, sb3[4 * q + 1], acc);
      acc = fmaf(g.z, sb3[4 * q + 2], acc); acc = fmaf(g.w, sb3[4 * q + 3], acc);
    }
    a.drel[e] = a.first ? acc : a.drel[e] + acc;
  }
}

struct RelGradEncArgs {
  int E;
  const int32_t* in_snd; const int32_t* in_rcv;
  const float* obj;                     // [n][3]
  const float* G0; long long g_ld;      // D_e, as ObjGradArgs::G0
  const float* rm_w0;                   // [2][150] Keras layout
  float* drel;                          // [E], added to
};

// drel[e] += u_e . (obj[r, 0:2] - obj[s, 0:2]), the difference formed as the forward pass's encoder input
template <bool SLAB>
__global__ void __launch_bounds__(256) k_rel_grad_enc(RelGradEncArgs a) {
  __shared__ float sw[2][kDEP];
  pdl_trigger();
  for (int c = threadIdx.x; c < kDEP; c += blockDim.x) {
    sw[0][c] = c < kDE ? a.rm_w0[c] : 0.f; sw[1][c] = c < kDE ? a.rm_w0[kDE + c] : 0.f;
  }
  __syncthreads();
  pdl_wait();
  for (long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x; e < a.E; e += (long long)gridDim.x * blockDim.x) {
    const long long s = a.in_snd[e], r = a.in_rcv[e];
    const float dx = a.obj[3 * r] - a.obj[3 * s], dy = a.obj[3 * r + 1] - a.obj[3 * s + 1];
    const float2 u = edge_u<SLAB>(a.G0, a.g_ld, e, sw);
    a.drel[e] += fmaf(u.y, dy, u.x * dx);
  }
}

}  // namespace spw
