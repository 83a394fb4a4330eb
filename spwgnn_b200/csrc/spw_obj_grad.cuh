// spw_obj_grad.cuh -- gradient of sum_i dlogits[i]*logit[i] with respect to the block features obj = [x, y, width] / 170
// (spw_backward_obj, DESIGN.md section 2), from the layer-0 pre-activation gradients the backward pass already holds:
//   D_e  [E][150]  rm layer 0 (input [x_r - x_s, y_r - y_s] of relation e = s -> r, Networks.py:58-62,75)
//   dQ1  [n][100]  om layer 0 (input [y_i, w_i], Networks.py:65-66,76)
// With u_e = (D_e . rm.w0[0,:], D_e . rm.w0[1,:]) and v_i = (dQ1_i . om.w0[0,:], dQ1_i . om.w0[1,:]):
//   d/dx_i = sum_{e: r(e)=i} u_e.0 - sum_{e: s(e)=i} u_e.0
//   d/dy_i = sum_{e: r(e)=i} u_e.1 - sum_{e: s(e)=i} u_e.1 + v_i.0
//   d/dw_i = v_i.1
// Thread = node.  In-edges are the receiver-major rows [in_off[i], in_off[i+1]), out-edges come through out_off / out_pos, so
// every relation row is read twice, once from each end.  Every sum runs in a fixed order (columns ascending, relations in CSR
// order) that depends on the tower alone: reruns are bit-identical.  Only the 150 real columns of D_e are read.
// Plain CUDA: the host emulator (tools/cuemu) compiles it unchanged.
#pragma once
#include "spw_common.cuh"

namespace spw {

struct ObjGradArgs {
  int n;
  const int32_t* in_off; const int32_t* out_off; const int32_t* out_pos;
  const float* G0; long long g_ld;      // D_e: column slab (g_ld = slab floats) or row-major [E][kDEP] (g_ld = kDEP)
  const float* dQ1; long long q_ld;     // dQ1: column slab [25][n][4] (q_ld = slab floats) or row-major [n][kDP] (q_ld = kDP)
  const float* rm_w0;                   // [2][150] Keras layout
  const float* om_w0;                   // [2][100]
  float* dobj;                          // [n][3], written
};

// columns 4q .. 4q+3 of row r: SLAB = true: column-slab array (quad q at p + q * ld, row r at + 4 r); false: row-major
template <bool SLAB>
__device__ __forceinline__ const float* quad_ptr(const float* p, long long ld, long long r, int q) {
  return SLAB ? p + (long long)q * ld + r * 4 : p + r * ld + 4 * q;
}

// u = (D_r . w[0,:], D_r . w[1,:]) over the 150 real columns, ascending
template <bool SLAB>
__device__ __forceinline__ float2 edge_u(const float* G0, long long ld, long long r, const float (*sw)[kDEP]) {
  float a0 = 0.f, a1 = 0.f;
#pragma unroll 1
  for (int q0 = 0; q0 < 36; q0 += 6) {
    float4 d[6];
#pragma unroll
    for (int k = 0; k < 6; ++k) d[k] = *reinterpret_cast<const float4*>(quad_ptr<SLAB>(G0, ld, r, q0 + k));
#pragma unroll
    for (int k = 0; k < 6; ++k) {
      const int c = 4 * (q0 + k);
      a0 = fmaf(d[k].x, sw[0][c], a0); a1 = fmaf(d[k].x, sw[1][c], a1);
      a0 = fmaf(d[k].y, sw[0][c + 1], a0); a1 = fmaf(d[k].y, sw[1][c + 1], a1);
      a0 = fmaf(d[k].z, sw[0][c + 2], a0); a1 = fmaf(d[k].z, sw[1][c + 2], a1);
      a0 = fmaf(d[k].w, sw[0][c + 3], a0); a1 = fmaf(d[k].w, sw[1][c + 3], a1);
    }
  }
  const float4 d36 = *reinterpret_cast<const float4*>(quad_ptr<SLAB>(G0, ld, r, 36));
  const float2 d37 = *reinterpret_cast<const float2*>(quad_ptr<SLAB>(G0, ld, r, 37));      // columns 148, 149 (150: ones, 151: pad)
  a0 = fmaf(d36.x, sw[0][144], a0); a1 = fmaf(d36.x, sw[1][144], a1);
  a0 = fmaf(d36.y, sw[0][145], a0); a1 = fmaf(d36.y, sw[1][145], a1);
  a0 = fmaf(d36.z, sw[0][146], a0); a1 = fmaf(d36.z, sw[1][146], a1);
  a0 = fmaf(d36.w, sw[0][147], a0); a1 = fmaf(d36.w, sw[1][147], a1);
  a0 = fmaf(d37.x, sw[0][148], a0); a1 = fmaf(d37.x, sw[1][148], a1);
  a0 = fmaf(d37.y, sw[0][149], a0); a1 = fmaf(d37.y, sw[1][149], a1);
  return make_float2(a0, a1);
}

// SLAB = true: column-slab arrays (tensor-core build); false: row-major arrays (FFMA build, the host emulator)
template <bool SLAB>
__global__ void __launch_bounds__(256) k_obj_grad_c(ObjGradArgs a) {
  __shared__ float sw[2][kDEP];
  __shared__ float so[2][kDP];
  pdl_trigger();
  for (int c = threadIdx.x; c < kDEP; c += blockDim.x) {        // weights: written by no kernel of the pass
    sw[0][c] = c < kDE ? a.rm_w0[c] : 0.f; sw[1][c] = c < kDE ? a.rm_w0[kDE + c] : 0.f;
    if (c < kDP) { so[0][c] = a.om_w0[c]; so[1][c] = a.om_w0[kDP + c]; }
  }
  __syncthreads();
  pdl_wait();
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < a.n; i += (long long)gridDim.x * blockDim.x) {
    float ix = 0.f, iy = 0.f, ox = 0.f, oy = 0.f;
    const int i0 = a.in_off[i], i1 = a.in_off[i + 1], o0 = a.out_off[i], o1 = a.out_off[i + 1];
#pragma unroll 2
    for (int e = i0; e < i1; ++e) {
      const float2 u = edge_u<SLAB>(a.G0, a.g_ld, e, sw);
      ix += u.x; iy += u.y;
    }
#pragma unroll 2
    for (int o = o0; o < o1; ++o) {
      const float2 u = edge_u<SLAB>(a.G0, a.g_ld, a.out_pos[o], sw);
      ox += u.x; oy += u.y;
    }
    float v0 = 0.f, v1 = 0.f;
#pragma unroll 5
    for (int q = 0; q < kDP / 4; ++q) {
      const float4 d = *reinterpret_cast<const float4*>(quad_ptr<SLAB>(a.dQ1, a.q_ld, i, q));
      v0 = fmaf(d.x, so[0][4 * q], v0); v1 = fmaf(d.x, so[1][4 * q], v1);
      v0 = fmaf(d.y, so[0][4 * q + 1], v0); v1 = fmaf(d.y, so[1][4 * q + 1], v1);
      v0 = fmaf(d.z, so[0][4 * q + 2], v0); v1 = fmaf(d.z, so[1][4 * q + 2], v1);
      v0 = fmaf(d.w, so[0][4 * q + 3], v0); v1 = fmaf(d.w, so[1][4 * q + 3], v1);
    }
    a.dobj[3 * i] = ix - ox;
    a.dobj[3 * i + 1] = (iy - oy) + v0;
    a.dobj[3 * i + 2] = v1;
  }
}

}  // namespace spw
