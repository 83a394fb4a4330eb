// spw_kernels.cuh -- forward / backward kernels of the propagation network (fp32, sm_100a).
//
// Math (reference: /root/reference/src/Networks.py:58-96, restated in SURVEY.md section 3.3), with
// two exact algebraic refactorings that remove 2.5x of the per-edge multiply-adds:
//   (1) the first relation-propagator layer is linear in its concatenated input
//       (Networks.py:86-87):  W1.[c_e, p_s, p_r] + b1 = (W1a.c_e + b1) + W1b.p_s + W1c.p_r
//       -> A_e = W1a.c_e + b1 once per edge, S_i = W1b.p_i and R_i = W1c.p_i once per NODE per step;
//   (2) its last layer is linear and is followed by the sum over incoming edges
//       (Networks.py:87-88):  sum_e (W3.h2_e + b3) = W3.(sum_e h2_e) + deg_i.b3
//       -> the receiver-segmented sum runs on the 150-wide hidden state, W3 runs once per node.
// Per edge and step only h2 = relu(W2.relu(A_e + S_s + R_r) + b2) remains (one 150x150 layer).
//
// Tiles: 128 rows (edges in receiver-major order, or nodes) x <=160 columns per CTA, 256 threads,
// thread tile 16x5 (or 16x4), activations chained through shared memory, weights streamed
// from L2 (spw_common.cuh).  All reductions run in a fixed order: results are bit-reproducible.
#pragma once
#include "spw_common.cuh"

namespace spw {

// =================================================================================================
// weight packing: Keras [in][out] tensors -> zero-padded [Kp][ldw] matrices (optionally transposed)
// =================================================================================================
struct PackDesc {
  const float* src; int src_ld, row0, col0, K, N, transpose;
  float* dst; int Kp, ldw;
};
constexpr int kMaxPack = 28;
struct PackArgs { PackDesc d[kMaxPack]; int n; };

__global__ void __launch_bounds__(256) k_pack_weights(PackArgs a) {
  const PackDesc d = a.d[blockIdx.y];
  const int total = d.Kp * d.ldw;
  for (int idx = blockIdx.x * blockDim.x + threadIdx.x; idx < total; idx += gridDim.x * blockDim.x) {
    const int k = idx / d.ldw, n = idx - k * d.ldw;
    float v = 0.f;
    if (k < d.K && n < d.N)
      v = d.transpose ? d.src[(size_t)(d.row0 + n) * d.src_ld + d.col0 + k]
                      : d.src[(size_t)(d.row0 + k) * d.src_ld + d.col0 + n];
    d.dst[idx] = v;
  }
}

// FP32 pipe micro-benchmark (roofline denominator for the FFMA kernels; bench.py)
__global__ void __launch_bounds__(256) k_ffma_peak(float* __restrict__ out, int iters) {
  float a[16];
  const float x = 1.0f + 1e-7f * threadIdx.x, y = 1e-9f * blockIdx.x;
#pragma unroll
  for (int i = 0; i < 16; ++i) a[i] = (float)i;
  for (int it = 0; it < iters; ++it) {
#pragma unroll
    for (int i = 0; i < 16; ++i) a[i] = fmaf(a[i], x, y);
  }
  float s = 0.f;
#pragma unroll
  for (int i = 0; i < 16; ++i) s += a[i];
  out[blockIdx.x * blockDim.x + threadIdx.x] = s;
}

// =================================================================================================
// small elementwise / per-node kernels
// =================================================================================================
// object-encoder layer 0 (Networks.py:65-66,71,76; K = 2): out[i][c] = relu(y*W[0][c] + w*W[1][c] + b[c])
__global__ void __launch_bounds__(256) k_obj_enc0(const float* __restrict__ obj, int n, const float* __restrict__ W,
                                                  const float* __restrict__ b, float* __restrict__ out) {
  const int total = n * kDP;
  for (int idx = blockIdx.x * blockDim.x + threadIdx.x; idx < total; idx += gridDim.x * blockDim.x) {
    const int i = idx / kDP, c = idx - i * kDP;
    const float y = obj[3 * (size_t)i + 1], w = obj[3 * (size_t)i + 2];
    out[idx] = relu_f(fmaf(w, W[kDP + c], fmaf(y, W[c], b[c])));
  }
}

__global__ void __launch_bounds__(256) k_deg_to_float(const int32_t* __restrict__ in_off, int n, float* __restrict__ degf) {
  pdl_trigger();
  pdl_wait();
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x)
    degf[i] = (float)(in_off[i + 1] - in_off[i]);
}

// head (Networks.py:93-96): logit_i = U5_i . V2[:,0] + c2[0]; one warp per node
__global__ void __launch_bounds__(256) k_logit(const float* __restrict__ U, int n, const float* __restrict__ V2raw,
                                               const float* __restrict__ c2raw, float* __restrict__ logits,
                                               float* __restrict__ probs) {
  const int lane = threadIdx.x & 31;
  const int wpb = blockDim.x >> 5;
  for (int i = blockIdx.x * wpb + (threadIdx.x >> 5); i < n; i += gridDim.x * wpb) {
    float s = 0.f;
    for (int c = lane; c < kDP; c += 32) s = fmaf(U[(size_t)i * kDP + c], V2raw[(size_t)c * (kDP + 1)], s);
#pragma unroll
    for (int m = 16; m >= 1; m >>= 1) s += __shfl_xor_sync(0xffffffffu, s, m);
    if (lane == 0) {
      const float z = s + c2raw[0];
      logits[i] = z;
      if (probs) probs[i] = 1.f / (1.f + expf(-z));
    }
  }
}

// dUpre5[i][c] = dlogit_i * V2[c][0] * [U5[i][c] > 0]
__global__ void __launch_bounds__(256) k_logit_bwd(const float* __restrict__ dlogits, const float* __restrict__ U, int n,
                                                   const float* __restrict__ V2raw, float* __restrict__ dU) {
  const int total = n * kDP;
  for (int idx = blockIdx.x * blockDim.x + threadIdx.x; idx < total; idx += gridDim.x * blockDim.x) {
    const int i = idx / kDP, c = idx - i * kDP;
    dU[idx] = U[idx] > 0.f ? dlogits[i] * V2raw[(size_t)c * (kDP + 1)] : 0.f;
  }
}

// Keras binary_crossentropy on clipped probabilities + d(mean loss)/d(logit) (Networks.py:102)
__global__ void __launch_bounds__(256) k_bce_grad(const float* __restrict__ logits, const float* __restrict__ target,
                                                  int n, double inv_count, float* __restrict__ dlogits,
                                                  double* __restrict__ stats) {
  __shared__ double s_loss[256];
  __shared__ double s_acc[256];
  double loss = 0.0, correct = 0.0;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
    const float z = logits[i], y = target[i];
    const float p = 1.f / (1.f + expf(-z));
    const float eps = 1e-7f;
    const float pc = fminf(fmaxf(p, eps), 1.f - eps);
    loss += -((double)y * (double)logf(pc) + (1.0 - (double)y) * (double)logf(1.f - pc));
    correct += ((p > 0.5f) == (y > 0.5f)) ? 1.0 : 0.0;
    // d/dz: clip passes gradient only strictly inside (eps, 1-eps); dL/dpc * dp/dz = (pc - y)
    const bool inside = (p > eps) && (p < 1.f - eps);
    dlogits[i] = inside ? (float)((double)(pc - y) * inv_count) : 0.f;
  }
  s_loss[threadIdx.x] = loss; s_acc[threadIdx.x] = correct;
  __syncthreads();
  for (int off = 128; off >= 1; off >>= 1) {
    if ((int)threadIdx.x < off) { s_loss[threadIdx.x] += s_loss[threadIdx.x + off]; s_acc[threadIdx.x] += s_acc[threadIdx.x + off]; }
    __syncthreads();
  }
  if (threadIdx.x == 0) { atomicAdd(&stats[0], s_loss[0]); atomicAdd(&stats[1], s_acc[0]); }
}

// =================================================================================================
// generic fused linear layer on node rows:  Y = post( act( sum_s X_s.W_s + rowscale*bias + addend ) )
// =================================================================================================
struct LinSeg { const float* X; const float* W; int ldx; int K; int Kp; };
struct LinArgs {
  int M, nseg, N;
  LinSeg seg[3];
  const float* bias;       // [N] or null
  const float* rowscale;   // [M] per-row multiplier of the bias (in-degree) or null
  const float* addend;     // [M][ld_add] pre-activation addend or null
  int ld_add;
  int act;                 // 0 none, 1 relu, 2 tanh
  const float* mulsrc;     // post-activation factor source or null
  int ld_mul;
  int mulmode;             // 1: *= [mulsrc > 0]   2: *= (1 - mulsrc^2)
  float* Y; int ldy;       // columns N..ldy-1 are written as 0
  int accumulate;          // Y += result
  float post_scale;        // multiplies the result before accumulation (1/keep in the backward of a dropout)
  uint32_t drop_thresh; uint32_t drop_seed; float drop_inv_keep;   // drop_thresh > 0: inverted dropout after act
};

template <int CN, int TMR>
__global__ void __launch_bounds__(kThreads, (TMR <= 64 ? 2 : 1)) k_linear(LinArgs a) {
  SPW_DYN_SMEM(smem_raw);
  float* smem = reinterpret_cast<float*>(smem_raw);
  constexpr int ROWS = TMR / 8;
  float* Xs[3];
  int off = 0;
  for (int s = 0; s < a.nseg; ++s) { Xs[s] = smem + off; off += TMR * a.seg[s].Kp; }
  float* Wst = smem + off;
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int ntiles = (a.M + TMR - 1) / TMR;
  for (int tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
    const int r0 = tile * TMR;
    const int rows = imin(TMR, a.M - r0);
    for (int s = 0; s < a.nseg; ++s) {
      const LinSeg sg = a.seg[s];
      const int k4 = sg.Kp >> 2;
      for (int idx = tid; idx < TMR * k4; idx += kThreads) {
        const int r = idx / k4, c = (idx - r * k4) << 2;
        float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
        if (r < rows) {
          const float* p = sg.X + (size_t)(r0 + r) * sg.ldx + c;
          if (c + 3 < sg.K) {
            v = *reinterpret_cast<const float4*>(p);
          } else {
            if (c < sg.K) v.x = p[0];
            if (c + 1 < sg.K) v.y = p[1];
            if (c + 2 < sg.K) v.z = p[2];
          }
        }
        *reinterpret_cast<float4*>(Xs[s] + (size_t)r * sg.Kp + c) = v;
      }
    }
    __syncthreads();
    float acc[ROWS][CN];
    zero_acc<ROWS, CN>(acc);
    for (int s = 0; s < a.nseg; ++s)
      gemm_tile_acc<ROWS, CN>(acc, Xs[s], a.seg[s].Kp, warp * ROWS, a.seg[s].W, a.seg[s].Kp, Wst);
    // epilogue (registers -> global)
    const bool vec4 = (CN == 4) && ((a.ldy & 3) == 0) && (lane * 4 + 3 < a.ldy);
#pragma unroll
    for (int r = 0; r < ROWS; ++r) {
      const int row = warp * ROWS + r;
      if (row >= rows) continue;
      const size_t grow = (size_t)(r0 + row);
      const float rs = a.rowscale ? a.rowscale[grow] : 1.f;
      float v[CN];
#pragma unroll
      for (int i = 0; i < CN; ++i) {
        const int col = lane * CN + i;
        float t = 0.f;
        if (col < a.N) {
          t = acc[r][i];
          if (a.bias) t = fmaf(rs, a.bias[col], t);
          if (a.addend) t += a.addend[grow * a.ld_add + col];
          if (a.act == 1) t = relu_f(t);
          else if (a.act == 2) t = tanhf(t);
          if (a.mulmode == 1) t = a.mulsrc[grow * a.ld_mul + col] > 0.f ? t : 0.f;
          else if (a.mulmode == 2) { const float m = a.mulsrc[grow * a.ld_mul + col]; t *= (1.f - m * m); }
          if (a.drop_thresh) t = dropout_apply(t, a.drop_seed, (uint32_t)(grow * 128 + col), a.drop_thresh, a.drop_inv_keep);
          t *= a.post_scale;
          if (a.accumulate) t += a.Y[grow * a.ldy + col];
        }
        v[i] = t;
      }
      if (vec4) {
        *reinterpret_cast<float4*>(a.Y + grow * a.ldy + lane * 4) = make_float4(v[0], v[1], v[2], v[CN - 1]);
      } else {
#pragma unroll
        for (int i = 0; i < CN; ++i) {
          const int col = lane * CN + i;
          if (col < a.ldy) a.Y[grow * a.ldy + col] = v[i];
        }
      }
    }
    __syncthreads();
  }
}

// =================================================================================================
// generic weight gradient on node rows: part[cta] = X^T . dY (+ bias row from a ones / rowscale column)
// =================================================================================================
struct WgArgs {
  int M;                   // rows to contract over
  const float* X; int ldx; int Kin; int xmod;   // X row = r % xmod (xmod = 0: r)
  const float* rowscale;   // value of the virtual column Kin (null: 1.0)
  int rsmod;               // rowscale row = r % rsmod (rsmod = 0: r)
  const float* dY; int ldy; int N;
  float* part;             // [gridDim.x][16*TA * 16*TB]
};

template <int TA, int TB, int TMR, int MINB>
__global__ void __launch_bounds__(kThreads, MINB) k_wgrad(WgArgs a) {
  SPW_DYN_SMEM(smem_raw);
  float* Xs = reinterpret_cast<float*>(smem_raw);
  constexpr int LX = 16 * TA, LY = 16 * TB;
  float* Ys = Xs + TMR * LX;
  const int tid = threadIdx.x;
  float acc[TA][TB];
#pragma unroll
  for (int i = 0; i < TA; ++i)
#pragma unroll
    for (int j = 0; j < TB; ++j) acc[i][j] = 0.f;
  const int ntiles = (a.M + TMR - 1) / TMR;
  const bool xvec = (a.ldx & 3) == 0, yvec = (a.ldy & 3) == 0;
  for (int tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
    const int r0 = tile * TMR;
    const int rows = imin(TMR, a.M - r0);
    for (int idx = tid; idx < TMR * (LX / 4); idx += kThreads) {
      const int r = idx / (LX / 4), c = (idx - r * (LX / 4)) * 4;
      float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
      if (r < rows) {
        const size_t xr = a.xmod ? (size_t)((r0 + r) % a.xmod) : (size_t)(r0 + r);
        const float* p = a.X + xr * a.ldx + c;
        if (xvec && c + 3 < a.Kin) {
          v = *reinterpret_cast<const float4*>(p);
        } else {
          const float one = a.rowscale ? a.rowscale[a.rsmod ? (size_t)((r0 + r) % a.rsmod) : (size_t)(r0 + r)] : 1.f;
          v.x = c < a.Kin ? p[0] : (c == a.Kin ? one : 0.f);
          v.y = c + 1 < a.Kin ? p[1] : (c + 1 == a.Kin ? one : 0.f);
          v.z = c + 2 < a.Kin ? p[2] : (c + 2 == a.Kin ? one : 0.f);
          v.w = c + 3 < a.Kin ? p[3] : (c + 3 == a.Kin ? one : 0.f);
        }
      }
      *reinterpret_cast<float4*>(Xs + (size_t)r * LX + c) = v;
    }
    for (int idx = tid; idx < TMR * (LY / 4); idx += kThreads) {
      const int r = idx / (LY / 4), c = (idx - r * (LY / 4)) * 4;
      float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
      if (r < rows) {
        const float* p = a.dY + (size_t)(r0 + r) * a.ldy + c;
        if (yvec && c + 3 < a.N) {
          v = *reinterpret_cast<const float4*>(p);
        } else {
          if (c < a.N) v.x = p[0];
          if (c + 1 < a.N) v.y = p[1];
          if (c + 2 < a.N) v.z = p[2];
          if (c + 3 < a.N) v.w = p[3];
        }
      }
      *reinterpret_cast<float4*>(Ys + (size_t)r * LY + c) = v;
    }
    __syncthreads();
    wgrad_tile_acc<TA, TB>(acc, Xs, LX, Ys, LY, TMR);
    __syncthreads();
  }
  wgrad_flush<TA, TB, false>(acc, a.part + (size_t)blockIdx.x * (LX * LY));
}

// fixed-order sum over per-CTA partials -> compact Keras-layout gradient (+ bias from row Kin)
struct RedArgs {
  const float* part; int nparts; int part_stride; int src_ld;   // src_ld: row length (linear layout only)
  int TA, TB;                                                   // > 0: thread-major layout of wgrad_flush<TA,TB>;
                                                                // TA < 0: tensor-core layout [2][160][128] of tc::k_wgrad_tc (TB = first feature of tile 1)
  int Kin, N;
  float* dW; int dst_ld, dst_row0, dst_col0;   // null: skip the matrix
  float* db; int db_off;                       // null: skip the bias row
};
// Eight sub-sums per output element: sub-sum g covers parts g, g+8, g+16, ... in order, then the eight are combined in a fixed order --
// deterministic, and 8 independent load chains per element instead of one long dependent one.  On the GPU warp g of a block holds
// sub-sum g and lane = element, elements taken in the order they lie in the partial (tensor-core layout: the feature index runs
// fastest), so that a warp reads 128 contiguous bytes of every part; with eight LANES per element every lane read its own sector.
__device__ __forceinline__ void reduce_parts_body(const RedArgs& a) {
  const int total = (a.Kin + 1) * a.N;
#ifndef SPW_EMU
  __shared__ float sub[8][32];
  const int g = threadIdx.x >> 5, lane = threadIdx.x & 31;
  for (int base = blockIdx.x * 32; base < total; base += gridDim.x * 32) {
    const int idx = base + lane;
    const bool in_range = idx < total;
    int k = 0, n = 0;
    if (in_range) {
      if (a.TA < 0) { n = idx / (a.Kin + 1); k = idx - n * (a.Kin + 1); }
      else { k = idx / a.N; n = idx - k * a.N; }
    }
    const bool want = in_range && !((k == a.Kin && !a.db) || (k < a.Kin && !a.dW));
    float s = 0.f;
    if (want) {
      const float* p;
      if (a.TA > 0) {
        const int ja = k / a.TA, ea = k - ja * a.TA, jb = n / a.TB, eb = n - jb * a.TB;
        p = a.part + (size_t)(ea * a.TB + eb) * kThreads + (ja * 16 + jb);
      } else if (a.TA < 0) {
        p = k < 128 ? a.part + (size_t)n * 128 + k : a.part + (size_t)(160 + n) * 128 + (k - a.TB);
      } else {
        p = a.part + (size_t)k * a.src_ld + n;
      }
#pragma unroll 4
      for (int c = g; c < a.nparts; c += 8) s += p[(size_t)c * a.part_stride];
    }
    sub[g][lane] = s;
    __syncthreads();
    if (g == 0 && want) {
      // fixed combination order: ((s0 + s4) + (s2 + s6)) + ((s1 + s5) + (s3 + s7))
      s = ((sub[0][lane] + sub[4][lane]) + (sub[2][lane] + sub[6][lane])) + ((sub[1][lane] + sub[5][lane]) + (sub[3][lane] + sub[7][lane]));
      if (k < a.Kin) a.dW[(size_t)(a.dst_row0 + k) * a.dst_ld + a.dst_col0 + n] = s;
      else a.db[a.db_off + n] = s;
    }
    __syncthreads();
  }
#else
  // host emulator: the same eight sub-sums and combination order, computed by one thread per element
  const int g = threadIdx.x & 7;
  const int per_block = blockDim.x >> 3;
  for (int base = blockIdx.x * per_block; base < total; base += gridDim.x * per_block) {
    const int idx = base + (threadIdx.x >> 3);
    const bool in_range = idx < total;
    const int k = in_range ? idx / a.N : 0, n = in_range ? idx - k * a.N : 0;
    const bool want = in_range && !((k == a.Kin && !a.db) || (k < a.Kin && !a.dW));
    if (!want || g != 0) continue;
    const float* p;
    if (a.TA > 0) {
      const int ja = k / a.TA, ea = k - ja * a.TA, jb = n / a.TB, eb = n - jb * a.TB;
      p = a.part + (size_t)(ea * a.TB + eb) * kThreads + (ja * 16 + jb);
    } else if (a.TA < 0) {
      p = k < 128 ? a.part + (size_t)n * 128 + k : a.part + (size_t)(160 + n) * 128 + (k - a.TB);
    } else {
      p = a.part + (size_t)k * a.src_ld + n;
    }
    float sub[8];
    for (int gg = 0; gg < 8; ++gg) {
      sub[gg] = 0.f;
      for (int c = gg; c < a.nparts; c += 8) sub[gg] += p[(size_t)c * a.part_stride];
    }
    const float s = ((sub[0] + sub[4]) + (sub[2] + sub[6])) + ((sub[1] + sub[5]) + (sub[3] + sub[7]));
    if (k < a.Kin) a.dW[(size_t)(a.dst_row0 + k) * a.dst_ld + a.dst_col0 + n] = s;
    else a.db[a.db_off + n] = s;
  }
#endif
}
__global__ void __launch_bounds__(256) k_reduce_parts(RedArgs a) {
  pdl_trigger();
  pdl_wait();
  reduce_parts_body(a);
}
#ifndef SPW_EMU
// every reduction of a backward pass in ONE launch (blockIdx.y = job): the fifteen small launches between the weight-gradient kernels
// cost ~12 us each on the dependent-launch chain for ~4 us of memory traffic
constexpr int kMaxRedJobs = 16;
struct RedJobs { RedArgs j[kMaxRedJobs]; };
__global__ void __launch_bounds__(256) k_reduce_multi(const __grid_constant__ RedJobs jobs) {
  pdl_trigger();
  pdl_wait();
  reduce_parts_body(jobs.j[blockIdx.y]);
}
#endif

// =================================================================================================
// edge kernels
// =================================================================================================
// shared helper: activation tile epilogue  dst[row][col] = f(acc) with the bias "ones" column at kDE
//   (col 150 = 1 for valid rows so that a later X^T.dY also yields the bias gradient, col 151 = 0)
template <int ROWS, class F>
__device__ __forceinline__ void store_act_tile(const float (&acc)[ROWS][5], float* dst, int warp, int lane, int rows, F f) {
#pragma unroll
  for (int r = 0; r < ROWS; ++r) {
    const int row = warp * ROWS + r;
#pragma unroll
    for (int i = 0; i < 5; ++i) {
      const int col = lane * 5 + i;
      if (col >= kDEP) continue;
      float v = 0.f;
      if (row < rows) {
        if (col < kDE) v = f(acc[r][i], row, col);
        else if (col == kDE) v = 1.f;
      }
      dst[(size_t)row * kDEP + col] = v;
    }
  }
}

// relation-encoder layer 0 into a shared tile (Networks.py:58-62,69,75; K = 2):
//   X0[r][k] = relu(dx*W0[0][k] + dy*W0[1][k] + b0[k]),   [dx,dy] = pos_receiver - pos_sender
template <int TMR>
__device__ __forceinline__ void build_x0(float* X0, float* sdx, float* sdy, const float* __restrict__ obj,
                                         const int32_t* __restrict__ in_snd, const int32_t* __restrict__ in_rcv, int e0,
                                         int rows, const float* __restrict__ W0, const float* __restrict__ b0) {
  const int tid = threadIdx.x;
  if (tid < TMR) {
    float dx = 0.f, dy = 0.f;
    if (tid < rows) {
      const int s = in_snd[e0 + tid], rc = in_rcv[e0 + tid];
      dx = obj[3 * (size_t)rc] - obj[3 * (size_t)s];
      dy = obj[3 * (size_t)rc + 1] - obj[3 * (size_t)s + 1];
    }
    sdx[tid] = dx; sdy[tid] = dy;
  }
  __syncthreads();
  for (int idx = tid; idx < TMR * kDEP; idx += kThreads) {
    const int r = idx / kDEP, k = idx - r * kDEP;
    float v = 0.f;
    if (r < rows) {
      if (k < kDE) v = relu_f(fmaf(sdy[r], W0[kDE + k], fmaf(sdx[r], W0[k], b0[k])));
      else if (k == kDE) v = 1.f;
    }
    X0[idx] = v;
  }
}

struct EdgeEncArgs {
  int E;
  const int32_t* in_snd; const int32_t* in_rcv;
  const float* obj;
  const float* W0; const float* b0;                       // raw rm.w0 [2][150], rm.b0
  const float* RM1; const float* RM2; const float* RM3;   // packed [152][160]
  const float* b1; const float* b2; const float* b3;      // raw biases [150]
  const float* W1A; const float* bA;                      // packed rmp.w0[0:150], raw rmp.b0
  float* A;                                               // [E][152]
  float* X0; float* X1; float* X2; float* C;              // [E][152] each, training only (null: not saved)
  uint32_t drop_thresh; uint32_t drop_seed; float drop_inv_keep;   // dropout on c_e (Networks.py:77)
};

constexpr int kTME = 64;    // edge-tile rows of the forward edge kernels (two CTAs per SM)

// shared tile [rows][152] -> global rows, 128-bit coalesced
__device__ __forceinline__ void tile_to_global(const float* Xs, float* G, int e0, int rows) {
  for (int idx = threadIdx.x; idx < rows * (kDEP / 4); idx += kThreads)
    reinterpret_cast<float4*>(G + (size_t)e0 * kDEP)[idx] = reinterpret_cast<const float4*>(Xs)[idx];
}
__device__ __forceinline__ void tile_from_global(float* Xs, const float* G, int e0, int rows, int tile_rows) {
  for (int idx = threadIdx.x; idx < tile_rows * (kDEP / 4); idx += kThreads)
    reinterpret_cast<float4*>(Xs)[idx] = idx < rows * (kDEP / 4) ? reinterpret_cast<const float4*>(G + (size_t)e0 * kDEP)[idx]
                                                                 : make_float4(0.f, 0.f, 0.f, 0.f);
}

// K2a: c_e = relu(rm(diff))  (4 layers) and A_e = W1a.c_e + b1, all inside one CTA tile
__global__ void __launch_bounds__(kThreads, 2) k_edge_encode(EdgeEncArgs a) {
  SPW_DYN_SMEM(smem_raw);
  constexpr int ROWS = kTME / 8;
  float* Xa = reinterpret_cast<float*>(smem_raw);
  float* Xb = Xa + kTME * kDEP + 8;
  float* Wst = Xb + kTME * kDEP + 8;
  float* sdx = Wst + 2 * kKT * kLdwE;
  float* sdy = sdx + kTME;
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int ntiles = (a.E + kTME - 1) / kTME;
  for (int tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
    const int e0 = tile * kTME;
    const int rows = imin(kTME, a.E - e0);
    build_x0<kTME>(Xa, sdx, sdy, a.obj, a.in_snd, a.in_rcv, e0, rows, a.W0, a.b0);
    __syncthreads();
    if (a.X0) tile_to_global(Xa, a.X0, e0, rows);
    float acc[ROWS][5];
    zero_acc<ROWS, 5>(acc);
    gemm_tile_acc<ROWS, 5>(acc, Xa, kDEP, warp * ROWS, a.RM1, kDEP, Wst);
    store_act_tile<ROWS>(acc, Xb, warp, lane, rows, [&](float v, int, int c) { return relu_f(v + a.b1[c]); });
    __syncthreads();
    if (a.X1) tile_to_global(Xb, a.X1, e0, rows);
    zero_acc<ROWS, 5>(acc);
    gemm_tile_acc<ROWS, 5>(acc, Xb, kDEP, warp * ROWS, a.RM2, kDEP, Wst);
    store_act_tile<ROWS>(acc, Xa, warp, lane, rows, [&](float v, int, int c) { return relu_f(v + a.b2[c]); });
    __syncthreads();
    if (a.X2) tile_to_global(Xa, a.X2, e0, rows);
    zero_acc<ROWS, 5>(acc);
    gemm_tile_acc<ROWS, 5>(acc, Xa, kDEP, warp * ROWS, a.RM3, kDEP, Wst);
    store_act_tile<ROWS>(acc, Xb, warp, lane, rows, [&](float v, int r, int c) {
      float t = relu_f(v + a.b3[c]);
      if (a.drop_thresh) t = dropout_apply(t, a.drop_seed, (uint32_t)((e0 + r) * 160 + c), a.drop_thresh, a.drop_inv_keep);
      return t;
    });
    __syncthreads();
    if (a.C) tile_to_global(Xb, a.C, e0, rows);
    zero_acc<ROWS, 5>(acc);
    gemm_tile_acc<ROWS, 5>(acc, Xb, kDEP, warp * ROWS, a.W1A, kDEP, Wst);
    // A tile -> Xa (free), then 128-bit coalesced rows to HBM
#pragma unroll
    for (int r = 0; r < ROWS; ++r) {
      const int row = warp * ROWS + r;
#pragma unroll
      for (int i = 0; i < 5; ++i) {
        const int col = lane * 5 + i;
        if (col < kDEP) Xa[(size_t)row * kDEP + col] = col < kDE ? acc[r][i] + a.bA[col] : 0.f;
      }
    }
    __syncthreads();
    for (int idx = tid; idx < rows * (kDEP / 4); idx += kThreads)
      reinterpret_cast<float4*>(a.A + (size_t)e0 * kDEP)[idx] = reinterpret_cast<const float4*>(Xa)[idx];
    __syncthreads();
  }
}

// H1 tile: relu(A_e + S_sender + R_receiver).  One warp per row, 128-bit coalesced row gathers, four
// rows (24 loads per lane) in flight at a time so the gather is bandwidth- not latency-bound.
template <int TMR>
__device__ __forceinline__ void build_h1(float* H1, int* srcv, const float* __restrict__ A, const float* __restrict__ S,
                                         const float* __restrict__ R, const int32_t* __restrict__ in_snd,
                                         const int32_t* __restrict__ in_rcv, int e0, int rows) {
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  constexpr int C4 = kDEP / 4;        // 38 float4 per row
  constexpr int RPW = TMR / 8;        // rows per warp
  const int r0 = warp * RPW;
  int my_s = -1, my_r = -1;
  if (lane < RPW && r0 + lane < rows) { my_s = in_snd[e0 + r0 + lane]; my_r = in_rcv[e0 + r0 + lane]; }
  if (lane < RPW) srcv[r0 + lane] = my_r;
  const float4 z4 = make_float4(0.f, 0.f, 0.f, 0.f);
  for (int rb = 0; rb < RPW; rb += 4) {
    float4 va[4][2], vs[4][2], vr[4][2];
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int s = __shfl_sync(0xffffffffu, my_s, rb + j), rc = __shfl_sync(0xffffffffu, my_r, rb + j);
      const size_t e = (size_t)(e0 + r0 + rb + j);
#pragma unroll
      for (int p = 0; p < 2; ++p) {
        const int c = lane + 32 * p;
        if (rc >= 0 && c < C4) {
          va[j][p] = reinterpret_cast<const float4*>(A + e * kDEP)[c];
          vs[j][p] = reinterpret_cast<const float4*>(S + (size_t)s * kDEP)[c];
          vr[j][p] = reinterpret_cast<const float4*>(R + (size_t)rc * kDEP)[c];
        } else {
          va[j][p] = z4; vs[j][p] = z4; vr[j][p] = z4;
        }
      }
    }
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int rc = __shfl_sync(0xffffffffu, my_r, rb + j);
      float4* dst = reinterpret_cast<float4*>(H1 + (size_t)(r0 + rb + j) * kDEP);
#pragma unroll
      for (int p = 0; p < 2; ++p) {
        const int c = lane + 32 * p;
        if (c >= C4) continue;
        float4 h;
        h.x = relu_f(va[j][p].x + vs[j][p].x + vr[j][p].x); h.y = relu_f(va[j][p].y + vs[j][p].y + vr[j][p].y);
        h.z = relu_f(va[j][p].z + vs[j][p].z + vr[j][p].z); h.w = relu_f(va[j][p].w + vs[j][p].w + vr[j][p].w);
        if (c == C4 - 1) { h.z = rc >= 0 ? 1.f : 0.f; h.w = 0.f; }   // columns 150 (bias ones) and 151 (pad)
        dst[c] = h;
      }
    }
  }
}

struct EdgeStepArgs {
  int E;
  const int32_t* in_snd; const int32_t* in_rcv; const int32_t* in_off;
  const float* A; const float* S; const float* R;     // [E][152], [n][152], [n][152]
  const float* W2; const float* b2;                   // packed rmp.w1, raw rmp.b1
  float* H2S;                                         // [n][152] sum over in-edges of h2
  float* part_first; float* part_last;                // [ntiles][152] segments cut by a tile boundary
  uint32_t* maskbits;                                 // [E][8] relu mask of h2 (training) or null:
                                                      //   bit (col & 31) of word (col >> 5), 5 words used
};

// K2b: per step -- gather, hidden layer 2, relu, deterministic receiver-segmented sum
__global__ void __launch_bounds__(kThreads, 2) k_edge_step(EdgeStepArgs a) {
  SPW_DYN_SMEM(smem_raw);
  constexpr int ROWS = kTME / 8;
  float* Xa = reinterpret_cast<float*>(smem_raw);
  float* Xb = Xa + kTME * kDEP + 8;
  float* Wst = Xb + kTME * kDEP + 8;
  int* srcv = reinterpret_cast<int*>(Wst + 2 * kKT * kLdwE);
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int ntiles = (a.E + kTME - 1) / kTME;
  for (int tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
    const int e0 = tile * kTME;
    const int rows = imin(kTME, a.E - e0);
    build_h1<kTME>(Xa, srcv, a.A, a.S, a.R, a.in_snd, a.in_rcv, e0, rows);
    __syncthreads();
    float acc[ROWS][5];
    zero_acc<ROWS, 5>(acc);
    gemm_tile_acc<ROWS, 5>(acc, Xa, kDEP, warp * ROWS, a.W2, kDEP, Wst);
    store_act_tile<ROWS>(acc, Xb, warp, lane, rows, [&](float v, int, int c) { return relu_f(v + a.b2[c]); });
    __syncthreads();
    if (a.maskbits) {   // relu bits of h2 for the backward pass (h2 > 0 <=> pre-activation > 0)
      for (int idx = tid; idx < rows * 5; idx += kThreads) {
        const int r = idx / 5, w = idx - r * 5;
        uint32_t m = 0u;
        for (int b = 0; b < 32; ++b) {
          const int col = 32 * w + b;
          if (col < kDE && Xb[(size_t)r * kDEP + col] > 0.f) m |= 1u << b;
        }
        a.maskbits[(size_t)(e0 + r) * 8 + w] = m;
      }
    }
    // receiver-segmented sum in row (= ascending sender = slot) order; one warp per node
    const int n_first = srcv[0], n_last = srcv[rows - 1];
    for (int node = n_first + warp; node <= n_last; node += kThreads / 32) {
      const int s0 = a.in_off[node], s1 = a.in_off[node + 1];
      const int lo = imax(s0, e0) - e0, hi = imin(s1, e0 + rows) - e0;
      if (hi <= lo) continue;
      float* dst;
      if (s0 >= e0 && s1 <= e0 + rows) dst = a.H2S + (size_t)node * kDEP;
      else if (s0 < e0) dst = a.part_first + (size_t)tile * kDEP;
      else dst = a.part_last + (size_t)tile * kDEP;
      for (int c = lane; c < kDEP; c += 32) {
        float s = 0.f;
        if (c < kDE)
          for (int r = lo; r < hi; ++r) s += Xb[(size_t)r * kDEP + c];
        dst[c] = s;
      }
    }
    __syncthreads();
  }
}

// segments cut by a tile boundary: H2S[node] = last-part of tile b + first-part of tile b+1
__global__ void __launch_bounds__(256) k_fix_boundaries(int E, int tile_rows, const int32_t* __restrict__ in_rcv,
                                                        const float* __restrict__ part_first,
                                                        const float* __restrict__ part_last, float* __restrict__ H2S) {
  const int lane = threadIdx.x & 31, wpb = blockDim.x >> 5;
  const int ntiles = (E + tile_rows - 1) / tile_rows;
  for (int b = blockIdx.x * wpb + (threadIdx.x >> 5); b + 1 < ntiles; b += gridDim.x * wpb) {
    const int e = (b + 1) * tile_rows;
    const int node = in_rcv[e - 1];
    if (in_rcv[e] != node) continue;
    for (int c = lane; c < kDEP; c += 32)
      H2S[(size_t)node * kDEP + c] = part_last[(size_t)b * kDEP + c] + part_first[(size_t)(b + 1) * kDEP + c];
  }
}

struct EdgeStepBwdArgs {
  int E;
  const int32_t* in_snd; const int32_t* in_rcv;
  const float* A; const float* S; const float* R;
  const float* W2T;
  const uint32_t* maskbits; // [E][8] relu mask of h2 written by k_edge_step in the forward pass
  const float* dH2S;        // [n][152]
  float* dA;                // [E][152] accumulated over the 5 steps
  float* DH1;               // [E][152] d(pre-activation of h1) of this step
  float* partW2;            // [gridDim.x][160*160]
  int first;                // first step processed (l = 5): dA is written, not accumulated
};

// K4b: per step backward of K2b -- rebuild h1 (gather), d h2 from the saved relu bits, dW2 partials,
// and (DGRAD) d(h1 pre-activation) = (d h2 . W2^T) * relu'(h1).  The GPU build runs the data gradient on the
// tensor cores (tc::k_edge_dgrad_tc) and instantiates DGRAD = false here.
template <bool DGRAD>
__global__ void __launch_bounds__(kThreads, 1) k_edge_step_bwd(EdgeStepBwdArgs a) {
  SPW_DYN_SMEM(smem_raw);
  float* Xa = reinterpret_cast<float*>(smem_raw);
  float* Xb = Xa + kTM * kDEP + 8;
  float* Wst = Xb + kTM * kDEP + 8;
  int* srcv = reinterpret_cast<int*>(Wst + 2 * kKT * kLdwE);
  uint32_t* smask = reinterpret_cast<uint32_t*>(srcv + kTM);
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int ntiles = (a.E + kTM - 1) / kTM;
  float* part = a.partW2 + (size_t)blockIdx.x * (160 * 160);
  constexpr int C4 = kDEP / 4;
  for (int tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
    const int e0 = tile * kTM;
    const int rows = imin(kTM, a.E - e0);
    build_h1<kTM>(Xa, srcv, a.A, a.S, a.R, a.in_snd, a.in_rcv, e0, rows);
    for (int idx = tid; idx < kTM * 5; idx += kThreads) {
      const int r = idx / 5, i = idx - r * 5;
      smask[idx] = r < rows ? a.maskbits[(size_t)(e0 + r) * 8 + i] : 0u;
    }
    __syncthreads();
    // dH2pre[row][col] = mask ? dH2S[receiver][col] : 0   (a dY operand: no ones column)
    for (int rb = warp * 16; rb < warp * 16 + 16; rb += 4) {
      float4 d[4][2];
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const int rc = srcv[rb + j];
#pragma unroll
        for (int p = 0; p < 2; ++p) {
          const int c = lane + 32 * p;
          d[j][p] = (rc >= 0 && c < C4) ? reinterpret_cast<const float4*>(a.dH2S + (size_t)rc * kDEP)[c]
                                        : make_float4(0.f, 0.f, 0.f, 0.f);
        }
      }
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const uint32_t* mw = smask + (rb + j) * 5;
#pragma unroll
        for (int p = 0; p < 2; ++p) {
          const int c = lane + 32 * p;
          if (c >= C4) continue;
          const int col = 4 * c;
          float4 v = d[j][p];
          const uint32_t bits = mw[col >> 5] >> (col & 31);     // 4 consecutive columns never straddle a word
          v.x = (col < kDE && (bits & 1u)) ? v.x : 0.f;
          v.y = (col + 1 < kDE && (bits & 2u)) ? v.y : 0.f;
          v.z = (col + 2 < kDE && (bits & 4u)) ? v.z : 0.f;
          v.w = (col + 3 < kDE && (bits & 8u)) ? v.w : 0.f;
          reinterpret_cast<float4*>(Xb + (size_t)(rb + j) * kDEP)[c] = v;
        }
      }
    }
    __syncthreads();
    {
      float wacc[10][10];
#pragma unroll
      for (int i = 0; i < 10; ++i)
#pragma unroll
        for (int j = 0; j < 10; ++j) wacc[i][j] = 0.f;
      wgrad_tile_acc<10, 10>(wacc, Xa, kDEP, Xb, kDEP, kTM);
      if (a.first && tile == (int)blockIdx.x) wgrad_flush<10, 10, false>(wacc, part);
      else wgrad_flush<10, 10, true>(wacc, part);
    }
    if (!DGRAD) { __syncthreads(); continue; }
    float acc[16][5];
    zero_acc<16, 5>(acc);
    gemm_tile_acc<16, 5>(acc, Xb, kDEP, warp * 16, a.W2T, kDEP, Wst);
    // masked result -> Xb (free after the GEMM), then 128-bit coalesced rows to HBM
#pragma unroll
    for (int r = 0; r < 16; ++r) {
      const int row = warp * 16 + r;
#pragma unroll
      for (int i = 0; i < 5; ++i) {
        const int col = lane * 5 + i;
        if (col < kDEP) Xb[(size_t)row * kDEP + col] = (col < kDE && Xa[(size_t)row * kDEP + col] > 0.f) ? acc[r][i] : 0.f;
      }
    }
    __syncthreads();
    for (int idx = tid; idx < rows * C4; idx += kThreads) {
      const float4 v = reinterpret_cast<const float4*>(Xb)[idx];
      const size_t g = (size_t)e0 * C4 + idx;
      reinterpret_cast<float4*>(a.DH1)[g] = v;
      if (a.first) {
        reinterpret_cast<float4*>(a.dA)[g] = v;
      } else {
        float4 o = reinterpret_cast<const float4*>(a.dA)[g];
        o.x += v.x; o.y += v.y; o.z += v.z; o.w += v.w;
        reinterpret_cast<float4*>(a.dA)[g] = o;
      }
    }
    __syncthreads();
  }
}

// dS_i = sum over out-edges, dR_i = sum over in-edges of DH1 (fixed order); one warp per node
__global__ void __launch_bounds__(256) k_gather_dsr(int n, const int32_t* __restrict__ in_off,
                                                    const int32_t* __restrict__ out_off,
                                                    const int32_t* __restrict__ out_pos, const float* __restrict__ DH1,
                                                    float* __restrict__ dS, float* __restrict__ dR) {
  const int lane = threadIdx.x & 31, wpb = blockDim.x >> 5;
  constexpr int C4 = kDEP / 4;
  for (int i = blockIdx.x * wpb + (threadIdx.x >> 5); i < n; i += gridDim.x * wpb) {
    const int i0 = in_off[i], i1 = in_off[i + 1], o0 = out_off[i], o1 = out_off[i + 1];
    for (int c = lane; c < C4; c += 32) {
      float4 s = make_float4(0.f, 0.f, 0.f, 0.f);
      for (int e = i0; e < i1; ++e) {
        const float4 v = reinterpret_cast<const float4*>(DH1 + (size_t)e * kDEP)[c];
        s.x += v.x; s.y += v.y; s.z += v.z; s.w += v.w;
      }
      reinterpret_cast<float4*>(dR + (size_t)i * kDEP)[c] = s;
      s = make_float4(0.f, 0.f, 0.f, 0.f);
      for (int e = o0; e < o1; ++e) {
        const float4 v = reinterpret_cast<const float4*>(DH1 + (size_t)out_pos[e] * kDEP)[c];
        s.x += v.x; s.y += v.y; s.z += v.z; s.w += v.w;
      }
      reinterpret_cast<float4*>(dS + (size_t)i * kDEP)[c] = s;
    }
  }
}

struct EdgeEncBwdArgs {
  int E;
  const int32_t* in_snd; const int32_t* in_rcv;
  const float* obj;
  const float* W0; const float* b0;
  const float* RM1; const float* RM2; const float* RM3;
  const float* b1; const float* b2; const float* b3;
  const float* RM1T; const float* RM2T; const float* RM3T; const float* W1AT;
  const float* dA;          // [E][152] total gradient w.r.t. A_e
  const float* X1; const float* X2; const float* C;   // [E][152] activations saved by k_edge_encode
  float inv_keep;           // 1/(1-rate) of the dropout applied to c_e in the forward pass (1 if none)
  float* partM;             // [gridDim.x][4][160*160]: W1A, RM3, RM2, RM1
  float* part0;             // [gridDim.x][3][152]: d rm.w0 row 0, row 1, d rm.b0
  float* G0;                // [E][152] or null: the gradient w.r.t. the pre-activation of rm layer 0 (columns 0..149; spw_backward_obj)
};

constexpr int kTMB = 64;    // rows per tile in the encoder backward (5 resident activation tiles)

// K4a: backward of K2a -- recompute the 4 encoder layers per 64-edge tile, then walk back
__global__ void __launch_bounds__(kThreads, 1) k_edge_encode_bwd(EdgeEncBwdArgs a) {
  SPW_DYN_SMEM(smem_raw);
  constexpr int TILE = kTMB * kDEP + 8;
  float* Ba = reinterpret_cast<float*>(smem_raw);
  float* Bb = Ba + TILE;
  float* Bc = Bb + TILE;
  float* Bd = Bc + TILE;
  float* Be = Bd + TILE;
  float* Wst = Be + TILE;
  float* sdx = Wst + 2 * kKT * kLdwE;
  float* sdy = sdx + kTMB;
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int ntiles = (a.E + kTMB - 1) / kTMB;
  float* partM = a.partM + (size_t)blockIdx.x * (4 * 160 * 160);
  float* part0 = a.part0 + (size_t)blockIdx.x * (3 * kDEP);
  bool first = true;
  for (int tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
    const int e0 = tile * kTMB;
    const int rows = imin(kTMB, a.E - e0);
    // ---- layer inputs: X0 (Ba) is rebuilt (K = 2); X1 (Bb), X2 (Bc), C (Bd) come back from the forward
    //      pass (saved with their bias "ones" column); dA tile -> Be (a dY operand: no ones column)
    build_x0<kTMB>(Ba, sdx, sdy, a.obj, a.in_snd, a.in_rcv, e0, rows, a.W0, a.b0);
    tile_from_global(Bb, a.X1, e0, rows, kTMB);
    tile_from_global(Bc, a.X2, e0, rows, kTMB);
    tile_from_global(Bd, a.C, e0, rows, kTMB);
    tile_from_global(Be, a.dA, e0, rows, kTMB);
    __syncthreads();
    float acc[8][5];
    // ---- backward.  Each stage: dW += X^T.dY (bias via the ones column), dX = (dY.W^T) * relu'
    auto stage = [&](const float* X, float* dY, const float* WT, float* dXout, float* part, float scale) {
      float wacc[10][10];
#pragma unroll
      for (int i = 0; i < 10; ++i)
#pragma unroll
        for (int j = 0; j < 10; ++j) wacc[i][j] = 0.f;
      wgrad_tile_acc<10, 10>(wacc, X, kDEP, dY, kDEP, kTMB);
      if (first) wgrad_flush<10, 10, false>(wacc, part); else wgrad_flush<10, 10, true>(wacc, part);
      zero_acc<8, 5>(acc);
      gemm_tile_acc<8, 5>(acc, dY, kDEP, warp * 8, WT, kDEP, Wst);
      // mask with the layer input's relu (X holds post-relu values; X > 0 <=> pre-activation > 0)
#pragma unroll
      for (int r = 0; r < 8; ++r) {
        const int row = warp * 8 + r;
#pragma unroll
        for (int i = 0; i < 5; ++i) {
          const int col = lane * 5 + i;
          if (col >= kDEP) continue;
          float v = 0.f;
          if (row < rows && col < kDE && X[(size_t)row * kDEP + col] > 0.f) v = acc[r][i] * scale;
          dXout[(size_t)row * kDEP + col] = v;
        }
      }
      __syncthreads();
    };
    stage(Bd, Be, a.W1AT, Be, partM, a.inv_keep);                    // A = C.W1a + b   : dC  -> Be (in place)
    stage(Bc, Be, a.RM3T, Bd, partM + 1 * 160 * 160, 1.f);    // C = relu(X2.W3) : dX2 -> Bd
    stage(Bb, Bd, a.RM2T, Be, partM + 2 * 160 * 160, 1.f);    // X2              : dX1 -> Be
    stage(Ba, Be, a.RM1T, Bd, partM + 3 * 160 * 160, 1.f);    // X1              : dX0 -> Bd
    // layer 0 (K = 2): d rm.w0[0][k] = sum_r dx_r dX0[r][k], [1][k] with dy, d rm.b0[k] = sum_r dX0[r][k]
    for (int k = tid; k < kDE; k += kThreads) {
      float g0 = 0.f, g1 = 0.f, gb = 0.f;
      for (int r = 0; r < rows; ++r) {
        const float d = Bd[(size_t)r * kDEP + k];
        g0 = fmaf(sdx[r], d, g0); g1 = fmaf(sdy[r], d, g1); gb += d;
      }
      if (first) { part0[k] = g0; part0[kDEP + k] = g1; part0[2 * kDEP + k] = gb; }
      else { part0[k] += g0; part0[kDEP + k] += g1; part0[2 * kDEP + k] += gb; }
    }
    if (a.G0)
      for (int idx = tid; idx < rows * kDE; idx += kThreads) {
        const int r = idx / kDE, k = idx - r * kDE;
        a.G0[(size_t)(e0 + r) * kDEP + k] = Bd[(size_t)r * kDEP + k];
      }
    first = false;
    __syncthreads();
  }
}

}  // namespace spw
