/* spwgnn.h -- C ABI of libspwgnn.so: the B200 (sm_100a) hot path of SPWGNN's tower-stability
 * propagation network.  Plain pointers and sizes only; no torch / C++ types cross this boundary.
 *
 * What each entry point replaces in the reference (paths under /root/reference/src):
 *   spw_edges_*        the relation-matrix loops            main.py:66-81, TowerCreator.py:415-428,
 *                                                           JengaBuilder.py:313-326
 *   spw_forward        the Keras graph behind .predict/.fit Networks.py:22-99 (+ Blocks.py:12-91)
 *   spw_bce_grad       loss + its gradient seed             Networks.py:102 (binary_crossentropy)
 *   spw_backward       TF autodiff of that graph            Networks.py:101-102 (compile/fit)
 * The reference has no FFI of its own (pure Python on Keras); INTEGRATION.md shows the ctypes
 * binding a maintainer would add to Networks.py.
 *
 * Conventions
 *   - every pointer is a DEVICE pointer unless the name ends in _host; the caller owns all memory;
 *     the library allocates nothing persistent and never synchronises the device.
 *   - every call enqueues kernels on `stream` (a cudaStream_t passed as void*) and returns.
 *   - return value: 0 = ok, negative = SpwStatus; spw_last_error() gives a thread-local message.
 *   - towers are ragged: tower t owns nodes [node_off[t], node_off[t+1]); 2 <= N_t <= SPW_MAX_NODES
 *     is not required (N_t may be 0 or 1: such towers simply have no edges), N_t <= SPW_MAX_NODES is.
 *   - float tensors are fp32, row-major; all pointers must be 16-byte aligned.
 */
#ifndef SPWGNN_H
#define SPWGNN_H
#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define SPW_VERSION 1
#define SPW_MAX_NODES 64      /* blocks per tower handled by the edge builder's per-tower CTA */
#define SPW_N_STEPS 5         /* Networks.py:83 */
#define SPW_PROP_DIM 100      /* Networks.py:29 */
#define SPW_SMALL_MAX_NODES 32  /* blocks per tower of the one-CTA-per-tower inference (spw_forward_towers) */

typedef enum {
  SPW_OK = 0,
  SPW_ERR_BAD_ARG = -1,       /* null / misaligned pointer, negative size */
  SPW_ERR_UNSUPPORTED = -2,   /* shape outside the limits above */
  SPW_ERR_WORKSPACE = -3,     /* workspace too small */
  SPW_ERR_LAUNCH = -4         /* CUDA launch failure (message carries cudaGetErrorString) */
} SpwStatus;

/* The 22 parameter tensors, Keras Dense layout kernel[in][out], bias[out] (Blocks.py:22-27):
 *   rm  2->150->150->150->150   om 2->100->100   rmp 350->150->150->100   omp 300->100->101
 * Used const for weights, mutable for gradients (same struct, same shapes). */
typedef struct {
  float* rm_w[4];  float* rm_b[4];
  float* om_w[2];  float* om_b[2];
  float* rmp_w[3]; float* rmp_b[3];
  float* omp_w[2]; float* omp_b[2];
} SpwParams;

/* A packed batch of tower graphs.  Built by spw_edges_count + spw_edges_fill. */
typedef struct {
  int32_t n_towers;
  int32_t n_nodes;            /* sum of N_t */
  int32_t n_edges;            /* active edges (host copy of edge_off[n_towers]) */
  const int32_t* node_off;    /* [n_towers+1] */
  const int32_t* in_off;      /* [n_nodes+1]  receiver-major CSR: in-edges of node i are [in_off[i], in_off[i+1]) */
  const int32_t* in_snd;      /* [n_edges]    sender node (global id) of receiver-major edge */
  const int32_t* in_rcv;      /* [n_edges]    receiver node of receiver-major edge */
  const int32_t* out_off;     /* [n_nodes+1]  slot-order (sender-major) CSR: out-edges of node i */
  const int32_t* out_pos;     /* [n_edges]    receiver-major position of slot-order edge e */
} SpwGraph;

int spw_version(void);
const char* spw_last_error(void);

/* ---- measurement hooks (bench.py) --------------------------------------------------------
 * spw_launch_count: kernels launched by this library since it was loaded.
 * spw_profile(1/0): bracket every kernel launch with CUDA events on its stream.
 * spw_profile_report: synchronise those events and write "name launches total_ms" lines.
 * spw_ffma_peak: FP32-pipe micro-benchmark, 2*16*iters flops per thread, grid x 256 threads. */
long long spw_launch_count(void);
int spw_profile(int enable);
int spw_profile_report(char* buf, size_t cap);
int spw_ffma_peak(float* out, int grid, int iters, void* stream);
/* tcgen05 / TMEM self test (3xTF32): D[128][160] = A[128][152] . W[K][N] (K<=152, N<=160); scratch: 48640 floats;
 * status (device int): 1 = ok, -1 = the MMA completion barrier timed out. */
int spw_tc_selftest(const float* A, const float* W, int K, int N, float* D, float* scratch, int* status, void* stream);
/* CTA-pair (tcgen05 cta_group::2) self test: one cluster of two CTAs, each with half of the weight operand in its shared
 * memory and its own 128 rows in tensor memory: D[256][160] = A[256][152] . W[K][N] (K <= 152, N <= 160, 3xTF32);
 * scratch: 4 * 19 * 8 * 80 floats; status[2] (device ints): 1 = ok, -1 = the MMA completion barrier timed out. */
int spw_tc2_selftest(const float* A, const float* W, int K, int N, float* D, float* scratch, int* status, void* stream);
/* generic tensor-core linear layer (the node-level / relation-encoder building block), exposed for unit tests:
 *   Y[M][ldy] = post(act([X0 | X1].W + rowscale*bias + addend)), W in Keras layout [K0 + K1][N] (Blocks.py:22-27);
 *   act 0 none / 1 relu / 2 tanh; mulmode 1: *= [mulsrc > 0], 2: *= (1 - mulsrc^2); NB (MMA N) = 112 or 160, N <= NB,
 *   2*ceil((K0+K1)/8)*8 + NB <= 512; scratch: 2 * ceil((K0 + K1) / 8) * 8 * NB floats; X1 may be null (K1 = 0). */
int spw_tc_linear(int M, const float* X0, int ldx0, int K0, const float* X1, int ldx1, int K1, const float* W, int N, int NB,
                  const float* bias, const float* rowscale, const float* addend, int ld_add, int act, const float* mulsrc,
                  int ld_mul, int mulmode, float* Y, int ldy, int accumulate, float post_scale, int ones_col, float* scratch,
                  void* stream);

/* pipelined column-slab linear layer (the round-2 building block of every GEMM-shaped layer), exposed for unit tests.
 * Activations are stored column-slab major: element (row, c) of a view at p + ((col0 + c) >> 3) * slab + row * 8 + ((col0 + c) & 7)
 * (slab = allocated rows * 8 floats, col0 % 4 == 0).  Y = post(act(X.W + rowscale*bias + addend)); mulmode 3 multiplies by the
 * word-major sign bits bits_in ([8][M][4 bytes]); bits_out receives the sign bits of the result.  scratch: 2*ceil(K/8)*8*NB floats. */
int spw_csl_linear(int M, const float* X, long long x_slab, int x_col0, int K, const float* W, int N, int NB, const float* bias,
                   const float* rowscale, const float* addend, long long add_slab, int add_col0, int act, const float* mulsrc,
                   long long mul_slab, int mul_col0, int mulmode, const uint8_t* bits_in, uint8_t* bits_out, float* Y,
                   long long y_slab, int y_col0, int accumulate, float post_scale, int ones_col, int write_pad, float* scratch,
                   void* stream);

/* ---- edge-index construction (replaces main.py:66-81) ------------------------------------
 * Edge m->j (m != j, same tower) is active iff sqrt(dx*dx + dy*dy) < thr evaluated in IEEE
 * double with separately rounded multiplies/add/sqrt -- numpy's np.linalg.norm(...,axis=1) --
 * or unconditionally when fully_connected != 0.  Slot order: sender m outer, receiver j inner,
 * slot = m*(N-1) + (j < m ? j : j-1)  (main.py:69-81).
 *
 * spw_edges_count: per-node degrees and the per-tower edge prefix sum.
 *   deg_out/deg_in [n_nodes], edge_off [n_towers+1] (edge_off[n_towers] = total active edges).
 *   max_nodes_per_tower: the caller's max N_t (host value; checked against SPW_MAX_NODES).     */
int spw_edges_count(const double* pos_xy /*[n_nodes][2]*/, const int32_t* node_off, int32_t n_towers,
                    int32_t n_nodes, int32_t max_nodes_per_tower, double thr, int fully_connected,
                    int32_t* deg_out, int32_t* deg_in, int32_t* edge_off, void* stream);

/* spw_edges_fill: the edge list in slot order (snd/rcv/slot, the reference's non-zero columns)
 * plus the receiver-major / sender-major CSR views the kernels consume.  Any of snd/rcv/slot may
 * be NULL.  All outputs sized by edge_off[n_towers] (read it back from spw_edges_count, or size
 * for the worst case sum N_t*(N_t-1)).                                                          */
int spw_edges_fill(const double* pos_xy, const int32_t* node_off, int32_t n_towers, int32_t n_nodes,
                   int32_t max_nodes_per_tower, double thr, int fully_connected, const int32_t* edge_off,
                   int32_t* snd, int32_t* rcv, int32_t* slot,
                   int32_t* in_off, int32_t* in_snd, int32_t* in_rcv,
                   int32_t* out_off, int32_t* out_pos, void* stream);

/* ---- network ---------------------------------------------------------------------------- */
/* ---- device-side synthetic layouts (SURVEY.md section 8f, row N4) ------------------------------------------------
 * Physics-free Jenga layout sampler of JengaBuilder.create_world (JengaBuilder.py:137-192: widths randint(50,300), gaps
 * randint(0,50), first layer spans x in [400,1100]) with a counter-based generator (tower t, draw c -> splitmix64), so
 * that large sweeps are generated where they are consumed.  spwgnn_b200/synth.py:g_jenga_ctr is the bit-identical numpy
 * restatement.
 *   spw_sample_sizes: node_off[t+1] - node_off[t] = n_lo + draw_0(t) % (n_hi - n_lo + 1), prefix-summed in place.
 *   spw_sample_jenga: raw[n][3] = [x, y, width] in pixels (f64), obj[n][3] = raw / 170 (f32, main.py:91),
 *                     pos[n][2] = positions for the relation test (raw, or raw / 170 with inference_glue);
 *                     any of the three outputs may be null. */
int spw_sample_sizes(uint64_t seed, int32_t n_towers, int32_t n_lo, int32_t n_hi, int32_t* node_off, void* stream);
int spw_sample_jenga(uint64_t seed, int32_t n_towers, const int32_t* node_off, double* raw, float* obj, double* pos,
                     int inference_glue, void* stream);
/*   spw_sample_tower: same outputs for TowerCreator layouts (TowerCreator.py:106-187, 265-271): 150 x 80 blocks stacked in
 *                     layers plus one dropped block on top, which is object 0 of its tower (TowerCreator.py:451);
 *                     every tower needs >= 2 blocks (spw_sample_sizes with n_lo >= 2); restated by synth.g_tower_ctr. */
int spw_sample_tower(uint64_t seed, int32_t n_towers, const int32_t* node_off, double* raw, float* obj, double* pos,
                     int inference_glue, void* stream);

/* ---- demolish searches (SURVEY.md section 8f, row N3) -------------------------------------------------------------------
 * The reference scores N candidate removals (JengaBuilder.remove_to_demolish, JengaBuilder.py:236-269) or 100 candidate drop
 * poses (TowerCreator.drop_to_demolish, TowerCreator.py:276-319) with one batch-1 predict call each and takes
 * argmin sum_i p_i.  Here the candidates are built on the device and scored as ONE packed inference batch:
 *   spw_candidates_remove: raw [N][3] (pixels) -> N towers of N - 1 blocks (tower c lacks block c, order kept):
 *                          obj [N (N-1)][3] = raw / 170, pos [N (N-1)][2] = positions for the relation test;
 *   spw_candidates_drop:   raw [N][3], poses [K][2] -> K towers of N + 1 blocks, the dropped block (poses[c], `width`) is
 *                          object 0 of tower c (TowerCreator.py:451);
 *   spw_tower_sums:        sums[t] = sum of probs over the blocks of tower t (double, block order: the callers' Python loop),
 *                          argmin (nullable, device int32) = index of the first minimum (np.argmin). */
int spw_candidates_remove(const double* raw, int32_t n_blocks, float* obj, double* pos, int inference_glue, void* stream);
int spw_candidates_drop(const double* raw, int32_t n_blocks, const double* poses, int32_t n_poses, double width, float* obj, double* pos,
                        int inference_glue, void* stream);
int spw_tower_sums(const float* probs, const int32_t* node_off, int32_t n_towers, double* sums, int32_t* argmin, void* stream);

/* Bytes of workspace spw_forward/spw_backward need.  training != 0 also reserves the node-level
 * state the backward pass reads (5 propagation steps x per-node activations) and per-edge
 * gradient staging.  The same workspace must be passed, untouched, to spw_backward.            */
size_t spw_workspace_bytes(int32_t n_nodes, int32_t n_edges, int training);

/* Where a TRAINING forward pass leaves the relu states the backward pass uses (parity tests read them back to evaluate the
 * fp64 oracle on the same piecewise-linear branch: tests/test_gpu_parity.py::test_gradient_deviation_is_relu_kinks).
 * out[0] = rows of a sign-bit array (byte-slab u8 [20][rows]: bit c & 7 of byte [c >> 3][row], rows in receiver-major edge
 * order); out[1] = bytes from one array of a group to the next; byte offsets into the workspace of: out[2] the 4 encoder
 * arrays (relu of rm layers 0-3, Networks.py:75), out[3] the 5 per-step arrays of rmp layer 0 (h1), out[4] of rmp layer 1
 * (h2, Networks.py:84-87); out[5] = U, float column-slab [25 quads][5 n][4] (omp layer 0 after relu, step l = rows l n ..),
 * out[6] = Q and out[7] = Q1, float column-slab [25][n][4] (om layers 1 and 0 after relu, Networks.py:76).               */
int spw_saved_state_layout(int32_t n_nodes, int32_t n_edges, int64_t* out /*[8]*/);

/* The whole column-slab workspace, exposed for unit tests (tests/test_gpu_stages.py checks every launch of a training step
 * against an fp64 evaluation of that one launch on the arrays it read).  spw_workspace_layout fills out[0 .. count) and
 * returns count (SPW_ERR_BAD_ARG if cap < count): first the byte offset of every named array (0 where the mode does not use
 * the array), then slots, slotsGP (per-step slots of U / S / R / H2S and of [g | p]), bits_rows and bits_floats (rows and
 * floats of one sign-bit array), edge_stride_floats (floats between the per-step h1 arrays), the two partial strides (floats)
 * and the workspace size in bytes.  spw_workspace_layout_names gives the comma-separated names in the same order.        */
const char* spw_workspace_layout_names(void);
int spw_workspace_layout(int32_t n_nodes, int32_t n_edges, int training, int64_t* out, int cap);

/* Forward (Networks.py:58-96).  obj [n_nodes][3] = [x, y, width]/170 (main.py:91).
 * logits [n_nodes] (channel 0 of the last object-propagator output, Networks.py:94);
 * probs  [n_nodes] sigmoid(logits) or NULL.  training: keep state for spw_backward.
 * dropout_rate / dropout_seed: inverted dropout on the relation and object encodings
 * (Networks.py:77-78, rate 0.1 in the reference), applied only when training != 0 and rate > 0;
 * the mask is a stateless hash of (seed, element index), see dropout_hash in spw_common.cuh.    */
int spw_forward(const SpwParams* w, const SpwGraph* g, const float* obj, float* logits, float* probs,
                void* workspace, size_t workspace_bytes, int training, float dropout_rate,
                uint64_t dropout_seed, void* stream);

/* Inference with ONE CTA per tower and ONE kernel launch per call: the function of spw_forward(training = 0), for batches of
 * small towers (a batch-1 predict is about 47 launches through spw_forward).  Plain fp32 FFMA; every sum runs in a fixed
 * order that depends on the tower alone, so a tower's logits are the same bits whatever else is in the batch and wherever
 * it sits in it (spw_forward's tiled receiver sums cannot promise that).  Weights are read in the Keras layout of SpwParams.
 *   max_nodes_per_tower: the caller's max N_t (host value, <= SPW_SMALL_MAX_NODES, else SPW_ERR_UNSUPPORTED); it sizes the
 *                        shared memory.  A tower with more blocks than that gets NaN logits (and probs) and nothing else
 *                        of it is written.  Any number of edges per tower (in-degree <= N_t - 1).
 *   obj [n_nodes][3], logits [n_nodes], probs [n_nodes] or NULL: as spw_forward.
 *   workspace: at least spw_forward_towers_bytes(n_nodes, n_edges) bytes (the per-edge A_e = c_e.W1a + b1, 152 floats per
 *              edge), 16-byte aligned; it may be NULL when that size is 0.  Nothing in it is kept after the call.
 * n_nodes == 0 launches nothing. */
size_t spw_forward_towers_bytes(int32_t n_nodes, int32_t n_edges);
int spw_forward_towers(const SpwParams* w, const SpwGraph* g, int32_t max_nodes_per_tower, const float* obj, float* logits,
                       float* probs, void* workspace, size_t workspace_bytes, void* stream);

/* The backward pass of spw_forward_towers, in ONE launch with one CTA per tower: each tower's logits and the gradients of
 * sum_i (dlogits[i] logit_i + dprobs[i] p_i) with respect to the block features and, optionally, the relation weights,
 * p = sigmoid(logit).  The forward pass is spw_forward_towers' code, so the logits are its bits; every sum runs in a fixed
 * order that depends on the tower alone, so a tower's logits, dobj and drel are the same bits whatever else is in the
 * batch and wherever it sits in it.  Plain fp32 FFMA, no dropout.
 *   max_nodes_per_tower: as spw_forward_towers; a tower with more blocks gets NaN logits, dobj rows and drel of its
 *                        relations, and nothing else of it is written.
 *   dlogits, dprobs [n_nodes]: the seed dlogit_i = dlogits[i] + dprobs[i] p_i (1 - p_i); either may be NULL (read as 0),
 *                              not both.
 *   logits: NULL or [n_nodes], written with spw_forward_towers' values.
 *   dobj [n_nodes][3], 16-byte aligned: as spw_backward_obj.
 *   drel: NULL or [n_edges] in the receiver-major relation order, as spw_backward_rel; may be NULL when n_edges == 0.
 *   workspace: at least spw_backward_towers_bytes(n_nodes, n_edges) bytes, 16-byte aligned.  Nothing in it is kept after
 *              the call.
 * n_nodes == 0 launches nothing. */
size_t spw_backward_towers_bytes(int32_t n_nodes, int32_t n_edges);
int spw_backward_towers(const SpwParams* w, const SpwGraph* g, int32_t max_nodes_per_tower, const float* obj,
                        const float* dlogits, const float* dprobs, float* logits, float* dobj, float* drel,
                        void* workspace, size_t workspace_bytes, void* stream);

/* Keras binary_crossentropy on probabilities clipped to [1e-7, 1-1e-7] (Networks.py:102), mean over
 * `count` outputs (pass the GLOBAL number of blocks when data-parallel).  Writes dlogits [n_nodes]
 * = d(mean loss)/d(logit) and adds the summed loss and the number of correct (p>0.5)==target
 * predictions into stats[0], stats[1] (double[2], must be zeroed by the caller).               */
int spw_bce_grad(const float* logits, const float* target, int32_t n_nodes, double count,
                 float* dlogits, double* stats, void* stream);

/* Backward: gradients of sum_i dlogits[i]*logit[i] w.r.t. all 22 tensors, written (not
 * accumulated) to grads.  Deterministic: fixed tile->CTA assignment, fixed-order reductions.
 * dropout_rate must equal the rate of the matching spw_forward call (the masks are implicit in the saved state). */
int spw_backward(const SpwParams* w, const SpwGraph* g, const float* obj, const float* dlogits,
                 void* workspace, size_t workspace_bytes, const SpwParams* grads, float dropout_rate,
                 void* stream);

/* Gradient of sum_i dlogits[i]*logit[i] with respect to obj [n_nodes][3] ([x, y, width]/170), the relations of g held
 * fixed, written (not accumulated) to dobj [n_nodes][3] (16-byte aligned).  No weight gradient is computed.
 * workspace / dropout_rate: as spw_backward (the workspace of a training spw_forward, passed untouched; the rate of that
 * forward); the forward state in it is left unchanged.  Deterministic: every sum runs in a fixed order that depends on the
 * tower alone.  n_nodes == 0 launches nothing.  SPW_ERR_UNSUPPORTED on the round-1 data path (SPW_CSL=0). */
int spw_backward_obj(const SpwParams* w, const SpwGraph* g, const float* obj, const float* dlogits, void* workspace,
                     size_t workspace_bytes, float dropout_rate, float* dobj, void* stream);

/* Gradient of sum_i dlogits[i]*logit[i] with respect to the relation weights: relation e = (s -> r) gets a weight w_e that
 * multiplies both of its one-hot entries (sender_relations[s, e] and receiver_relations[r, e] of the reference's dense input),
 * and drel[e] = d/dw_e at w = 1, the relations of g held in place: the sum of the Keras gradients with respect to those two
 * entries.  drel [n_edges] (4-byte aligned) is written, not accumulated; drel[k] belongs to the receiver-major relation
 * in_snd[k] -> in_rcv[k].  The relation o of the sender-major (slot) order, the order of the reference's relation columns
 * within a tower, is drel[out_pos[o]].  dobj: NULL, or [n_nodes][3] (16-byte aligned) receiving spw_backward_obj's result
 * bit for bit from the same pass.  No weight gradient is computed.  workspace / dropout_rate: as spw_backward_obj; the
 * forward state in it is left unchanged.  Deterministic: every sum runs in a fixed order that depends on the tower alone.
 * n_nodes == 0 launches nothing, and n_edges == 0 launches nothing for drel (drel may then be NULL).  SPW_ERR_UNSUPPORTED
 * on the round-1 data path (SPW_CSL=0). */
int spw_backward_rel(const SpwParams* w, const SpwGraph* g, const float* obj, const float* dlogits, void* workspace,
                     size_t workspace_bytes, float dropout_rate, float* drel, float* dobj, void* stream);

/* Gradient of sum_i dlogits[i]*logit[i] with respect to every input of the reference's model (Networks.py:22-99), from one
 * backward pass without weight gradients: the dense relation tensors sender_relations / receiver_relations (B, N, R) and the
 * propagation input (B, N, 100), at the relations of g and propagation = 0, and the objects.
 *   drs, drr [n_edges][max_nodes_per_tower] (4-byte aligned): row k belongs to the receiver-major relation in_snd[k] -> in_rcv[k]
 *     (its reference slot: see spw_backward_rel), column j to local block j of its tower: d/dsender_relations[j, slot] and
 *     d/dreceiver_relations[j, slot].  Entries j >= N_t are written as 0.
 *   drr_free [n_nodes] (4-byte aligned): d/dreceiver_relations[j, slot] of block j at every inactive (all-zero) slot of its tower,
 *     the same value for all of them (the column's message, that of a zero input, would be delivered to j); d/dsender_relations
 *     is 0 there.  The message is taken without dropout.
 *   dprop [n_nodes][100] (16-byte aligned): d/dpropagation.
 *   dobj: NULL, or [n_nodes][3] (16-byte aligned) receiving spw_backward_obj's result bit for bit.
 * max_nodes_per_tower: the largest N_t of g (<= SPW_MAX_NODES); a larger tower gets NaN in its rows of drs, drr and drr_free.
 * workspace / dropout_rate: as spw_backward_obj; the forward state in it is left unchanged.  scratch: at least
 * spw_backward_inputs_bytes(n_nodes, n_edges) bytes, 16-byte aligned.  All outputs are written, not accumulated.
 * Deterministic: every sum runs in a fixed order that depends on the tower alone.  n_nodes == 0 launches nothing; with
 * n_edges == 0, drs and drr may be NULL.  SPW_ERR_UNSUPPORTED on the round-1 data path (SPW_CSL=0). */
size_t spw_backward_inputs_bytes(int32_t n_nodes, int32_t n_edges);
int spw_backward_inputs(const SpwParams* w, const SpwGraph* g, int32_t max_nodes_per_tower, const float* obj, const float* dlogits,
                        void* workspace, size_t workspace_bytes, float dropout_rate, void* scratch, size_t scratch_bytes,
                        float* drs, float* drr, float* drr_free, float* dprop, float* dobj, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* SPWGNN_H */
