/*
 * stmgcn_b200.h -- C ABI of libstmgcn_b200.so: the B200 (sm_100a) ST-MGCN hot path.
 *
 * The reference (underdoc-wang/ST-MGCN) has NO plugin / FFI / operator interface: its boundary is the
 * Python nn.Module surface (GCN.py:7-46, STMGCN.py:7-119).  This header is therefore the boundary a
 * binding for that surface calls into; each entry point names the reference lines whose arithmetic it
 * replaces.  The Python mirror of the reference modules (repo-root GCN.py / STMGCN.py) binds these with
 * ctypes (st-mgcn_b200/stmgcn_b200/_lib.py); INTEGRATION.md shows the stub.
 *
 * Conventions (SURVEY.md section 8(b)):
 *   - plain C types only: device pointers as void* / const float*, sizes as int64_t, flags as int32_t,
 *     the CUDA stream as void* (a cudaStream_t; NULL = legacy default stream).
 *   - every entry returns int32_t: 0 ok, >0 a cudaError_t, <0 an argument / shape / alignment error.
 *     stmgcn_last_error() returns a thread-local message for the last non-zero return.
 *   - the library never allocates per call and never frees caller memory; all tensors and workspaces are
 *     caller-owned device buffers.  Only graph handles own device memory (immutable after creation).
 *   - entries enqueue on the given stream and return; no device synchronisation inside (graph creation
 *     excepted: it must read back the non-zero count).
 *   - all feature tensors are fp32, "node-major": rows r = n * B + b (region n outer, window b inner),
 *     features contiguous.  (N, B, p) row-major == (N, B*p) row-major == (N*B, p) row-major.
 */
#ifndef STMGCN_B200_H_
#define STMGCN_B200_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define STMGCN_ABI_VERSION 5

/* error codes < 0 */
#define STMGCN_ERR_ARG      (-1)   /* null pointer / bad enum */
#define STMGCN_ERR_SHAPE    (-2)   /* size out of the supported range */
#define STMGCN_ERR_ALIGN    (-3)   /* pointer or leading dimension not aligned as required */
#define STMGCN_ERR_STATE    (-4)   /* handle does not carry what the call needs (e.g. no transpose) */

/* activation of the projection epilogue (GCN.py:42; the reference passes nn.ReLU or None) */
#define STMGCN_ACT_NONE 0
#define STMGCN_ACT_RELU 1

typedef struct stmgcn_graph stmgcn_graph_t;    /* opaque: CSR (+ CSR of the transpose) on one device */

int32_t     stmgcn_abi_version(void);
const char* stmgcn_last_error(void);
/* number of SMs of the current device (grid sizing is done inside; exposed for bench.py's records) */
int32_t     stmgcn_sm_count(void);
/* how many kernels this library has launched in this process (bench.py "gpu_launches") */
int64_t     stmgcn_launch_count(void);

/* ---- graph handles: the constant operand GCN.forward receives as A[k] (GCN.py:24-36) ------------- */
/* From one dense N x N support (row-major, leading dimension ld floats) already on the device: exact
 * zeros are dropped, everything else kept verbatim (so supports[1] of Adj_Preprocessor.process,
 * GCN.py:57-97, becomes the sparse rescaled Laplacian).  build_transpose != 0 also builds CSR of A^T
 * (needed by the backward, SURVEY.md section 8(a)). */
int32_t stmgcn_graph_from_dense(stmgcn_graph_t** out, const float* dense, int64_t n, int64_t ld,
                                int32_t build_transpose, void* stream);
/* From device CSR arrays (copied into the handle). rowptr has n+1 int32 entries. */
int32_t stmgcn_graph_from_csr(stmgcn_graph_t** out, int64_t n, int64_t nnz, const int32_t* rowptr,
                              const int32_t* colidx, const float* vals, int32_t build_transpose,
                              void* stream);
int32_t stmgcn_graph_destroy(stmgcn_graph_t* g);
int64_t stmgcn_graph_n(const stmgcn_graph_t* g);
int64_t stmgcn_graph_nnz(const stmgcn_graph_t* g);
/* copy the CSR (transpose != 0: of A^T) out to caller device buffers (tests / introspection) */
int32_t stmgcn_graph_export(const stmgcn_graph_t* g, int32_t transpose, int32_t* rowptr, int32_t* colidx,
                            float* vals, void* stream);

/* ---- K1: one Chebyshev recurrence step on the features --------------------------------------------
 * Y = alpha * op(A) X + beta * Z + gamma * U,   op(A) = A or A^T,  X/Z/U/Y: (N, f_total) fp32 row-major.
 * Z and U may be NULL (their terms vanish).  Forward step k (replaces the dense einsum GCN.py:35 and the
 * matrix recurrence GCN.py:134): alpha=2 (1 for k=1), beta=-1, Z=T_{k-2}X.  Backward (adjoint Clenshaw):
 * transpose=1, U = U_k.  Y must not alias X. */
int32_t stmgcn_cheb_spmm_step(const stmgcn_graph_t* g, int32_t transpose, float alpha, const float* x,
                              float beta, const float* z, float gamma, const float* u, float* y,
                              int64_t f_total, void* stream);

/* The same step with the GATHERED operand read from a bf16 copy (the bf16-arithmetic mode of the bf16-quoted
 * configurations: the kernel's time is its gather volume): x16 (N, f_total) bf16; z, u, y stay fp32; y16 (nullable) receives
 * the bf16 copy of y for the next step.  f_total must be a multiple of 8.  stmgcn_to_bf16 makes the first copy
 * (count elements, a multiple of 8). */
int32_t stmgcn_cheb_spmm_step16(const stmgcn_graph_t* g, int32_t transpose, float alpha, const void* x16,
                                float beta, const float* z, float gamma, const float* u, float* y, void* y16,
                                int64_t f_total, void* stream);
int32_t stmgcn_to_bf16(const float* x, void* y16, int64_t count, void* stream);

/* ---- layout: obs (B,T,N,C) -> node-major (STMGCN.py:36,39 sum over C + permute; :47 row order) ----
 * xo: (N,B,T,C) copy of obs;  xt: (N,B,T) = sum_c obs.  xo may be NULL when C == 1 (xt is then xo). */
int32_t stmgcn_obs_to_node_major(const float* obs, float* xo, float* xt, int64_t b, int64_t t,
                                 int64_t n, int64_t c, void* stream);

/* ---- K2: stacked-K projection (GCN.py:37-42) --------------------------------------------------------
 * Two kernel families, one set of entries each.  stmgcn_proj_fwd / _bwd run the exact-FFMA CUDA-core kernels for any
 * shape, with pooling; stmgcn_proj_fwd_tc / _bwd_tc run the tcgen05 3xTF32 kernels (every fp32 operand split into tf32
 * hi + lo, three passes) for p = q = 64 and ks <= 8, and reject anything else.
 *
 * out[r,:] = act( sum_k S_k[r,:] W[k*p:(k+1)*p, :] + bias ),  r in [0, rows), S_k = s + k*stride_k
 * (rows x p, row-major), W: (ks*p, q) row-major, bias: q or NULL.
 * Optional gate pooling (STMGCN.py:41-42), requires q == p: pool[(r % b_inner)*q + j] +=
 * S_0[r,j] + out[r,j]  (caller zeroes pool; sum over regions of x_hat, not yet divided by N). */
int32_t stmgcn_proj_fwd(const float* s, int64_t stride_k, int32_t ks, int64_t rows, int32_t p,
                        const float* w, const float* bias, int32_t q, int32_t act, float* out,
                        float* pool, int64_t b_inner, void* stream);
/* backward of the projection.  dZ = dOut (.) [out > 0] (act = RELU) with dOut either a full (rows, q)
 * tensor (d_out) or, when d_out_bcast != NULL, the broadcast dOut[r,:] = d_out_bcast[(r % b_inner), :] *
 * bcast_scale (the mean-pool adjoint dz/N, STMGCN.py:42).  dz_work: (rows, q) workspace receiving dZ.
 * Accumulates (+=) dw (ks*p, q) and dbias (q, may be NULL) -- caller zeroes them -- and, if u != NULL,
 * writes U_k = dZ W_k^T into u + k*stride_u (rows x p); wt is then W^T, (q, ks*p) row-major. */
int32_t stmgcn_proj_bwd(const float* s, int64_t stride_k, int32_t ks, int64_t rows, int32_t p,
                        const float* wt, int32_t q, int32_t act, const float* out, const float* d_out,
                        const float* d_out_bcast, float bcast_scale, int64_t b_inner, float* dz_work,
                        float* dw, float* dbias, float* u, int64_t stride_u, void* stream);
/* Tensor-core operand images of W (ks*64, 64), ks <= 8: img_fwd: ks*64*64*2 floats; img_bwd (may be NULL): one
 * 2*2*256*32-float image per group of 4 supports (two images when ks > 4), ZERO-FILLED by the caller (rows beyond ks*64
 * stay zero). */
int32_t stmgcn_proj_pack_tc(const float* w, int32_t ks, float* img_fwd, float* img_bwd, void* stream);
/* stmgcn_proj_fwd on the tensor cores: p = q = 64, 1 <= ks <= 8, no pooling; wimg = img_fwd of stmgcn_proj_pack_tc.
 * s, wimg and out 16-byte aligned, stride_k a multiple of 4. */
int32_t stmgcn_proj_fwd_tc(const float* s, int64_t stride_k, int32_t ks, int64_t rows, const float* wimg,
                           const float* bias, int32_t act, float* out, void* stream);
/* stmgcn_proj_bwd on the tensor cores: p = q = 64, 1 <= ks <= 8, a full d_out, and U is always produced (u required);
 * wimg_t = img_bwd of stmgcn_proj_pack_tc.  s, wimg_t, out, d_out, dz_work and u 16-byte aligned, stride_k and stride_u
 * multiples of 4. */
int32_t stmgcn_proj_bwd_tc(const float* s, int64_t stride_k, int32_t ks, int64_t rows, const float* wimg_t,
                           int32_t act, const float* out, const float* d_out, float* dz_work, float* dw, float* dbias,
                           float* u, int64_t stride_u, void* stream);

/* ---- K3a: context gate (STMGCN.py:42-43) -----------------------------------------------------------
 * z = pool / n_regions; a1 = z fcw^T + fcb; s = sigmoid(relu(a1) fcw^T + fcb).  All (B, T); fcw (T,T). */
int32_t stmgcn_gate_fwd(const float* pool, int64_t b, int32_t t, int64_t n_regions, const float* fcw,
                        const float* fcb, float* z, float* a1, float* s, void* stream);
/* d_s -> d_fcw (+=), d_fcb (+=), d_z (B,T) */
int32_t stmgcn_gate_bwd(const float* d_s, const float* z, const float* a1, const float* s, int64_t b,
                        int32_t t, const float* fcw, float* d_fcw, float* d_fcb, float* d_z, void* stream);

/* ---- K3b (exact fp32, any H <= 128): shared-weight LSTM, one call per direction (STMGCN.py:44, :47-50) ------------
 * The CUDA-core path for every shape the tensor-core kernels below do not cover (H != 64 or C > 4), and the on-device
 * reference the parity tests compare them with.  Weights are passed packed, H = hid, columns gate-interleaved
 * col = 4*unit + gate (gate order i,f,g,o):
 *   wx     : (C, 4H)      = W_ih_l0^T                      (layer-0 input weights)
 *   wp[l]  : (kd_l, 4H)   = W_hh_0^T (l = 0, kd_0 = H) or [W_ih_l^T ; W_hh_l^T] (l > 0, kd_l = 2H)
 *   bp[l]  : (4H)         = b_ih_l + b_hh_l
 *   wpt[l] : (4H, kd_l)   = wp[l]^T                        (backward data operand)
 * State / tape tensors, rows r = n*B + b, fp32 row-major:
 *   hs, cs: (L, T, R, H);  gates: (L, T, R, 4H) post-activation, gate-interleaved (NULL in inference);
 * xo: (R, T, C) node-major observations, s_gate: (B, T) context gate (the modulation xo * s is fused into the layer-0
 * input read, STMGCN.py:44).  h0/c0: (L, R, H) or NULL (zeros, STMGCN.py:53-57).
 * The forward runs every timestep t = 0 .. T-1, layers 0..L-1 within a step.  Limits: H % 4 == 0, H <= 128, C <= 4,
 * L <= 8. */
int32_t stmgcn_lstm_fwd(int32_t t_len, int32_t n_layers, int64_t rows, int32_t hid, int32_t c_in, int64_t b_inner,
                        const float* xo, const float* s_gate, const float* wx, const float* const* wp,
                        const float* const* bp, const float* h0, const float* c0, float* hs, float* cs, float* gates,
                        void* stream);
/* BPTT through all timesteps t = T-1 .. 0 (layers top-down within a step), then the weight gradients layer by layer.
 * d_top: (R, H) gradient of hs[L-1][T-1].  Workspaces (none needs initialisation; h_n / c_n carry no gradient,
 * STMGCN.py:113): dh_rec, dc: (L, R, H); dx_work: (R, H).
 * gates is overwritten IN PLACE with the pre-activation gradients dA: the tape serves one backward only.
 * Accumulates (+=; caller zeroes): d_s (B,T) = sum_{n,c} dxmod * xo (gate adjoint, STMGCN.py:44), dwx (C,4H),
 * dbp[l] (4H), dwp[l] (kd_l, 4H) = [h_below_t | h_{t-1}]^T dA summed over all (t, r). */
int32_t stmgcn_lstm_bwd(int32_t t_len, int32_t n_layers, int64_t rows, int32_t hid, int32_t c_in, int64_t b_inner,
                        const float* xo, const float* s_gate, const float* wx, const float* const* wpt, const float* h0,
                        const float* c0, const float* hs, const float* cs, float* gates, const float* d_top,
                        float* dh_rec, float* dc, float* dx_work, float* d_s, float* dwx, float* const* dbp,
                        float* const* dwp, void* stream);

/* ---- K3b on the tensor cores (H = 64, C <= 4): bf16-plane LSTM without a gate tape -----------------------------
 * Same arithmetic contract as stmgcn_lstm_fwd / _bwd (STMGCN.py:44, :47-50; nn.LSTM semantics, fp32 state and
 * accumulation), different tape:
 *   hp : (L, T, P, R, 64) bf16 -- every hidden state as P planes; P = 2: hi = bf16(h), lo = bf16(h - hi) (3-pass
 *        "3xBF16" products, ~2^-18 operand error: fp32-grade, the 1e-4 parity bar holds with >10x margin);
 *        P = 1: hi only, single-pass bf16 products (the arithmetic of the bf16-quoted BASELINE configs).
 *   cs : (L, T, R_pad, 64) fp32, R_pad = ceil(R/128)*128, tile-blocked (element (r,u) at
 *        (((r/128)*16 + u/4)*128 + r%128)*4 + u%4).
 * No gate tape: the backward recomputes the gates from hp (which it needs anyway for the weight gradients).
 * stmgcn_lstm16_pack turns one layer's nn.LSTM parameters (native layout: w_ih (256, in), w_hh (256, 64), b_ih, b_hh
 * (256), gate order i,f,g,o) into the resident operand image wimg (layer 0: 64 KB, layers > 0: 128 KB; tiles
 * [(segment, plane)] of [256 gate-interleaved columns][64 k] bf16, 128-byte swizzled), bias (256) = b_ih + b_hh
 * gate-interleaved (col = 4*unit + gate) and, for layer 0, wih_t (C, 256) = W_ih^T gate-interleaved. */
int32_t stmgcn_lstm16_pack(const float* w_ih, const float* w_hh, const float* b_ih, const float* b_hh, int32_t layer,
                           int32_t c_in, void* wimg, float* bias, float* wih_t, void* stream);
/* The forward through all timesteps t = 0 .. T-1, layers 0..L-1 within a step (one launch per layer-step).
 * wimg[l] / bias[l]: layer l's operands from stmgcn_lstm16_pack.  h0p: (L, P, R, 64) bf16 planes of the initial hidden
 * state and c0: (L, R_pad, 64) fp32 tile-blocked, or both NULL (zeros, STMGCN.py:53-57).  At t = T-1 the fp32 hidden
 * state is also written: every layer into h_n (L, R, 64) when h_n != NULL, else only the top layer into h_top (R, 64) --
 * the (N,B,H) operand of the spatial GCN (STMGCN.py:50, :114).  C <= 4, L <= 8. */
int32_t stmgcn_lstm16_fwd(int32_t t_len, int32_t n_layers, int64_t rows, int32_t c_in, int64_t b_inner, int32_t planes,
                          const float* xo, const float* s_gate, const void* const* wimg, const float* const* bias,
                          const float* wih_t, const void* h0p, const float* c0, void* hp, float* cs, float* h_top,
                          float* h_n, void* stream);

/* grid (CTAs) the lstm16 kernels use for `rows` rows: the number of weight-gradient scratch slices per layer */
int32_t stmgcn_lstm16_grid(int64_t rows);
/* BPTT through all timesteps, layers top-down, then one reduction per layer into the nn.LSTM-native gradients.  Per
 * layer the kernel recomputes the gates from hp, forms dA, accumulates the weight and bias gradients and propagates
 * [dx_below | dh_prev].  A tile's rows never mix with other tiles', so each CTA walks its own tiles through time inside
 * a launch; a launch covers as many consecutive timesteps as keep a CTA's weight-gradient accumulation chain within
 * 6144 rows (cfg3: 3 steps, 4 launches per layer).  T <= 64, C <= 4, L <= 8.
 * Inputs: those of stmgcn_lstm16_fwd and its tape hp, cs; d_top (R_pad, 64) tile-blocked, the gradient of the top
 * layer's last hidden state.
 * Workspaces (fp32, tile-blocked where they have R_pad rows):
 *   dh_rec, dc : (R_pad, 64), no initialisation needed;
 *   dx_work    : min(2, L-1) slices of (T, R_pad, 64), no initialisation needed; NULL exactly when L == 1 (the gradient
 *                a layer passes to the layer below, for every step);
 *   dbp        : (L, 256) and d_s (B, T), both ZEROED by the caller; d_s receives the gate adjoint (STMGCN.py:44);
 *   dw_scratch : (L, stmgcn_lstm16_grid(rows), 128*256), no initialisation needed;
 *   zero_tile  : 16 KB of zeros (the h_prev operand at t = 0 without an initial state).
 * grads: 4*L device pointers in nn.LSTM parameter order, per layer d_w_ih (256, in_l), d_w_hh (256, 64), d_b_ih (256),
 * d_b_hh (256) (in_0 = C, else 64); overwritten, not accumulated. */
int32_t stmgcn_lstm16_bwd(int32_t t_len, int32_t n_layers, int64_t rows, int32_t c_in, int64_t b_inner, int32_t planes,
                          const float* xo, const float* s_gate, const void* const* wimg, const float* const* bias,
                          const float* wih_t, const void* h0p, const float* c0, const void* hp, const float* cs,
                          const float* d_top, float* dh_rec, float* dc, float* dx_work, float* d_s, float* dbp,
                          float* dw_scratch, const void* zero_tile, float* const* grads, void* stream);

/* ---- fusion over graphs + output FC (STMGCN.py:116-118) ------------------------------------------
 * feat = sum_m g[m] (each (R, G) node-major); y[b, n, c] = feat[n*B+b, :] . fcw[c, :] + fcb[c]. */
int32_t stmgcn_fuse_out_fwd(const float* const* g, int32_t m, int64_t n, int64_t b, int32_t gdim,
                            int32_t c, const float* fcw, const float* fcb, float* feat, float* y,
                            void* stream);
/* d_y (B,N,C) -> d_feat (R,G), d_fcw (C,G) +=, d_fcb (C) += */
int32_t stmgcn_fuse_out_bwd(const float* d_y, const float* feat, int64_t n, int64_t b, int32_t gdim,
                            int32_t c, const float* fcw, float* d_feat, float* d_fcw, float* d_fcb,
                            void* stream);

#ifdef __cplusplus
}
#endif
#endif /* STMGCN_B200_H_ */
