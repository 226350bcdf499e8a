/*
 * geniconet_b200 -- C ABI of the B200-native icosahedral-convolution hot path.
 *
 * The reference (hrdkjain/GenIcoNet) has NO FFI: its hot path is the Python module
 * surface  icocnn.ico_conv.{IcoConvS2S,IcoUpsampleS2S}  (models.py:5-6) and the loss
 * classes of losses.py.  This header is the boundary a maintainer binds instead
 * (ctypes stub shown in INTEGRATION.md); every entry point names the reference
 * interface it replaces.
 *
 * Conventions
 *   - plain C, no torch types; device pointers are raw CUDA device pointers that the
 *     caller owns; `stream` is a cudaStream_t passed as void*.
 *   - every function returns 0 on success, a negative gin_status on failure; the text of
 *     the last failure on the calling thread is gin_last_error().
 *   - the library never allocates device memory and keeps no device state: index tables
 *     ("plans") are built on the HOST into a caller buffer (gin_plan_build) and uploaded by
 *     the caller; ops take both copies: `plan_host` (launch geometry is read from its
 *     header) and `plan_dev` (the kernels read the tables).
 *   - activations are fp32, pixel-major / channel-minor ("channels last"):
 *     element (b, p, c) of a level-s map lives at  b*P*C + p*C + c,  P = 10*4^s,
 *     p = chart*n*2n + i*2n + j  (data.py:64-69, ico_utils.py:20-23).  The input of
 *     gin_hexconv_fwd / gin_hexconv_wgrad may instead use arbitrary element strides
 *     (sb, sp, sc) so the NCHW xyz input of models.py:104 needs no transpose.
 *   - corner_mode: 0 = 'zeros', 1 = 'average' (models.py:11, run.py:683).
 *   - the fp32 entry points gin_hexconv_{fwd,dgrad,wgrad} run the exact-fp32 CUDA-core kernels: with GIN_IMPL_AUTO
 *     the narrow xyz layer (Cin = 3) takes the warp-level memory-bound kernels (gin_narrow.cuh), anything else and
 *     GIN_IMPL_SIMT the generic fp32 gather-GEMM; the tcgen05 implicit GEMM (bf16 operands, fp32 accumulate in TMEM) is
 *     gin_cast_bf16 + gin_hexconv_*_bf16 and is what the Python layer uses whenever both channel counts are
 *     multiples of 64.
 */
#ifndef GENICONET_B200_H
#define GENICONET_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef enum {
  GIN_OK = 0,
  GIN_ERR_ARG = -1,       /* bad argument (shape, level, null pointer, alignment) */
  GIN_ERR_PLAN = -2,      /* plan blob does not match the call */
  GIN_ERR_CUDA = -3,      /* a CUDA runtime call / launch failed */
  GIN_ERR_UNSUPPORTED = -4
} gin_status;

enum { GIN_IMPL_AUTO = 0, GIN_IMPL_SIMT = 1, GIN_IMPL_TC = 2 };
enum { GIN_CORNER_ZEROS = 0, GIN_CORNER_AVERAGE = 1 };

int gin_version(void);
/* 1: forward-side 16-bit operands (activation copies, forward weight tiles) are fp16 (default), 0: bf16 (GIN_FWD_FP16=0).
 * Gradient-side operands are always bf16.  A checker needs this to round its operands the same way. */
int gin_forward_operand_is_fp16(void);
const char* gin_last_error(void);

/* ------------------------------------------------------------------ host: geometry -- */
/* Row a1 (SURVEY 8a): the chart-padding index map that icocnn builds inside
 * IcoConvS2S/IcoUpsampleS2S (absent source; rule restated in-tree at losses.py:22-31).
 * out[k][i+1][j+1], k<5, i in [-1,n], j in [-1,2n]  =  source pixel id, P (north pole),
 * P+1 (south pole) or -1 (cell never read).  gin_index_map_len = 5*(n+2)*(2n+2). */
int gin_index_map_len(int level);
int gin_index_map(int level, int32_t* out);

/* icocnn.utils.ico_geometry.get_ico_faces (losses.py:34) / get_icosahedral_grid
 * (generate.py:151): faces [20*4^s][3] (outward winding), vertices [P+2][3] (unit sphere). */
int gin_ico_faces_len(int level);
int gin_ico_faces(int level, int32_t* out);
int gin_ico_vertices(int level, float* out);

/* ------------------------------------------------------------------ host: plans ----- */
/* kind of plan: */
enum { GIN_PLAN_HEXCONV = 1, GIN_PLAN_UPSAMPLE = 2, GIN_PLAN_LOSS = 3 };
/* level = INPUT subdivision level of the layer (models.py:14,25-33: `subdivisions`);
 * stride in {1,2} (ignored unless HEXCONV). Returns bytes (0 on error). */
size_t gin_plan_bytes(int kind, int level, int stride, int corner_mode);
int gin_plan_build(int kind, int level, int stride, int corner_mode, void* host_buf, size_t bytes);

/* ------------------------------------------------------------------ device: hexconv -- */
/* Packed weights: one buffer holding the kernel-native copies of weight[Cout][Cin][7]
 * (fp32 [7][Cin][Cout] and [7][Cout][Cin]; bf16 K-major copies for tcgen05). */
size_t gin_hexconv_packed_bytes(int Cin, int Cout);
int gin_hexconv_pack_weights(const float* weight, void* packed, int Cin, int Cout, void* stream);

/* Only the bf16 tcgen05 tile images, of the weight [w0; w1] concatenated along Cout (w1 may be NULL with Cout1 = 0): the
 * fused chains run the two sibling convolutions of a residual block (models.py:25-33, 45-55) as one GEMM.  Channel counts
 * must be multiples of 64; `packed` has gin_hexconv_packed_bytes(Cin, Cout0 + Cout1) bytes (the fp32 parts stay unwritten). */
int gin_hexconv_pack_weights_bf16(const float* w0, int Cout0, const float* w1, int Cout1, void* packed, int Cin, void* stream);
/* The same for n <= 24 weights in ONE launch (host arrays of n entries each; w1[j] may be NULL with Cout1[j] = 0). */
int gin_hexconv_pack_weights_bf16_multi(int n, const float* const* w0, const int* Cout0, const float* const* w1, const int* Cout1,
                                        void* const* packed, const int* Cin, void* stream);

/* IcoConvS2S.forward (models.py:14,25-33,45-55,104,165,269,279): rows a1+a2+a3.
 * y[b,p,:] = bias + sum_t W_t^T x~[b, p+t, :] with the padding fused into the gather. */
int gin_hexconv_fwd(const void* plan_host, const void* plan_dev, const float* x, int64_t sb, int64_t sp, int64_t sc,
                    const void* packed, const float* bias /* may be NULL */, float* y,
                    int B, int Cin, int Cout, int impl, void* stream);
/* The xyz input layer (Cin = 3, models.py:104) inside a fused chain: the same forward, with the BatchNorm column sums of its output
 * taken in the epilogue (stats_ws: gin_hexconv_narrow_stats_ws_bytes(Cout); *nparts rows of [2][Cout] for gin_bn_stats_from_parts) and
 * y optionally written as fp16 (it is only read by BatchNorm kernels).  GIN_ERR_UNSUPPORTED for any other layer. */
size_t gin_hexconv_narrow_stats_ws_bytes(int Cout);
int gin_hexconv_fwd_narrow_stats(const void* plan_host, const void* plan_dev, const float* x, int64_t sb, int64_t sp, int64_t sc,
                                 const void* packed, const float* bias, void* y, int y_fp16, int B, int Cin, int Cout, float* stats_ws,
                                 int* nparts, void* stream);
/* autograd backward of the above (run.py:249), row a5: dgrad = adjoint of pad o conv. */
int gin_hexconv_dgrad(const void* plan_host, const void* plan_dev, const float* dy, const void* packed, float* dx,
                      int B, int Cin, int Cout, int impl, void* stream);
/* wgrad: dW[Cout][Cin][7], db[Cout] (db may be NULL). ws: gin_hexconv_wgrad_ws_bytes(). */
size_t gin_hexconv_wgrad_ws_bytes(int Cin, int Cout);
int gin_hexconv_wgrad(const void* plan_host, const void* plan_dev, const float* x, int64_t sb, int64_t sp, int64_t sc,
                      const float* dy, float* dW, float* db, void* ws,
                      int B, int Cin, int Cout, int impl, void* stream);

/* tcgen05 path.  The tensor-core kernels read a 16-bit copy of the gathered activation: gin_cast_bf16 writes
 * [B*P + 2B][C] = the pixels followed by the per-sample pole means (so a pole cell is an ordinary row).
 * `which` = 0: a conv INPUT x (level of `subdivisions`) in the FORWARD operand format (fp16 unless
 *              gin_forward_operand_is_fp16() == 0) -- what gin_hexconv_fwd_bf16 reads;
 *           1: a conv OUTPUT gradient dy (output level) in bf16 -- what dgrad and wgrad read;
 *           2: a conv INPUT x in bf16 -- what wgrad reads (a kind::f16 MMA needs both operands in one format; identical to
 *              which = 0 when the forward format is bf16).
 * Accumulation is fp32 in TMEM, outputs are fp32.  Needs Cin % 64 == 0 and Cout % 64 == 0. */
size_t gin_cast_bf16_bytes(int B, int level, int C);
int gin_cast_bf16(const void* plan_host, const void* plan_dev, int which, const float* x, void* xb, int B, int C, void* stream);
/* Same cast fused with the per-channel sums of x over all B*P pixels: with which = 1 this is the conv bias gradient
 * (IcoConvS2S.bias.grad = sum of dy over batch and pixels), obtained from the pass that reads dy anyway.
 * Needs (C/8) | 256.  ws: gin_cast_bf16_colsum_ws_bytes(C) bytes of scratch (contents irrelevant). Deterministic. */
size_t gin_cast_bf16_colsum_ws_bytes(int C);
int gin_cast_bf16_colsum(const void* plan_host, const void* plan_dev, int which, const float* x, void* xb, float* colsum, void* ws,
                         int B, int C, void* stream);
int gin_hexconv_fwd_bf16(const void* plan_host, const void* plan_dev, const void* xb, const void* packed, const float* bias,
                         float* y, int B, int Cin, int Cout, void* stream);
/* Forward that also leaves the BatchNorm statistics of its output behind: stats_ws (gin_hexconv_stats_ws_bytes(Cout) bytes)
 * receives *nparts rows of [2][Cout] per-CTA column sums of y and y^2 (taken in the epilogue, so the statistics cost no extra
 * pass over y); gin_bn_stats_from_parts turns a column slice of them into stat[4][C].  *nparts = 0 when the kernel that ran
 * cannot produce them (then call gin_bn_stats). */
size_t gin_hexconv_stats_ws_bytes(int Cout);
int gin_hexconv_fwd_bf16_stats(const void* plan_host, const void* plan_dev, const void* xb, const void* packed, const float* bias,
                               float* y, int B, int Cin, int Cout, float* stats_ws, int* nparts, void* stream);
/* The forward of the fused chains.  bias1 != NULL: two sibling convolutions run as ONE GEMM with concatenated output channels --
 * columns [0, split) take bias0, columns [split, Cout) take bias1 (no concatenated bias tensor has to be built).  y_fp16 != 0:
 * y is written as fp16 [B*P][Cout] (it is only read by the BatchNorm kernels below: half the bytes of its one write and three
 * reads; the statistics still come from the fp32 accumulators).  GIN_ERR_UNSUPPORTED when the plan / size does not run the
 * second-generation patch kernel (then use gin_hexconv_fwd_bf16_stats with an fp32 y). */
int gin_hexconv_fwd_bf16_stats2(const void* plan_host, const void* plan_dev, const void* xb, const void* packed, const float* bias0,
                                const float* bias1, int split, void* y, int y_fp16, int B, int Cin, int Cout, float* stats_ws,
                                int* nparts, void* stream);
int gin_hexconv_dgrad_bf16(const void* plan_host, const void* plan_dev, const void* dyb, const void* packed, float* dx,
                           int B, int Cin, int Cout, void* stream);
/* dy (fp32) is only read for db and may be NULL when db is NULL */
int gin_hexconv_wgrad_bf16(const void* plan_host, const void* plan_dev, const void* xb, const void* dyb, const float* dy,
                           float* dW, float* db, void* ws, int B, int Cin, int Cout, void* stream);

/* ------------------------------------------------------------------ device: upsample - */
/* IcoUpsampleS2S.forward (models.py:13,45,53), row a4, and its backward. */
int gin_upsample_fwd(const void* plan_host, const void* plan_dev, const float* x, float* y, int B, int C, void* stream);
int gin_upsample_bwd(const void* plan_host, const void* plan_dev, const float* dy, float* dx, int B, int C, void* stream);

/* ------------------------------------------------------------------ device: fused BN ---- */
/* SURVEY 8f rank 1: torch.nn.BatchNorm2d (training) + ReLU + residual add of models.py:37-39,59-61 fused with the bf16
 * operand cast of the next convolution.  All maps are pixel-major; `ld` = row stride in elements, so a column slice of a wider
 * matrix (the concatenated output of two sibling convolutions) is addressed without a copy.  Needs (C/8) | 256.
 * ws: gin_bn_ws_bytes(C) bytes of scratch.  Deterministic (two-stage reductions, fp64 finals).
 * gin_bn_stats: stat[4][C] = batch mean, invstd (biased variance, eps), scale = gamma*invstd, shift = beta - mean*scale;
 *   running_mean / running_var (may be NULL) get torch's momentum update with the unbiased variance. */
size_t gin_bn_ws_bytes(int C);
int gin_bn_stats(const float* y, int64_t ld, int64_t rows, int C, const float* gamma, const float* beta, float eps, float momentum,
                 float* running_mean, float* running_var, int64_t* num_batches_tracked /* may be NULL; += 1 */, float* stat, void* ws,
                 void* stream);
/* The same from per-CTA partial sums `parts` = nparts rows of [2][ld] (here pointing at the first of the C columns wanted). */
int gin_bn_stats_from_parts(const float* parts, int nparts, int64_t ld, int64_t rows, int C, const float* gamma, const float* beta, float eps,
                            float momentum, float* running_mean, float* running_var, int64_t* num_batches_tracked, float* stat, void* stream);
/* Two BatchNorms from column slices colA / colB of the same partial-sum rows (the two sibling convolutions of a residual block run
 * as one GEMM) in one launch. */
int gin_bn_stats_from_parts2(const float* parts, int nparts, int64_t ld, int64_t rows, int C, int colA, const float* gammaA, const float* betaA,
                             float epsA, float momentumA, float* rmeanA, float* rvarA, int64_t* nbtA, float* statA, int colB,
                             const float* gammaB, const float* betaB, float epsB, float momentumB, float* rmeanB, float* rvarB,
                             int64_t* nbtB, float* statB, void* stream);
/* out = act(y1*scale1 + shift1 [+ y2*scale2 + shift2]) at level `level`: out_b (may be NULL) = 16-bit [B*P + 2B][C] (pixels, then the
 * per-sample pole means) in the forward operand format -- exactly what gin_cast_bf16(which = 0) would produce from out;
 * out_f (may be NULL) = fp32 [B*P][C]; out_w (may be NULL) = the same rows as out_b in bf16 (which = 2: wgrad operand, ReLU mask). */
/* y_fp16 != 0: y1 / y2 (and y / yA / yB below) are fp16 maps (gin_hexconv_fwd_bf16_stats2), `ld` counts elements either way. */
int gin_bn_act_fwd(const void* y1, int64_t ld1, const float* stat1, const void* y2 /* may be NULL */, int64_t ld2, const float* stat2,
                   int y_fp16, int relu, void* out_b, float* out_f, void* out_w, int B, int level, int C, void* stream);
/* backward of out = act(bn(y) [+ ...]) with respect to y: g = dout * (mask_b > 0) (mask_b = a 16-bit copy of out, either format; NULL: no ReLU),
 * bstat[4][C] = dbeta, dgamma, mean(g), mean(g*yhat);  dy = scale*(g - mean(g) - yhat*mean(g*yhat)) is written as the bf16
 * copy dy_b [B*P + 2B][.] with row stride ldo (pole-mean rows included) and / or as fp32 dy_f with row stride ldf.
 * relu_from_y != 0 (with mask_b != NULL): the caller states that mask_b is the output of gin_bn_act_fwd(y, stat, relu = 1) itself; the
 * kernels may then re-evaluate out > 0 from y and stat (bit-identical arithmetic) instead of reading the mask -- 2 B / element
 * less traffic in each of the two passes. */
int gin_bn_act_bwd(const float* dout, int64_t ldg, const void* mask_b, const void* y, int64_t ld, int y_fp16, const float* stat, float* bstat,
                   void* dy_b, int64_t ldo, float* dy_f, int64_t ldf, void* ws, int B, int level, int C, int relu_from_y, void* stream);
/* Backward of out = relu(bnA(yA) + bnB(yB)) (the residual output of models.py:38-39, 60-61) with respect to yA and yB in one pass pair:
 * both BatchNorms see the same g = dout * (mask_b > 0), which is read once.  ws: gin_bn_pair_ws_bytes(C).
 * relu_from_y != 0: mask_b is the output of gin_bn_act_fwd(yA, statA, yB, statB, relu = 1); see gin_bn_act_bwd. */
size_t gin_bn_pair_ws_bytes(int C);
int gin_bn_act_bwd_pair(const float* dout, int64_t ldg, const void* mask_b, const void* yA, int64_t ldA, const float* statA, float* bstatA,
                        void* dyA_b, int64_t ldoA, const void* yB, int64_t ldB, const float* statB, float* bstatB, void* dyB_b, int64_t ldoB,
                        int y_fp16, void* ws, int B, int level, int C, int relu_from_y, void* stream);
/* IcoUpsampleS2S.forward whose result exists only as the next convolution's operand copy out_b = 16-bit [B*Pf + 2B][C] in the
 * forward operand format (upsample plan), plus (out_w, may be NULL) its bf16 twin for wgrad.  in: the fp32 coarse map
 * [B*Pc][C] (in_is_f32 = 1) or its forward-format operand copy [B*Pc + 2B][C] (0). */
int gin_upsample_bf16(const void* plan_host, const void* plan_dev, const void* in, int in_is_f32, void* out_b, void* out_w, int B, int C,
                      void* stream);

/* ------------------------------------------------------------------ device: VAE ------ */
/* VAE.reparameterize (models.py:89-92), row a6: eps ~ N(0,1) from Philox4x32-10
 * (seed, offset), z = eps*exp(0.5*logvar)+mu; eps is written out for the backward. */
int gin_reparam_fwd(const float* mu, const float* logvar, float* eps, float* z, int64_t n,
                    uint64_t seed, uint64_t offset, void* stream);
/* Same with the Philox offset taken as offset + *step, and *step incremented afterwards ON THE DEVICE: a captured CUDA graph
 * that is replayed every training step still draws fresh noise (a host-side offset is frozen into the graph). */
int gin_reparam_fwd_step(const float* mu, const float* logvar, float* eps, float* z, int64_t n, uint64_t seed, uint64_t offset,
                         uint64_t* step /* device */, void* stream);
int gin_reparam_bwd(const float* dz, const float* logvar, const float* eps, float* dmu, float* dlogvar,
                    int64_t n, void* stream);
/* KLD_Loss.forward (losses.py:92-108), row a9: out[0] = mean_b(-0.5*mean_i(1+lv-mu^2-exp(lv))). */
int gin_kld_fwd(const float* mu, const float* logvar, float* out, void* ws /* 4096 B */, int64_t n, void* stream);
int gin_kld_bwd(const float* mu, const float* logvar, const float* dout /* device scalar */, float scale,
                float* dmu, float* dlogvar, int64_t n, void* stream);

/* ------------------------------------------------------------------ device: losses --- */
/* Pole averaging + grid->vertex list (losses.py:22-31,49-51; ico_utils.py:10-24), row a7:
 * x [B,C,5n,2n] with element strides (sb, sp, sc) -> v [B][P+2][C]. */
int gin_pole_vertices_fwd(const void* plan_host, const void* plan_dev, const float* x, int64_t sb, int64_t sp, int64_t sc,
                          float* v, int B, int C, void* stream);
int gin_pole_vertices_bwd(const void* plan_host, const void* plan_dev, const float* dv, float* dx, int64_t sb, int64_t sp, int64_t sc,
                          int B, int C, void* stream);
/* compute_vertex_normals / compute_laplacian_batch (mesh.utils; losses.py:54,57). */
int gin_vertex_normals_fwd(const void* plan_host, const void* plan_dev, const float* v, float* nrm, int B, void* stream);
int gin_laplacian_fwd(const void* plan_host, const void* plan_dev, const float* v, float* lap, int B, void* stream);
/* Their backward (autograd through losses.py:54,57 when the reference's unmodified losses.py runs over the `mesh` shim):
 * g_nrm / g_lap [B][P+2][3] are the cotangents of the two outputs (either may be NULL), dv [B][P+2][3] receives the vertex
 * gradient.  ws: gin_ring_ops_ws_bytes(B, level). */
size_t gin_ring_ops_ws_bytes(int B, int level);
int gin_ring_ops_bwd(const void* plan_host, const void* plan_dev, const float* v, const float* g_nrm, const float* g_lap, float* dv,
                     void* ws, int B, void* stream);
/* Point2Point_Loss.forward (losses.py:47-82), row a8, fused: out[0..3] = l_pos, l_nor, l_lap,
 * f_pos*l_pos + f_nor*l_nor + f_lap*l_lap.  target [B][9][P+2] (generate.py:200-203).
 * ws: gin_p2p_ws_bytes(B, level). The backward re-derives everything from x/target. */
size_t gin_p2p_ws_bytes(int B, int level);
int gin_p2p_loss_fwd(const void* plan_host, const void* plan_dev, const float* x, int64_t sb, int64_t sp, int64_t sc,
                     const float* target, float f_pos, float f_nor, float f_lap,
                     float* out, void* ws, int B, void* stream);
int gin_p2p_loss_bwd(const void* plan_host, const void* plan_dev, const float* x, int64_t sb, int64_t sp, int64_t sc,
                     const float* target, float f_pos, float f_nor, float f_lap,
                     const float* dout /* device scalar */, float* dx, void* ws, int B, void* stream);

/* ------------------------------------------------------------------ device: decoder head --- */
/* `Conv2d(64,3,1) -> Tanh` (models.py:151-154) over a pixel-major activation: x [B*P][Cin] fp32, w [Cout][Cin], bias [Cout],
 * y / dy [B][Cout][P] (plain NCHW), dx [B*P][Cin], dw [Cout][Cin], db [Cout].  Only Cin = 64, Cout = 3 (GIN_ERR_UNSUPPORTED
 * otherwise: callers keep the stock modules).  ws: gin_head_ws_bytes(). */
size_t gin_head_ws_bytes(void);
int gin_head_fwd(const float* x, const float* w, const float* bias, float* y, int B, int64_t P, int Cin, int Cout, void* stream);
int gin_head_bwd(const float* x, const float* w, const float* y, const float* dy, float* dx, float* dw, float* db, void* ws,
                 int B, int64_t P, int Cin, int Cout, void* stream);

/* ------------------------------------------------------------------ device: evaluation metric (SURVEY 8f rank 4) --- */
/* ico_utils.py:26-44 computeDistance(mode='point2mesh') -> kaolin 0.9.1 point_to_mesh_distance: per point the SQUARED distance
 * to the closest triangle, and that triangle's index (lowest index among equal distances).
 * points [B][N][3], verts [B][V][3] fp32, faces [F][3] int32 (shared by the batch), dist [B][N] fp32, face_idx [B][N] int32 or NULL.
 * ws: gin_point_mesh_ws_bytes(B, N). */
size_t gin_point_mesh_ws_bytes(int B, int N);
int gin_point_mesh_distance(const float* points, const float* verts, const int32_t* faces, float* dist, int32_t* face_idx,
                            void* ws, int B, int N, int V, int F, void* stream);

/* ------------------------------------------------------------------ device: Chamfer distance --- */
/* One nearest neighbour between two batched fp32 point sets, x [B][N][3] and y [B][M][3], read with element strides (element (b, i, c)
 * of x at x[b*xsb + i*xsn + c*xsc]; the xyz rows of a [B][9][V] target are (9*V, 1, V)).  Brute force on the fp32 CUDA cores.
 * Forward: d_xy [B][N] = squared distance of x_i to its nearest point of y, idx_xy [B][N] = that point's index (int32; the lowest
 * index among equal distances); d_yx / idx_yx [B][M] the same towards x.  A direction runs when its distance output is given;
 * its index output may be NULL, an index output without its distance output is an error.  The distance is recomputed in
 * difference form for the chosen pair.  Deterministic.
 * Backward: dx [B][N][3] = 2 g_xy_i (x_i - y_idx_xy(i)) + sum_{j : idx_yx(j) = i} 2 g_yx_j (x_i - y_j), dy [B][M][3] symmetrically
 * (both contiguous; either may be NULL, not both).  g_xy [B][N] / g_yx [B][M] are the cotangents of d_xy / d_yx; either may be NULL
 * (one-sided loss), not both; a cotangent needs its indices.  The scatter sum is exact int64 fixed point: bit-reproducible, no
 * floating-point atomics.
 * ws: gin_chamfer_ws_bytes(B, N, M), contents irrelevant.  B = 0: no-op.  Needs N, M >= 1, B <= 65535, B*max(N, M) < 2^31. */
size_t gin_chamfer_ws_bytes(int B, int N, int M);
int gin_chamfer_fwd(const float* x, int64_t xsb, int64_t xsn, int64_t xsc, const float* y, int64_t ysb, int64_t ysn, int64_t ysc,
                    float* d_xy, int32_t* idx_xy, float* d_yx, int32_t* idx_yx, void* ws, int B, int N, int M, void* stream);
int gin_chamfer_bwd(const float* x, int64_t xsb, int64_t xsn, int64_t xsc, const float* y, int64_t ysb, int64_t ysn, int64_t ysc,
                    const int32_t* idx_xy, const float* g_xy, const int32_t* idx_yx, const float* g_yx, float* dx, float* dy, void* ws,
                    int B, int N, int M, void* stream);

/* ------------------------------------------------------------------ device: optimizer step --- */
/* The Adam step of the training loop (run.py:446 `torch.optim.Adam(model.parameters(), lr)`, run.py:250 `optimizer.step()`) over
 * a LIST of fp32 tensors in one launch; same arithmetic as torch.optim.Adam (amsgrad = maximize = False, L2 weight_decay):
 *   t = *step + 1;  g' = g + weight_decay*p;  m += (1-beta1)*(g'-m);  v = beta2*v + (1-beta2)*g'^2;
 *   p -= lr/(1-beta1^t) * m / (sqrt(v)/sqrt(1-beta2^t) + eps);  *step = t  (written when every tensor has been updated).
 * table_dev: GinAdamTensor[count] in device memory, all pointers device pointers.  chunk_first_dev: int32[count + 1], prefix sums
 * of ceil(n / gin_adam_chunk()) over the table (chunk_first[count] = total_chunks).  lr_dev != NULL: the learning rate is read
 * from the device at run time (a captured graph then follows a scheduler), else `lr`.  ticket_dev: one zero-initialised uint32
 * owned by the caller (left zero again by every call). */
typedef struct {
  float* p;          /* parameter, updated in place */
  const float* g;    /* gradient */
  float* m;          /* exp_avg */
  float* v;          /* exp_avg_sq */
  float* step;       /* fp32 scalar: number of steps taken so far */
  int64_t n;         /* elements */
} GinAdamTensor;
int gin_adam_chunk(void);
int gin_adam_step(const void* table_dev, const int32_t* chunk_first_dev, int count, int total_chunks, float lr, const float* lr_dev, float beta1,
                  float beta2, float eps, float weight_decay, void* ticket_dev, void* stream);

/* ------------------------------------------------------------------ device: eval-mode (inference) forward ---- */
/* Forward-only convolution with an eval-mode BatchNorm applied in the epilogue (second-generation patch kernel, stride 1 or 2).
 * Per output column: o = acc*scale[col] + shift[col] (the conv bias folded into shift: gin_bn_eval_consts); ReLU on columns
 * < relu_split; with res != NULL (fp32, or fp16 when res_fp16; row stride ld_res elements) o = relu(o + res[row][col]).
 * Columns < split go to destination 0, the others (split < Cout) to destination 1: out*_b = the 16-bit forward operand copy
 * [B*P + 2B][width] (pixels, then the pole means, bit for bit what gin_cast_bf16(which = 0) makes of the fp32 values), out*_f =
 * fp32 [B*P][width]; each may be NULL, not both.  split is a multiple of 64 in (0, Cout]; split == Cout: one destination.
 * ring_ws: gin_hexconv_affine_ring_bytes(B, Cout) bytes, needed when an operand copy is written.
 * GIN_ERR_UNSUPPORTED where gin_hexconv_fwd_bf16_stats2 would return it (compose it with gin_bn_act_fwd there). */
size_t gin_hexconv_affine_ring_bytes(int B, int Cout);
int gin_hexconv_fwd_affine(const void* plan_host, const void* plan_dev, const void* xb, const void* packed, const float* scale,
                           const float* shift, int relu_split, const void* res, int64_t ld_res, int res_fp16, int split, void* out0_b,
                           float* out0_f, void* out1_b, float* out1_f, float* ring_ws, int B, int Cin, int Cout, void* stream);
/* The eval constants of `count` BatchNorms in one launch, read from the device at run time (a captured graph follows later in-place
 * updates of the parameters and running statistics).  table_dev: GinBnEvalEntry[count] in device memory; max_C >= every C.
 *   scale = gamma*invstd, invstd = 1/sqrt(running_var + eps);  shift = beta + scale*(conv_bias - running_mean);
 *   stat (torch's gin_bn_stats layout, for gin_bn_act_fwd): running_mean, invstd, scale, beta - running_mean*scale. */
typedef struct {
  const float* gamma;          /* may be NULL: 1 */
  const float* beta;           /* may be NULL: 0 */
  const float* running_mean;
  const float* running_var;
  const float* conv_bias;      /* may be NULL: 0 */
  float* scale;                /* [C], may be NULL */
  float* shift;                /* [C], may be NULL */
  float* stat;                 /* [4][C], may be NULL */
  float eps;
  int C;
} GinBnEvalEntry;
int gin_bn_eval_consts(const void* table_dev, int count, int max_C, void* stream);

/* ------------------------------------------------------------------ device: eval-mode BatchNorm backward ---- */
/* Backward of out = relu(bn(y)) with bn in eval mode (running statistics; stat[4][C] as gin_bn_eval_consts writes it: running_mean,
 * invstd, scale = gamma*invstd, shift): g = dout * (out > 0), dy = scale*g -- ONE streaming pass, no reduction ahead of it.
 * The mask is re-evaluated from y and stat when relu_from_y != 0 (bit-identical to gin_bn_act_fwd(y, stat, relu = 1); mask_b is
 * then ignored), else read from mask_b (a 16-bit copy of out, either format; NULL: no ReLU).
 * dy is written as the bf16 copy dy_b [B*P + 2B][.] with row stride ldo (the pole-mean rows included, bit for bit what
 * gin_cast_bf16(which = 1) makes of the fp32 dy) and / or as fp32 dy_f with row stride ldf.
 * bsum (may be NULL: no reduction at all) = [3][C]: dbeta = sum g, dgamma = sum g*yhat (yhat = (y - running_mean)*invstd) and the
 * gradient of the conv bias that feeds the BatchNorm, scale * sum g (not zero in eval mode).  Two-stage, fixed-order fp64 sums.
 * C/8 divides 256 and C <= 256; every row stride >= C and a multiple of 8.  ws: gin_bn_eval_bwd_ws_bytes(C) when a sum is taken. */
size_t gin_bn_eval_bwd_ws_bytes(int C);
int gin_bn_eval_bwd(const float* dout, int64_t ldg, const void* mask_b, const void* y, int64_t ld, int y_fp16, const float* stat, float* bsum,
                    void* dy_b, int64_t ldo, float* dy_f, int64_t ldf, void* ws, int B, int level, int C, int relu_from_y, void* stream);
/* The residual output out = relu(bnA(yA) + bnB(yB)), both in eval mode: dout is read once, dyA_b / dyB_b are bf16 copies (pole
 * rows included) with row strides ldoA / ldoB.  bsumA / bsumB [3][C] as above, each may be NULL; relu_from_y: the mask is
 * re-evaluated exactly as gin_bn_act_fwd(yA, statA, yB, statB, relu = 1) computed out. */
int gin_bn_eval_bwd_pair(const float* dout, int64_t ldg, const void* mask_b, const void* yA, int64_t ldA, const float* statA, float* bsumA,
                         void* dyA_b, int64_t ldoA, const void* yB, int64_t ldB, const float* statB, float* bsumB, void* dyB_b, int64_t ldoB,
                         int y_fp16, void* ws, int B, int level, int C, int relu_from_y, void* stream);

/* number of kernel launches issued through this library since load (bench.py's gpu_launches) */
int64_t gin_launch_count(void);

#ifdef __cplusplus
}
#endif
#endif
