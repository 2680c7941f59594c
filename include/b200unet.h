/*
 * b200unet.h  --  C-ABI of the B200-native 3D U-Net forward/backward engine (libb200unet.so)
 *
 * Drop-in boundary for the ONE hot path of wolny/pytorch-3dunet (reference @ a33e2c7): everything that
 * `pytorch3dunet.unet3d.model.get_model(cfg)(x)` and its autograd execute.  The reference has no FFI of its
 * own (it is pure Python over torch.nn); each entry point below names the reference call site
 * (file:line relative to the reference checkout) whose ATen library call it replaces.
 *
 * Conventions
 *   - plain pointers and sizes only; no torch types.  All pointers are DEVICE pointers unless noted.
 *   - activations are bf16 "NDHWC": [N][D][H][W][C] contiguous, C % 8 == 0 (16-byte channel vectors).
 *   - every function only ENQUEUES work on `stream` (a cudaStream_t passed as void*); it never
 *     allocates, frees or synchronises.  Buffers are owned by the caller (PyTorch caching allocator).
 *   - return 0 on success, non-zero on error; b200_last_error() returns the message (thread local).
 *   - "partials": float [N][P][C][2] per-block partial sums (sum v, sum v*w); P is returned by the
 *     matching *_partials_count() query; reduce them with b200_partials_finalize (deterministic, fp64).
 */
#ifndef B200UNET_H_
#define B200UNET_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef void* b200_stream_t; /* cudaStream_t */

/* activation kinds (create_conv buildingblocks.py:45-51; ResNetBlock non_linearity :270-275) */
/* OR into b200_conv3_fwd's pmode: the bias table uses the phase-aware border classes of the virtual-concat convolution */
#define B200_PMODE_PHASE_BIAS 0x100
enum { B200_ACT_NONE = 0, B200_ACT_RELU = 1, B200_ACT_LEAKY = 2, B200_ACT_ELU = 3 };
/* conv implementation selector */
enum { B200_IMPL_AUTO = 0, B200_IMPL_DIRECT = 1, B200_IMPL_TCGEN05 = 2 };
/* final activation (model.py:93-98) */
enum { B200_FINAL_NONE = 0, B200_FINAL_SIGMOID = 1, B200_FINAL_SOFTMAX = 2 };

int b200_version(void);
/* copies the calling thread's last error message into buf (NUL terminated), returns its length */
int b200_last_error(char* buf, size_t len);
/* 1 if the current device is sm_100 (tcgen05 kernels usable), else 0 */
int b200_device_is_sm100(void);

/* ---- layout / input (datasets' ToTensor yields NCDHW fp32, augment/transforms.py:816-826) ---------- */
int b200_ncdhw_f32_to_ndhwc_f32(const float* src, float* dst, int N, int C, int D, int H, int W, b200_stream_t s);
int b200_ncdhw_f32_to_ndhwc_bf16(const float* src, void* dst, int N, int C, int D, int H, int W, b200_stream_t s);
int b200_ndhwc_bf16_to_ncdhw_f32(const void* src, float* dst, int N, int C, int D, int H, int W, b200_stream_t s);

/* ---- GroupNorm statistics (nn.GroupNorm, buildingblocks.py:75 -> native_group_norm) -------------- */
/* per-(n,c) sum / sum-of-squares of an NDHWC tensor -> partials [N][P][C][2]; P = b200_stats_partials_count */
int b200_stats_partials_count(int N, int C, long long voxels);          /* for b200_stats_ndhwc_bf16 */
int b200_stats_ndhwc_bf16(const void* x, int N, int C, long long voxels, float* partials, b200_stream_t s);
int b200_stats_ncdhw_f32_partials_count(long long voxels);              /* for b200_stats_ncdhw_f32 */
/* the raw network input, NCDHW fp32, any C (the first GroupNorm of order 'gcr' normalises the input itself) */
int b200_stats_ncdhw_f32(const float* x, int N, int C, long long voxels, float* partials, b200_stream_t s);
/* partials of (sum a, sum a*b) over two bf16 NDHWC tensors; P = b200_stats_partials_count */
int b200_stats2_ndhwc_bf16(const void* a, const void* b, int N, int C, long long voxels, float* partials, b200_stream_t s);
/* sums[N][C][2] (double) = sum over P of partials */
int b200_partials_finalize(const float* partials, int N, int P, int C, double* sums, b200_stream_t s);

/* Fold GroupNorm into the following conv (order 'g' before 'c'):
 *   x_hat = a[n,c]*x + b[n,c]   with a = gamma*rstd, b = beta - gamma*mean*rstd  (group stats from `sums`)
 *   wf[n][tap][co][ci] = bf16( W[co][ci][tap] * a[n][ci] )
 *   biascls[n][cls][co] = sum over the taps that are in-bounds for border class `cls` of sum_ci W[co][ci][tap]*b[n][ci]
 * (the reference zero-pads AFTER normalising, so the shift term only exists for in-bounds taps).
 * With sums == NULL (no GroupNorm before the conv): a=1, b=0, n_w = 1 weight copy, biascls = conv bias (or 0).
 * mean_rstd[N][G][2], ab[N][C][2] are saved for backward. */
int b200_gn_fold(const double* sums, const float* gamma, const float* beta, int G, double count,
                 const float* W, const float* conv_bias, int N, int Cin, int Cout,
                 void* wf, float* biascls, float* mean_rstd, float* ab, b200_stream_t s);
/* the same chain in two launches instead of four (engine.py conv3 / groupnorm_act): per-block partial sums -> fp64 sums + GroupNorm
   coefficients; folded weights + border-class bias table */
int b200_gn_stats_coeffs(const float* partials, int N, int P, int C, const float* gamma, const float* beta, int G, double count,
                         double* sums, float* mean_rstd, float* ab, b200_stream_t s);
int b200_fold_weights_bias(const float* W, const float* ab, const float* conv_bias, const double* sums, double count, int N, int Cin,
                           int Cout, void* wf, float* biascls, b200_stream_t s);
/* GroupNorm applied as a standalone op AFTER a conv (orders like 'cgr'): y = act(a*x+b), emits partials of y */
int b200_gn_apply_act(const void* x, const float* ab, int N, int C, long long voxels, int act, float slope,
                      void* y, float* partials, b200_stream_t s);
/* same with a residual input: y = act(a*x + b + residual)  (ResNetBlock `out += residual` after a conv3 whose order ends in 'g',
 * buildingblocks.py:243-288 with the block's default order 'cge'); residual may be NULL */
int b200_gn_apply_act_res(const void* x, const float* ab, const void* residual, int N, int C, long long voxels, int act, float slope,
                          void* y, float* partials, b200_stream_t s);
/* a,b only (no weight folding): ab[N][C][2], mean_rstd[N][G][2] */
int b200_gn_coeffs(const double* sums, const float* gamma, const float* beta, int G, double count,
                   int N, int C, float* mean_rstd, float* ab, b200_stream_t s);

/* ---- 3x3x3 convolution, padding 1 (nn.Conv3d, buildingblocks.py:56 -> cudnn_convolution) --------
 * y[n,v,co] = act( sum_{tap,ci} wf[n or 0][tap][co][ci] * x[n,v+tap-1,ci] + biascls[n or 0][cls(v)][co] (+ residual) )
 * x: bf16 NDHWC, or (x_is_f32) fp32 NDHWC (the network input; reference keeps fp32, transforms.py:816-826)
 * n_w: number of per-sample weight copies (N when GroupNorm is folded in, else 1)
 * n_b: same for biascls (N, 1 or 0 = no bias)
 * pmode: 0 no partials; 1 partials of (y, y*y) for the next GroupNorm; 2 partials of (y, y*aux) (GroupNorm backward)
 * P must equal b200_conv3_partials_count(...) for the chosen impl. */
int b200_conv3_partials_count(int impl, int N, int D, int H, int W, int Cin, int Cout);
int b200_conv3_resolve_impl(int impl, int N, int D, int H, int W, int Cin, int Cout, int x_is_f32);
int b200_conv3_fwd(int impl, const void* x, int x_is_f32, const void* wf, int n_w, const float* biascls, int n_b,
                   const void* residual, int act, float slope,
                   int N, int D, int H, int W, int Cin, int Cout,
                   void* y, int pmode, const void* aux, float* partials, b200_stream_t s);
/* dgrad weights: wd[tap'][ci][co] = bf16(W[co][ci][26-tap'])  (convolution_backward's input gradient) */
int b200_prep_dgrad_weights(const float* W, int Cin, int Cout, void* wd, b200_stream_t s);

/* wgrad: G[n][split][tap][ci][co] (fp32) = sum_v dz[n,v,co] * x[n,v+tap-1,ci]  (raw, zero padded x)
 * S = b200_conv3_wgrad_splits(...) */
int b200_conv3_wgrad_resolve_impl(int impl, int N, int D, int H, int W, int Cin, int Cout, int x_is_f32);
int b200_conv3_wgrad_splits(int impl, int N, int D, int H, int W, int Cin, int Cout, int x_is_f32);
int b200_conv3_wgrad(int impl, const void* x, int x_is_f32, const void* dz,
                     int N, int D, int H, int W, int Cin, int Cout, float* G, b200_stream_t s);
/* T[n][tap][co] = sum over v with v+tap-1 in bounds of dz[n,v,co]  (the GroupNorm shift term of wgrad);
 * scratch: b200_border_tap_sums_workspace(...) floats */
int b200_border_tap_sums_workspace(int N, int D, int H, int W, int C);
int b200_border_tap_sums(const void* dz, int N, int D, int H, int W, int C, float* T, float* scratch, b200_stream_t s);
/* same, with the per-channel totals of dz supplied as partial sums [N][Ptot][C][2] (column 0) by the kernel that produced dz
 * (b200_gn_bwd_apply_stats) */
int b200_border_tap_sums_pre(const void* dz, int N, int D, int H, int W, int C, const float* tot_partials, int Ptot, float* T, float* scratch,
                             b200_stream_t s);
/* dW[co][ci][tap] = sum_n ( a[n][ci] * sum_split G + b[n][ci] * T[n][tap][co] ); ab == NULL -> a=1,b=0.
 * Gsum (optional) [N][27][Cin][Cout] receives sum_split G for b200_gn_bwd_sums_from_wgrad (then called with S = 1) */
int b200_wgrad_finalize(const float* G, int N, int S, int Cin, int Cout, const float* ab, const float* T,
                        float* dW, float* Gsum, b200_stream_t s);
/* bias gradient for convs that have one: db[co] = sum_{n,tap=center...}: simply sum_n,v dz = T[n][13][co] summed */
int b200_bias_grad_from_T(const float* T, int N, int C, float* db, b200_stream_t s);

/* GroupNorm-backward sums of a conv's INPUT from the wgrad by-products (G, T) and the weights:
 * sums2[n][ci] = ( sum_v dxhat , sum_v dxhat*x ) -- no extra pass over activations */
int b200_gn_bwd_sums_from_wgrad(const float* G, int S, const float* T, const float* W, int N, int Cin, int Cout,
                                double* sums2, b200_stream_t s);

/* ---- GroupNorm backward (native_group_norm_backward) ------------------------------------------------
 * sums2[N][C][2] = (sum dxhat, sum dxhat*x) ; coef[N][C][3] = (A,B,Cc) with dx = A*dxhat + B*x + Cc */
int b200_gn_bwd_coeffs(const double* sums2, const float* gamma, const float* mean_rstd, int G, double count,
                       int N, int C, float* coef, float* dgamma, float* dbeta, b200_stream_t s);
/* out = (A*dxhat + B*x + Cc) * act'(x) [+ gadd]
 * (x is the post-activation output of its producer when act != NONE; gadd: an already accumulated gradient of the
 *  same shape in "dz form", may alias out) */
int b200_gn_bwd_apply(const void* dxhat, const void* x, const float* coef, int N, int C, long long voxels,
                      int act, float slope, const void* gadd, void* out, b200_stream_t s);
/* same, also emitting partials [N][P][C][2] = (sum out, sum out^2) per block (P = b200_stats_partials_count): the per-channel totals of the
 * gradient it writes, which the NEXT layer's b200_border_tap_sums_pre takes instead of re-reading the tensor */
int b200_gn_bwd_apply_stats(const void* dxhat, const void* x, const float* coef, int N, int C, long long voxels,
                            int act, float slope, const void* gadd, void* out, float* partials, b200_stream_t s);
/* out = g[..., g_co:g_co+C] * act'(y) [+ gadd] : plain masking / accumulation; g is read with channel stride g_cs */
int b200_act_bwd(const void* g, int g_cs, int g_co, const void* y, int N, int C, long long voxels, int act, float slope,
                 const void* gadd, void* out, b200_stream_t s);
/* the same, also emitting the per-channel totals of the result (partials [N][b200_stats_partials_count][C][2]) for the producer conv's
   border-tap sums */
int b200_act_bwd_stats(const void* g, int g_cs, int g_co, const void* y, int N, int C, long long voxels, int act, float slope,
                       const void* gadd, void* out, float* partials, b200_stream_t s);

/* ---- MaxPool3d(2) (buildingblocks.py:356 -> max_pool3d_with_indices), floor mode ---------------- */
int b200_maxpool_fwd(const void* x, int N, int D, int H, int W, int C, void* y, float* partials, b200_stream_t s);
int b200_maxpool_partials_count(int N, int D, int H, int W, int C);
/* dz_full = scatter(dpooled to first argmax of x_full) * act'(x_full) [+ gadd] */
int b200_maxpool_bwd(const void* dpooled, const void* x_full, int N, int D, int H, int W, int C,
                     int act, float slope, const void* gadd, void* dz_full, b200_stream_t s);
/* fused with a deferred GroupNorm backward of another consumer of x: dz = scatter(dpooled)*act'(x) + (A*dxhat + B*x + C)*act'(x); per-channel
   totals of dz to partials [N][P][C][2], P = b200_maxpool_bwd_partials_count (engine.py maxpool backward) */
int b200_maxpool_bwd_partials_count(int N, int D, int H, int W, int C);
int b200_maxpool_bwd_gn(const void* dpooled, const void* x_full, int N, int D, int H, int W, int C, int act, float slope, const void* dxhat,
                        const float* coef, void* dz_full, float* partials, b200_stream_t s);

/* AvgPool3d(2) (Encoder pool_type='avg', buildingblocks.py:358-363 -> avg_pool3d), floor mode; P = b200_maxpool_partials_count */
int b200_avgpool_fwd(const void* x, int N, int D, int H, int W, int C, void* y, float* partials, b200_stream_t s);
int b200_avgpool_bwd(const void* dpooled, const void* x_full, int N, int D, int H, int W, int C,
                     int act, float slope, const void* gadd, void* dz_full, b200_stream_t s);

/* ---- nearest upsample to the encoder's size + channel concat (buildingblocks.py:614, :491) ------ */
int b200_upcat_fwd(const void* enc, int C0, const void* x, int C1, int N, int D, int H, int W, int d, int h, int w,
                   void* cat, float* partials, b200_stream_t s);
int b200_upcat_partials_count(int N, int D, int H, int W, int C);
/* dx_small = (sum over destination voxels that map to each source voxel of dcat[..., C0:]) * act'(x_small) */
int b200_upcat_bwd(const void* dcat, int C0, int C1, const void* x_small, int N, int D, int H, int W, int d, int h, int w,
                   int act, float slope, void* dx_small, b200_stream_t s);

/* same join with InterpolateUpsampling(mode='trilinear') (buildingblocks.py:598-614 -> upsample_trilinear3d, align_corners=False):
 * cat[..., C0:] = trilinear(x -> (D,H,W)); bwd is the adjoint in gather form. P = b200_upcat_partials_count */
int b200_upcat_trilinear_fwd(const void* enc, int C0, const void* x, int C1, int N, int D, int H, int W, int d, int h, int w,
                             void* cat, float* partials, b200_stream_t s);
int b200_upcat_trilinear_bwd(const void* dcat, int C0, int C1, const void* x_small, int N, int D, int H, int W, int d, int h, int w,
                             int act, float slope, void* dx_small, b200_stream_t s);

/* ---- final 1x1x1 conv + Sigmoid/Softmax (model.py:89,141-147) ------------------------------------ */
int b200_final_conv_fwd(const void* x, int N, long long voxels, int C, const float* W, const float* bias, int Cout,
                        int final_act, float* logits, float* probs, b200_stream_t s);
int b200_final_conv_bwd_partials_count(int N, long long voxels, int C, int Cout);
/* dz = (sum_o dlogits[o] W[o][c]) * act'(x); partials[P][Cout*C + Cout] for dW and dbias */
int b200_final_conv_bwd(const float* dlogits, const void* x, int N, long long voxels, int C, const float* W, int Cout,
                        int act, float slope, void* dz, float* partials, b200_stream_t s);
/* generic deterministic reduction out[K] = sum_p partials[p][K] */
int b200_reduce_rows(const float* partials, int P, int K, float* out, b200_stream_t s);

/* ---- implementation-specific entry points (what the dispatchers above call; exported for tests/profiling) --- */
int b200_conv3_igemm_supported(int N, int D, int H, int W, int Cin, int Cout);
int b200_conv3_igemm_partials_count(int N, int D, int H, int W, int Cin, int Cout);
int b200_conv3_igemm_fwd(const void* x, const void* wf, int n_w, const float* biascls, int n_b, const void* residual, int act,
                         float slope, int N, int D, int H, int W, int Cin, int Cout, void* y, int pmode, const void* aux,
                         float* partials, b200_stream_t s);
int b200_conv3_direct_partials_count(int N, int D, int H, int W, int Cout);
int b200_conv3_direct_fwd(const void* x, int x_is_f32, const void* wf, int n_w, const float* biascls, int n_b, const void* residual,
                          int act, float slope, int N, int D, int H, int W, int Cin, int Cout, void* y, int pmode, const void* aux,
                          float* partials, b200_stream_t s);
int b200_conv3_direct_wgrad_splits(int N, int D, int H, int W, int Cin, int Cout, int x_is_f32);
int b200_conv3_direct_wgrad(const void* x, int x_is_f32, const void* dz, int N, int D, int H, int W, int Cin, int Cout, float* G,
                            b200_stream_t s);
int b200_conv3_wgrad_igemm_supported(int N, int D, int H, int W, int Cin, int Cout);
int b200_conv3_wgrad_igemm_splits(int N, int D, int H, int W, int Cin, int Cout);
int b200_conv3_wgrad_igemm(const void* x, const void* dz, int N, int D, int H, int W, int Cin, int Cout, float* G, b200_stream_t s);


/* ---- residual family: 1x1x1 conv with bias (ResNetBlock.conv1, buildingblocks.py:251) ------------------------------
 * y[v,co] = sum_ci W[co][ci] x[v,ci] + bias[co]; transposed=1 reads W as [Cin][Cout]^T (input gradient). partials of y. */
int b200_pointwise_partials_count(int N, long long voxels, int Cout);
int b200_pointwise_fwd(const void* x, int x_is_f32, const float* W, int transposed, const float* bias, int N, long long voxels,
                       int Cin, int Cout, void* y, float* partials, b200_stream_t s);
/* partial rows [N*P][Cout*Cin + Cout] of dW, db; reduce with b200_reduce_rows */
/* ---- gradient w.r.t. the fp32 network input (autograd of the first conv on x: buildingblocks.py:56, ResNetBlock.conv1 :251) ------------
 * b200_input_dgrad_conv3: dx[n][ci][v] (fp32 NCDHW) = scale * sum_tap sum_co W[co][ci][tap] * dz[n, v - (tap-1), co]
 *   dz: 16-bit NDHWC gradient of the conv output; W: fp32 (Cout,Cin,3,3,3), rounded to 16 bits like every other data-gradient operand.
 *   Cin == 1 and Cout in {8,16,32}: warp-level MMA kernel; any other Cin (Cout % 8 == 0): CUDA-core kernel.  Fixed summation order, no
 *   atomics.  partials (optional, then x = the NCDHW fp32 input is required): [N][P][Cin][2] = per-block (sum dx, sum dx*x),
 *   P = b200_input_dgrad_partials_count, for the GroupNorm backward of a first layer that starts with a GroupNorm.
 * b200_gn_bwd_apply_ncdhw_f32: out = scale * (A*dxhat + B*x + Cc), coef[N][C][3] = (A, B, Cc) from b200_gn_bwd_coeffs; out may alias dxhat.
 * b200_pointwise_dgrad_f32: dx[n][ci][v] (fp32 NCDHW) = scale * sum_co W[co][ci] * dy[n,v,co]  (W fp32 (Cout,Cin)). */
int b200_input_dgrad_partials_count(int N, int D, int H, int W, int Cin, int Cout);
int b200_input_dgrad_conv3(const void* dz, const float* W, int N, int D, int H, int Wd, int Cin, int Cout, float scale, const float* x,
                           float* dx, float* partials, b200_stream_t s);
int b200_gn_bwd_apply_ncdhw_f32(const float* dxhat, const float* x, const float* coef, int N, int C, long long voxels, float scale,
                                float* out, b200_stream_t s);
int b200_pointwise_dgrad_f32(const void* dy, const float* W, int N, long long voxels, int Cin, int Cout, float scale, float* dx,
                             b200_stream_t s);

/* ---- "virtual concat" decoder convolution: conv3(GN(cat(enc, nearest_up2x(b)))) without the upsampled / concatenated tensor
 * (replaces F.interpolate + torch.cat + SingleConv of Decoder.forward, buildingblocks.py:466-497, when the encoder feature is
 * exactly 2x the low-res one).  y = conv3_enc(enc) [+bias, +R, act, stats: b200_conv3_fwd with pmode | B200_PMODE_PHASE_BIAS,
 * residual = R] where R = b200_conv3_up_phase_fwd(b).  Layouts: wf_enc bf16 [n_w][27][Cout][C0]; wp bf16 [n_w][8 phases][8][Cout][C1];
 * biascls [n_w][64][Cout] with per-axis classes {0 low face, 1 interior even, 2 high face, 3 interior odd};
 * wd_enc bf16 [27][C0][Cout]; wd_up bf16 [64][C1][Cout]; Q fp32 [N][S][64][Cout][C1]; G fp32 [N][27][C0+C1][Cout]. */
int b200_gn_fold_upcat(const double* sums, const float* gamma, const float* beta, int G, double count, const float* W,
                       const float* conv_bias, int N, int C0, int C1, int Cout, void* wf_enc, void* wp, float* biascls, float* mean_rstd,
                       float* ab, b200_stream_t s);
int b200_conv3_up_supported(int N, int d, int h, int w, int C1, int Cout);
int b200_conv3_up_phase_fwd(const void* b, const void* wp, int n_w, int N, int d, int h, int w, int C1, int Cout, void* R, b200_stream_t s);
int b200_upcat_prep_dgrad_weights(const float* W, int C0, int C1, int Cout, void* wd_enc, void* wd_up, b200_stream_t s);
int b200_conv3_up_dgrad(const void* dz, const void* wd, int N, int d, int h, int w, int Cout, int C1, void* dxb, b200_stream_t s);
/* z-stacked version of the same (large low-res planes): parts = scratch for 4 partial gradients [4][N][d][h][w][C1] (16-bit) */
int b200_conv3_up_dgrad_zs_supported(int N, int d, int h, int w, int Cout, int C1);
int b200_conv3_up_dgrad_zs(const void* dz, const void* wd, int N, int d, int h, int w, int Cout, int C1, void* parts, void* dxb, b200_stream_t s);
int b200_conv3_up_wgrad_splits(int N, int d, int h, int w, int Cout, int C1);
int b200_conv3_up_wgrad(const void* dz, const void* b, int N, int d, int h, int w, int Cout, int C1, float* Q, b200_stream_t s);
int b200_upcat_assemble_wgrad(const float* G_enc, int S1, const float* Q, int S2, int N, int C0, int C1, int Cout, float* G,
                              b200_stream_t s);

/* ---- fused BCEDiceLoss on fp32 logits [N][C][V] (reference losses.py:187-201; SURVEY section 8(f) row f-3).
 * fwd: partials float [N*C][P][4] (P = b200_bce_dice_partials_count), loss float[1], coef float[1 + 2*C] = (1/count, (k1_c, k2_c)...);
 * bwd: dlogits = d loss / d logits (for an upstream gradient of 1) from the saved coefficients. */
int b200_bce_dice_partials_count(int N, int C, long long V);
int b200_bce_dice_fwd(const float* logits, const float* target, int N, int C, long long V, float alpha, float eps, float* partials,
                      float* loss, float* coef, b200_stream_t s);
int b200_bce_dice_bwd(const float* logits, const float* target, const float* coef, int N, int C, long long V, float* dlogits,
                      b200_stream_t s);

/* 1x1x1 conv on the tensor cores (C_in, C_out multiples of 16; bf16 input): the tcgen05 conv / wgrad kernels over a flat voxel list.
 * wq: bf16 [Cout][Cin] from b200_pointwise_prep_weights (transposed=1 gives the dgrad operand [Cin][Cout]); bias fp32 [Cout] or NULL;
 * partials [N][P][Cout][2] (P = b200_pointwise_tc_partials_count) or NULL; G [N][S][Cin][Cout] fp32 (S = ..._wgrad_splits). */
int b200_pointwise_prep_weights(const float* W, int Cin, int Cout, int transposed, void* wq, b200_stream_t s);
int b200_pointwise_tc_supported(int N, long long vox, int Cin, int Cout);
int b200_pointwise_tc_partials_count(int N, long long vox);
int b200_pointwise_tc_fwd(const void* x, const void* wq, const float* bias, int N, long long vox, int Cin, int Cout, void* y,
                          float* partials, b200_stream_t s);
int b200_pointwise_tc_wgrad_splits(int N, long long vox, int Cin, int Cout);
int b200_pointwise_tc_wgrad(const void* x, const void* dy, int N, long long vox, int Cin, int Cout, float* G, b200_stream_t s);
int b200_pointwise_wgrad_partials_count(int N, long long voxels);
int b200_pointwise_wgrad(const void* x, int x_is_f32, const void* dy, int N, long long voxels, int Cin, int Cout, float* partials,
                         b200_stream_t s);
/* ---- ConvTranspose3d(k3,s2,p1,bias=False) + nearest resize to the encoder size + sum-join
 * (TransposeConvUpsampling buildingblocks.py:617-664, Decoder._joining :493), built from the tensor-core 3x3x3 conv:
 *   conv_transpose3d(x, Wt) == conv3d(zero_insert(x), Wc, padding 1),  Wc[co][ci][k] = Wt[ci][co][26-k]  (Wt: (Cin,Cout,3,3,3)) */
int b200_zero_insert(const void* x, int N, int d, int h, int w, int C, void* xz /* [N,2d-1,2h-1,2w-1,C] */, b200_stream_t s);
int b200_subsample2_bwd(const void* dxz, const void* x, int N, int d, int h, int w, int C, int act, float slope, const void* gadd, void* out,
                        b200_stream_t s);
int b200_resize_add_partials_count(int N, int D, int H, int W, int C);
/* out[o] = enc[o] + T[nearest_src(o)], T on the (sd,sh,sw) grid; partials of out */
int b200_resize_add_fwd(const void* T, const void* enc, int N, int sd, int sh, int sw, int D, int H, int W, int C, void* out, float* partials,
                        b200_stream_t s);
/* dT[N,2d-1,2h-1,2w-1,C] = adjoint of the nearest resize applied to dout[N,D,H,W,C] */
int b200_deconv_gather(const void* dout, int N, int d, int h, int w, int D, int H, int W, int C, void* dT, b200_stream_t s);
/* to_conv=1: Wc[co][ci][k] = Wt[ci][co][26-k]; to_conv=0: dWt[ci][co][k] = dWc[co][ci][26-k] */
int b200_deconv_weight_permute(const float* src, int Cin, int Cout, int to_conv, float* dst, b200_stream_t s);

/* ---- the same transposed conv + join by OUTPUT PARITY PHASES (8x fewer MACs; used when the encoder feature is exactly twice the low-res
 * size): P[j] = T[j-1] on the (2d)^3 grid computed on the low-res lattice (27 (phase, tap) products, 8 accumulators per CTA), then
 * out[j] = enc[j] + P[max(j,1)] (= the nearest resize of the (2d-1)^3 grid).  Backward: gp = fold(g) (adjoint of j -> max(j,1)),
 * dx = 3x3x3 stride-2 convolution of gp, dWt[e] = sum_u gp[2u+e] (x) x[u].
 * wq bf16 [27][Cout][Cin] ((phase, tap) order), wd bf16 [27][Cin][Cout], Q fp32 [N][S][27][Cout][Cin] (S = ..._wgrad_splits). */
int b200_deconv_phase_supported(int N, int d, int h, int w, int Cin, int Cout);
int b200_deconv_phase_weights(const float* Wt, int Cin, int Cout, void* wq, void* wd, b200_stream_t s);
int b200_deconv_phase_fwd(const void* x, const void* wq, int N, int d, int h, int w, int Cin, int Cout, void* P, b200_stream_t s);
int b200_shift_add_fwd(const void* P, const void* enc, int N, int D, int H, int W, int C, void* out, float* partials, b200_stream_t s);
int b200_shift_fold_bwd(const void* g, int N, int D, int H, int W, int C, void* gp, b200_stream_t s);
int b200_deconv_phase_dgrad(const void* gp, const void* wd, int N, int d, int h, int w, int Cout, int Cin, void* dx, b200_stream_t s);
int b200_deconv_phase_wgrad_splits(int N, int d, int h, int w, int Cout, int Cin);
int b200_deconv_phase_wgrad(const void* gp, const void* x, int N, int d, int h, int w, int Cout, int Cin, float* Q, b200_stream_t s);
int b200_deconv_phase_wgrad_finalize(const float* Q, int rows, int Cin, int Cout, float* dWt, b200_stream_t s);

/* ---- scSE, reduction_ratio 1 (ChannelSpatialSELayer3D se.py:96-114; cSE :18-51, sSE :54-93) ----------------------------
 * gates: smean[N][C] = channel means (from the producer's partial sums), h = relu(W1 s + b1), g = sigmoid(W2 h + b2) */
int b200_se_gates_fwd(const double* sums, double count, const float* W1, const float* b1, const float* W2, const float* b2, int N, int C,
                      float* smean, float* h, float* g, b200_stream_t s);
int b200_scse_partials_count(int N, long long voxels, int C);
/* q[n,v] = sigmoid(ws . y[v,:] + bs[0]) (saved for backward); out = max(y*g, y*q); bs: device pointer to the 1-element conv bias */
int b200_scse_apply_fwd(const void* y, const float* g, const float* ws, const float* bs, int N, long long voxels, int C, void* out, float* q,
                        b200_stream_t s);
/* tmp = d out/d y without the channel-mean path; partials [N][P][C][2] = (d g, d ws per sample); dbs_part [N][P] */
int b200_scse_bwd1(const void* dout, const void* y, const float* g, const float* q, const float* ws, int N, long long voxels, int C, void* tmp,
                   float* partials, float* dbs_part, b200_stream_t s);
/* gate MLP backward; coef[N][C][3] = (1, 0, ds/V) feeds b200_gn_bwd_apply(tmp, y, coef) to finish d y. scratch: 2*N*C floats */
int b200_se_gates_bwd(const double* sums2, const float* smean, const float* h, const float* g, const float* W1, const float* W2, int N, int C,
                      double count, float* coef, float* dW1, float* db1, float* dW2, float* db2, float* dws, float* scratch, b200_stream_t s);

/* ---- sliding-window inference either side of the model (SURVEY section 8(f) rows f-1 / f-2) ------------------------------------
 * gather: out[C][pz][py][px] = reflect-padded vol[C][Z][Y][X] at (z0+z, y0+y, x0+x); (z0,y0,x0) = patch start minus halo, may be
 * negative / reach past the end by less than one volume size (datasets/utils.py:518-546 mirror_pad + hdf5.py:16-20). */
int b200_patch_gather_f32(const float* vol, int C, int Z, int Y, int X, int z0, int y0, int x0, int pz, int py, int px, float* out,
                          b200_stream_t s);
/* scatter: crop the halo (hz,hy,hx) off pred[C][pz][py][px] and write it at (z0,y0,x0) of out[C][Z][Y][X], but only the voxels
 * whose LAST covering patch is this one: owner_a[c] (device int[size_a]) == (iz,iy,ix) -- the reference's write order
 * (predictor.py:148-193, later patches overwrite earlier ones) evaluated analytically, so every voxel is written exactly once. */
int b200_patch_scatter_f32(const float* pred, int C, int pz, int py, int px, int hz, int hy, int hx, float* out, int Z, int Y, int X,
                           int z0, int y0, int x0, int iz, int iy, int ix, const int* owner_z, const int* owner_y, const int* owner_x,
                           b200_stream_t s);

/* ---- fused Adam over a flat fp32 buffer (create_optimizer utils.py:246-316 -> torch.optim.Adam, L2 weight decay in the gradient;
 * SURVEY section 8(f) row f-4).  bc1 = 1 - beta1^t, bc2 = 1 - beta2^t; g is read as g*grad_scale (1/world after a sum-allreduce). */
int b200_adam_step(float* p, const float* g, float* m, float* v, long long n, float lr, float beta1, float beta2, float eps, float wd,
                   float bc1, float bc2, float grad_scale, b200_stream_t s);

/* debug builds only (make DEBUG=1 -> -DB200_DEBUG): per-CTA wait-cycle counters of the halo kernel (16 x int64 per CTA); NULL
 * disables.  In a production build the counters are compiled out and this call is a no-op returning 1. */
int b200_set_debug_buffer(void* buf);

#ifdef __cplusplus
}
#endif
#endif /* B200UNET_H_ */
