/* az_stereo.h -- C ABI of libaz_stereo.so: the B200 (sm_100a) implementation of
 * ActiveZero's stereo-matching hot path.
 *
 * Convention (modelled on the reference's own raw-pointer launch convention,
 * /root/reference/utils/warp_ops.py:79-93: args = data_ptr()s + int dims,
 * stream = torch.cuda.current_stream().cuda_stream):
 *   - every pointer is a DEVICE pointer to a dense, contiguous NCHW / NCDHW
 *     float32 tensor unless the comment says otherwise;
 *   - `stream` is a cudaStream_t passed as void*; the call only enqueues work
 *     on it: it never allocates, never frees, never synchronises;
 *   - the caller owns every buffer (inputs, outputs, workspaces) and keeps it
 *     alive until the stream has passed the call;
 *   - the return value is a cudaError_t as int (0 = success); AZ_ERR_* (< 0)
 *     flags an argument the library rejects before launching anything;
 *   - stateless and re-entrant; one process per GPU.
 * All citations are relative to /root/reference.
 */
#ifndef AZ_STEREO_H
#define AZ_STEREO_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define AZ_ERR_BAD_ARG (-1)      /* null pointer / non-positive dim / unsupported size */
#define AZ_ERR_UNALIGNED (-2)    /* pointer not aligned as the fast path requires (never returned: falls back) */

/* Library / build identification: returns "az_stereo <ver> sm_100a". */
const char* az_version(void);
/* Human-readable text for a non-zero return value of any function below. */
const char* az_error_string(int code);

/* ---- a1/a2: concat cost volume -- nets/psmnet/psmnet.py:151-165 (= psmnet_3.py:149-163) ----
 * vol[b,c,i,y,x]   = L[b,c,y,x]      (x >= i, else 0),  c in [0,C)
 * vol[b,C+c,i,y,x] = R[b,c,y,x-i]    (x >= i, else 0)
 * L,R: [B,C,H,W]; vol: [B,2C,Dq,H,W].  Every element of vol is written (no memset needed). */
int az_concat_volume_fwd(const float* L, const float* R, float* vol,
                         int64_t B, int64_t C, int64_t H, int64_t W, int64_t Dq, void* stream);
/* Autograd of the slice assignments of psmnet.py:158-164 (atomic-free gather):
 * gL[b,c,y,x] = sum_{i<=min(x,Dq-1)} gvol[b,c,i,y,x];  gR[b,c,y,x] = sum_{i<Dq, x+i<W} gvol[b,C+c,i,y,x+i].
 * gL / gR may each be NULL (that half is skipped). */
int az_concat_volume_bwd(const float* gvol, float* gL, float* gR,
                         int64_t B, int64_t C, int64_t H, int64_t W, int64_t Dq, void* stream);

/* The same volume and gradient in torch.channels_last_3d memory order [B][Dq][H][W][2C] (SURVEY.md §8f rank 2:
 * the layout in which cuDNN's 3-D convolutions consume it without transposing; psmnet.py:165-168 is the consumer).
 * C must be a multiple of 4 and vol / gvol 16-byte aligned. */
int az_concat_volume_fwd_ndhwc(const float* L, const float* R, float* vol,
                               int64_t B, int64_t C, int64_t H, int64_t W, int64_t Dq, void* stream);
int az_concat_volume_bwd_ndhwc(const float* gvol, float* gL, float* gR,
                               int64_t B, int64_t C, int64_t H, int64_t W, int64_t Dq, void* stream);

/* The same volume and gradient with 16-bit features (what torch.autocast's convolutions consume).  Every pointer is
 * a device pointer to bf16 or fp16 elements; L, R, gL, gR, vol, gvol all have the features' dtype.
 * Forward: vol is the formula of az_concat_volume_fwd applied to the 2-byte elements (a copy: exact, and the same
 *   for both dtypes, so it takes no dtype code).
 * Backward: gL / gR are the sums of az_concat_volume_bwd taken in fp32 over the upcast elements of gvol, in
 *   ascending i, then rounded ONCE to the dtype, to nearest even:  gL = RNE16(sum_i float(gvol[..,i,..])).
 *   This equals az_concat_volume_bwd on gvol.float() followed by .to(dtype), bit for bit.  gL / gR may each be NULL.
 * channels_last != 0: vol / gvol are in torch.channels_last_3d memory order [B][Dq][H][W][2C]; C must then be a
 *   multiple of 8 and vol / gvol 16-byte aligned (else AZ_ERR_BAD_ARG).  channels_last == 0: NCDHW, any C. */
#define AZ_DTYPE_BF16 1
#define AZ_DTYPE_F16 2
int az_concat_volume_fwd_16(const void* L, const void* R, void* vol,
                            int64_t B, int64_t C, int64_t H, int64_t W, int64_t Dq, int channels_last, void* stream);
int az_concat_volume_bwd_16(const void* gvol, void* gL, void* gR,
                            int64_t B, int64_t C, int64_t H, int64_t W, int64_t Dq, int dtype, int channels_last,
                            void* stream);

/* ---- SURVEY.md §8f rank 2, implicit clause: the first 3-D convolution of the aggregation with the volume left
 *      implicit -- nets/psmnet/psmnet.py:151-168 (volume + dres0[0] = Conv3d(64,32,3,1,1,bias=False)), psmnet_submodule.py:44-56.
 * out[b,co,d,y,x] = sum_{ci,kd,ky,kx} weight[co,ci,kd,ky,kx] * vol[b,ci,d+kd-1,y+ky-1,x+kx-1] (zero padding) with vol
 * the concat volume of az_concat_volume_fwd, never materialised: tcgen05 TF32 implicit GEMM, fp32 accumulation in
 * tensor memory.  L,R: [B,32,H,W]; out: [B,32,Dq,H,W]; wpacked: AZ_VOLUME_CONV0_PACKED_FLOATS (= 27*3072) floats produced ONCE per weight tensor by
 * az_volume_conv0_pack from the Conv3d weight [32,64,3,3,3]; scale/shift: float[32] or both NULL (an eval-mode
 * BatchNorm folded into the epilogue: out*scale+shift), relu != 0 applies max(.,0) last. */
#define AZ_VOLUME_CONV0_PACKED_FLOATS (27 * 3072)
int az_volume_conv0_pack(const float* weight, float* wpacked, void* stream);
int az_volume_conv0_fwd(const float* L, const float* R, const float* wpacked, const float* scale, const float* shift,
                        float* out, int64_t B, int64_t C, int64_t H, int64_t W, int64_t Dq, int relu, void* stream);
/* The same convolution with 16-bit features and output (dtype AZ_DTYPE_BF16 or AZ_DTYPE_F16), as torch.autocast runs
 * it: L, R: [B,32,H,W] and out: [B,32,Dq,H,W] of that dtype.  az_volume_conv0_pack_16 rounds each weight to the dtype
 * (RNE) before the TF32 packing -- what autocast does to cuDNN's weight; use its wpacked with the same dtype.  The
 * features are converted to fp32 at staging, which TF32 represents exactly, so the MMAs stay TF32 with fp32
 * accumulation; scale / shift (float[32] or both NULL) and the ReLU are applied in fp32, and each output is rounded
 * ONCE, to nearest even, at the store:  out = RNE16(relu(conv * scale + shift)). */
int az_volume_conv0_pack_16(const float* weight, float* wpacked, int dtype, void* stream);
int az_volume_conv0_fwd_16(const void* L, const void* R, const float* wpacked, const float* scale, const float* shift,
                           void* out, int64_t B, int64_t C, int64_t H, int64_t W, int64_t Dq, int relu, int dtype,
                           void* stream);
/* Backward of the raw convolution above (no scale/shift, no ReLU), without the volume or its gradient.  With
 * gout = dLoss/d out [B,32,Dq,H,W], Wl = weight[:, :32], Wr = weight[:, 32:] and, for each tap (kd,kx),
 * lo = max(0,1-kd), hi = min(Dq-1,Dq-kd):
 *   A[kd,kx][b,o,y,x] = sum_{d=lo}^{min(x+kx-kd,hi)} gout[b,o,d,y,x]
 *   Z[kd,kx][b,o,y,u] = sum_{d=lo}^{hi} gout[b,o,d,y,u+d+kd-kx]  over the d with 0 <= u+d+kd-kx <= min(W-1,W-kx)
 *   gL[b,c,y',x'] = sum_{o,kd,ky,kx} Wl[o,c,kd,ky,kx] * A[kd,kx][b,o,y'-ky+1,x'-kx+1]   (zero outside the image)
 *   gR[b,c,y',u]  = sum_{o,kd,ky,kx} Wr[o,c,kd,ky,kx] * Z[kd,kx][b,o,y'-ky+1,u]
 *   gW[o,c,kd,ky,kx]    = sum_{b,y',x'} A[kd,kx][b,o,y'-ky+1,x'-kx+1] * L[b,c,y',x']
 *   gW[o,32+c,kd,ky,kx] = sum_{b,y',u}  Z[kd,kx][b,o,y'-ky+1,u]       * R[b,c,y',u]
 * fp32 on the CUDA cores, fixed summation order, atomic-free (bit-identical run to run).  weight: the plain Conv3d
 * weight [32,64,3,3,3] (not the packed copy); L,R,gL,gR: [B,32,H,W]; gW: [32,64,3,3,3]; each of gL, gR, gW may be
 * NULL (that part is skipped) and all three are fully written.  C must be 32; any Dq.
 * workspace: az_volume_conv0_bwd_workspace_bytes(B,H,W,Dq) bytes, 16-byte aligned (holds the 18 planes A, Z). */
int64_t az_volume_conv0_bwd_workspace_bytes(int64_t B, int64_t H, int64_t W, int64_t Dq);
int az_volume_conv0_bwd(const float* gout, const float* L, const float* R, const float* weight,
                        float* gL, float* gR, float* gW, void* workspace,
                        int64_t B, int64_t C, int64_t H, int64_t W, int64_t Dq, void* stream);
/* The same backward with 16-bit tensors (dtype AZ_DTYPE_BF16 or AZ_DTYPE_F16): gout, L, R, gL and gR have that dtype.
 * weight_dtype is 0 (weight and gW are float32: autocast's fp32 master weight) or equal to dtype (weight and gW have
 * that dtype: a converted model); any other code, or C != 32, gives AZ_ERR_BAD_ARG.  Each 16-bit value is widened
 * exactly where it is read; an fp32 weight is rounded to dtype (RNE) before dfeat uses it, as az_volume_conv0_pack_16
 * and autocast round it.  The workspace (same size, fp32 planes and partials), every accumulator and every summation
 * order are az_volume_conv0_bwd's, and each 16-bit result is rounded ONCE, to nearest even, at its store:
 *   gL, gR = az_volume_conv0_bwd(gout.float(), L.float(), R.float(), w16.float()).to(dtype)   (w16 = weight rounded to dtype)
 *   gW     = az_volume_conv0_bwd(...)'s gW (which does not depend on the weight), .to(dtype) when weight_dtype == dtype
 * bit for bit.  fp16 results too large for the format become +-inf, as .to(torch.float16) makes them. */
int az_volume_conv0_bwd_16(const void* gout, const void* L, const void* R, const void* weight,
                           void* gL, void* gR, void* gW, void* workspace,
                           int64_t B, int64_t C, int64_t H, int64_t W, int64_t Dq,
                           int dtype, int weight_dtype, void* stream);

/* ---- a3: group-wise correlation volume -- NOT IN THE REFERENCE (SURVEY.md fact 1; parity unpinned) ----
 * vol[b,g,i,y,x] = (1/(C/G)) * sum_{c in group g} L[b,c,y,x]*R[b,c,y,x-i]  (x >= i, else 0); vol: [B,G,Dq,H,W]. */
int az_gwc_volume_fwd(const float* L, const float* R, float* vol,
                      int64_t B, int64_t C, int64_t H, int64_t W, int64_t Dq, int64_t G, void* stream);
int az_gwc_volume_bwd(const float* gvol, const float* L, const float* R, float* gL, float* gR,
                      int64_t B, int64_t C, int64_t H, int64_t W, int64_t Dq, int64_t G, void* stream);

/* ---- a4/a5: soft-argmin = F.softmax(cost,1) + DisparityRegression --
 *      nets/psmnet/psmnet.py:200-201,204-205,212-217 + nets/psmnet/psmnet_submodule.py:80-89 ----
 * disp[b,0,y,x] = sum_d d * softmax_d(cost[b,:,y,x]).  cost: [B,D,H,W] LOGITS; disp: [B,1,H,W];
 * lse (optional, may be NULL): [B,2,H,W] activation saved for the backward -- for each pixel the max logit m
 * (first B*H*W floats) and log2(sum_d 2^((cost_d - m)*log2(e))) (next B*H*W floats).  H*W*B must keep both
 * halves 16-byte aligned for the vector path (it falls back to scalar otherwise). */
int az_soft_argmin_fwd(const float* cost, float* disp, float* lse,
                       int64_t B, int64_t D, int64_t H, int64_t W, void* stream);
/* gcost[b,d,y,x] = softmax_d * (d - disp) * gdisp[b,0,y,x], softmax_d = 2^((cost_d - m)*log2(e) - log2sum) */
int az_soft_argmin_bwd(const float* cost, const float* disp, const float* lse, const float* gdisp, float* gcost,
                       int64_t B, int64_t D, int64_t H, int64_t W, void* stream);
/* The same operator with 16-bit logits: cost and gcost are bf16 or fp16 (dtype AZ_DTYPE_BF16 or AZ_DTYPE_F16, else
 * AZ_ERR_BAD_ARG); disp, lse and gdisp stay float32.
 * Forward: each logit is widened exactly (both formats fit inside fp32) and goes through the fp32 kernels' arithmetic
 *   unchanged, the kernel picked by the fp32 rule on the shape alone (H*W % 4 == 0 or not), never by the alignment of
 *   cost: disp and lse equal az_soft_argmin_fwd on cost.float() (a fresh, aligned tensor), bit for bit, for any
 *   element offset of cost.  disp stays fp32 on purpose (a bf16 disparity has a spacing of 0.5 px above 128 px).
 * Backward: the gradient is formed in fp32 exactly as az_soft_argmin_bwd forms it and rounded ONCE, to nearest even:
 *   gcost = RNE16(az_soft_argmin_bwd(cost.float(), ...)), bit for bit.
 * The AZ_SA_FWD developer knob applies to the fp32 entry point only. */
int az_soft_argmin_fwd_16(const void* cost, float* disp, float* lse,
                          int64_t B, int64_t D, int64_t H, int64_t W, int dtype, void* stream);
int az_soft_argmin_bwd_16(const void* cost, const float* disp, const float* lse, const float* gdisp, void* gcost,
                          int64_t B, int64_t D, int64_t H, int64_t W, int dtype, void* stream);

/* ---- SURVEY.md §8f rank 1: trilinear upsample fused into soft-argmin --
 *      nets/psmnet/psmnet.py:186-197,208-211 (F.interpolate(cost,(D,4H,4W),'trilinear',align_corners=False))
 *      followed by the soft-argmin above, without materialising the [B,D,H,W] logits.
 * lowres: [B,1,Dq,Hq,Wq] (= [B,Dq,Hq,Wq]); disp: [B,1,H,W]; stats (optional): [B,2,H,W] saved for the backward;
 * (D,H,W) is the output size (upsampling only: D >= Dq, H >= Hq, W >= Wq). */
int az_upsample_soft_argmin_fwd(const float* lowres, float* disp, float* stats,
                                int64_t B, int64_t Dq, int64_t Hq, int64_t Wq,
                                int64_t D, int64_t H, int64_t W, void* stream);
/* glow: [B,1,Dq,Hq,Wq], fully written (deterministic gather, no atomics);
 * workspace: az_upsample_soft_argmin_workspace_bytes(B,Dq,H,W,Wq) bytes. */
int64_t az_upsample_soft_argmin_workspace_bytes(int64_t B, int64_t Dq, int64_t H, int64_t W, int64_t Wq);
int az_upsample_soft_argmin_bwd(const float* lowres, const float* disp, const float* stats, const float* gdisp,
                                float* glow, void* workspace, int64_t B, int64_t Dq, int64_t Hq, int64_t Wq,
                                int64_t D, int64_t H, int64_t W, void* stream);
/* The same operator with 16-bit low-resolution logits: lowres and glow are bf16 or fp16 (dtype AZ_DTYPE_BF16 or
 * AZ_DTYPE_F16, else AZ_ERR_BAD_ARG); disp, stats, gdisp and the workspace (same size, fp32 planes) stay float32.
 * The logits are widened exactly when they are staged, and every instruction after that, the kernel selection included
 * (as at the AZ_USA_FWD default), is the fp32 operator's: disp and stats equal az_upsample_soft_argmin_fwd on
 * lowres.float(), and glow = RNE16(az_upsample_soft_argmin_bwd(lowres.float(), ...)), bit for bit (the fp32 sums of
 * the last reduction are rounded once, to nearest even, at the store). */
int az_upsample_soft_argmin_fwd_16(const void* lowres, float* disp, float* stats, int64_t B, int64_t Dq, int64_t Hq,
                                   int64_t Wq, int64_t D, int64_t H, int64_t W, int dtype, void* stream);
int az_upsample_soft_argmin_bwd_16(const void* lowres, const float* disp, const float* stats, const float* gdisp,
                                   void* glow, void* workspace, int64_t B, int64_t Dq, int64_t Hq, int64_t Wq,
                                   int64_t D, int64_t H, int64_t W, int dtype, void* stream);

/* ---- a6: bilinear disparity warp -- utils/reprojection.py:13-35 (apply_disparity) ----
 * out[b,c,i,j] = bilinear2D(img[b,c]; xs, ys), zeros padding, align_corners=False, with the reference's
 * fp32 op order: f = lin_x[j] + disp/W; g = 2f-1; xs = ((g+1)*W-1)/2 (same for y with lin_y[i], H).
 * lin_x [W], lin_y [H]: DEVICE copies of torch.linspace(0,1,n) (reprojection.py:18-24).
 * img,out: [B,C,H,W]; disp: [B,1,H,W] (already signed: the reference passes -pred_disp_l). */
int az_warp_fwd(const float* img, const float* disp, const float* lin_x, const float* lin_y, float* out,
                int64_t B, int64_t C, int64_t H, int64_t W, void* stream);
/* gdisp [B,1,H,W] and gimg [B,C,H,W] (each may be NULL) are fully WRITTEN (no zero-fill by the caller).  The image
 * gradient is a deterministic gather per image row with order-independent fixed-point accumulation; torch's
 * grid_sampler backward uses float atomics. */
int az_warp_bwd(const float* img, const float* disp, const float* lin_x, const float* lin_y,
                const float* gout, float* gimg, float* gdisp,
                int64_t B, int64_t C, int64_t H, int64_t W, void* stream);

/* ---- a7/a8: fused warp + masked-MSE reprojection loss --
 *      utils/reprojection.py:81-96 (ps = 1), :99-127 (patch, ps odd) ----
 * loss = sum_{b,k,i,j} m[b,i,j] * (Wu - Lu)^2 / (K * sum m),  K = C*ps*ps, with Lu/Ru the zero-padded
 * ps x ps unfold of tgt/src and Wu = apply_disparity(Ru, sign*disp) (reprojection.py:102-118).
 *   tgt, src : [B,C,H,W] (tgt = image compared against, src = image that is warped)
 *   disp     : [B,1,H,W];  sign = -1 reproduces apply_disparity(src, -disp), +1 apply_disparity(src, disp)
 *   mask     : [B,1,H,W] uint8 (0/1) or NULL (= all ones)
 *   warped   : [B,C,H,W] or NULL; for ps == 1 the warped image (reprojection.py:89); for ps > 1 the Fold image of
 *              reprojection.py:120-125 (what az_patch_fold computes), produced in the same pass as the loss
 *   gpre     : [B,1,H,W] or NULL; m * sum_k (Wu-Lu) * dWu/dxs, consumed by az_reproj_loss_bwd
 *   loss_out : float[1];  stats: double[2] = {sum of squares, sum m} (device), kept for the backward
 *   workspace: az_reproj_workspace_bytes(B,H) bytes, 16-byte aligned
 * Empty mask => loss = NaN, as the reference (F.mse_loss of an empty selection). */
int64_t az_reproj_workspace_bytes(int64_t B, int64_t H);
int az_reproj_loss_fwd(const float* tgt, const float* src, const float* disp, float sign, const uint8_t* mask,
                       const float* lin_x, const float* lin_y, int64_t ps,
                       float* warped, float* gpre, float* loss_out, double* stats, void* workspace,
                       int64_t B, int64_t C, int64_t H, int64_t W, void* stream);
/* gdisp[b,0,i,j] = gloss[0] * sign * 2/(K*sum m) * gpre[b,0,i,j] */
int az_reproj_loss_bwd(const float* gpre, const double* stats, const float* gloss, float sign,
                       float* gdisp, int64_t B, int64_t C, int64_t H, int64_t W, int64_t ps, void* stream);
/* Image gradients of the same loss (the reference differentiates its "feature or image" inputs too).  The
 * arguments tgt .. ps and the shapes are the forward's; stats and gloss as for az_reproj_loss_bwd.  With
 * r_k(i,j) = Wu_k(i,j) - Lu_k(i,j), p = (ps-1)/2 and rho_k(i,j) = gloss * 2 * m(i,j) * r_k(i,j) / (K * sum m):
 *   gtgt[b,c,y,x] = - sum_{ky,kx} rho_{(c,ky,kx)}(y+p-ky, x+p-kx)   over in-image (i,j)  (adjoint of the Unfold)
 *   gsrc[b,c,Y,X] = + sum rho_k(i,j) * wy_a(i) * wx_b(i,j)  over the bilinear corners (a,b) of the forward's sample
 *                   position that are valid in the unfolded plane, with Y = y0(i)+a+ky-p, X = x0(i,j)+b+kx-p inside
 *                   the image (adjoint of the warp of the unfolded planes)
 * The residuals are recomputed from tgt, src, disp and mask (no [B,K,H,W] intermediate, no workspace, no host
 * synchronisation).  gtgt and gsrc are [B,C,H,W] or NULL; every element of a non-NULL one is written exactly once
 * (no zero-fill by the caller) and nothing else is written.  Deterministic: fixed-order sums and order-independent
 * 64-bit fixed-point accumulation, no float atomics; two calls give bit-identical results.  sum m == 0 (empty mask)
 * gives exact zeros (the reference's gradient of an empty selection).  A non-finite input read by a row of gsrc
 * makes that row NaN.  Shapes: those of az_reproj_loss_fwd, any odd ps up to 4095.  Returns 0 at once when both
 * outputs are NULL. */
int az_reproj_loss_img_bwd(const float* tgt, const float* src, const float* disp, float sign, const uint8_t* mask,
                           const float* lin_x, const float* lin_y, int64_t ps, const double* stats,
                           const float* gloss, float* gtgt, float* gsrc,
                           int64_t B, int64_t C, int64_t H, int64_t W, void* stream);
/* Visualisation output of get_reproj_error_patch: Fold (overlap-sum) of the warped unfolded planes,
 * cropped by (ps-1)/2 (reprojection.py:120-125).  vis: [B,C,H,W]. */
int az_patch_fold(const float* src, const float* disp, float sign, const float* lin_x, const float* lin_y,
                  int64_t ps, float* vis, int64_t B, int64_t C, int64_t H, int64_t W, void* stream);

/* ---- a9: bilinear rescaling of the multi-scale loss -- utils/reprojection.py:153-158 ----
 * One launch for the four F.interpolate(..., scale_factor=r, mode="bilinear") calls of one scale:
 * tgt_o, src_o: [B,C,Ho,Wo]; disp_o = interpolate(disp) * disp_mul: [B,1,Ho,Wo] (disp may be NULL);
 * mask_o = interpolate(mask.float()).bool(): [B,1,Ho,Wo] uint8 (mask NULL = all ones; mask_o may be NULL).
 * scale_h, scale_w = 1/r as float32 (what torch passes to upsample_bilinear2d when scale_factor is given);
 * Ho = floor(H*r), Wo = floor(W*r). */
int az_bilinear_rescale_fwd(const float* tgt, const float* src, const float* disp, const uint8_t* mask,
                            float* tgt_o, float* src_o, float* disp_o, uint8_t* mask_o,
                            int64_t B, int64_t C, int64_t H, int64_t W, int64_t Ho, int64_t Wo,
                            float scale_h, float scale_w, float disp_mul, void* stream);
/* gin[B,1,H,W] = disp_mul * (adjoint of the bilinear downscaling) gout[B,1,Ho,Wo]; deterministic gather. */
int az_bilinear_rescale_bwd(const float* gout, float* gin, int64_t B, int64_t H, int64_t W, int64_t Ho, int64_t Wo,
                            float scale_h, float scale_w, float disp_mul, void* stream);

/* ---- a10: integer scatter warp -- utils/warp_ops.py:20-47 kernels + :55-95 host ----
 * dst[n,c,y,j+disp[n,0,y,j]] = src[n,c,y,j]; among sources landing on one column the largest |disp| wins
 * (== the reference kernels' last-writer order); holes = 0.  src,dst: [N,C,H,W] float32; disp: [N,1,H,W] int32.
 * sign_flags: int32[1] device, zero-filled by the caller; bit0 set if any disp > 0, bit1 if any disp < 0
 * (the reference asserts the disparities do not mix signs, warp_ops.py:73-77). May be NULL. */
int az_scatter_warp(const float* src, const int32_t* disp, float* dst, int32_t* sign_flags,
                    int64_t N, int64_t C, int64_t H, int64_t W, void* stream);

/* The trainer's ground-truth chain around a10 in one launch -- /root/reference/train.py:255-272 (test.py:109-110):
 *   r   = F.interpolate(disp2x, scale_factor=0.5, mode="nearest")        (source pixel (2y, 2j); H = H2/2, W = W2/2)
 *   out = apply_disparity_cu(r, r.type(torch.int))                       (the payload is the disparity itself)
 *   mask = (out < max_disp) * (out > 0)                                  (train.py:272)
 * disp2x: [N,1,H2,W2] float32; disp_out: [N,1,H,W] float32; mask_out: [N,1,H,W] uint8 (0/1) or NULL;
 * sign_flags as in az_scatter_warp. */
int az_scatter_warp_gt(const float* disp2x, float* disp_out, uint8_t* mask_out, int32_t* sign_flags,
                       float max_disp, int64_t N, int64_t H2, int64_t W2, void* stream);

/* ---- a11: temporal IR pattern -- tools/temporal_ir.py:35-40, 93-114 ----
 * frames: [B,T,H,W] uint8 -> pattern [B,H,W] float32 in {0,1}: per-pixel least-squares slope over t,
 * |fit[T-1]-fit[0]|/255, per-image min-max normalise, minus ks x ks box blur (BORDER_REFLECT_101),
 * > threshold.  Evaluated in exact integer arithmetic (the reference's float64 chain reduces to integer sums and one
 * comparison, csrc/temporal_ir.cu); T <= 4096.  workspace: az_temporal_ir_workspace_bytes(B,H,W) bytes, 16-byte aligned. */
int64_t az_temporal_ir_workspace_bytes(int64_t B, int64_t H, int64_t W);
int az_temporal_ir(const uint8_t* frames, float* pattern, void* workspace,
                   int64_t B, int64_t T, int64_t H, int64_t W, int64_t ks, double threshold, void* stream);

/* ---- a12: local contrast normalisation -- utils/reprojection.py:175-200 ----
 * image: [B,Cin,H,W], only channel 0 is used (:184-185); zero-padded ks x ks window mean and population
 * std; normed = (img - mean)/(std + eps).  normed, std: [B,1,H,W]. */
int az_local_contrast_norm(const float* image, float* normed, float* std, int64_t B, int64_t Cin,
                           int64_t H, int64_t W, int64_t ks, float eps, void* stream);

/* ---- SURVEY.md §8f rank 3: sim-domain IR pattern -- datasets/dataset_utils.py:12-17 (get_ir_pattern, ks = 0)
 *      and :33-46 (get_smoothed_ir_pattern2, ks > 0: minus the cv2 INTER_AREA down(//ks)-then-up resampling) ----
 * img_ir, img_no_ir: [B,H,W], uint8 (is_u8 != 0; divided by 255 in float64 as the reference's loader does) or
 * float64 (is_u8 == 0); pattern: [B,H,W] float32 in {0,1}; float64 arithmetic in OpenCV's summation order.
 * workspace: az_sim_ir_pattern_workspace_bytes(B,H,W,ks) bytes. */
int64_t az_sim_ir_pattern_workspace_bytes(int64_t B, int64_t H, int64_t W, int64_t ks);
int az_sim_ir_pattern(const void* img_ir, const void* img_no_ir, int is_u8, float* pattern, void* workspace,
                      int64_t B, int64_t H, int64_t W, int64_t ks, double threshold, void* stream);

/* ---- SURVEY.md §8f rank 4: fused error metrics -- utils/cascade_metrics.py:16-57 (compute_err_metric) ----
 * One pass + one 64-byte read instead of seven boolean gathers with .item() syncs.
 * disp_gt, depth_gt, disp_pred: [B,1,H,W]; depth_pred: [B,1,H,W] or NULL (then focal_length*baseline/disp_pred
 * with focal_length, baseline: float[B]); mask: [B,1,H,W] uint8.
 * out: double[8] (device) = { n, sum|ddisp|, #(|ddisp|>1), #(|ddisp|>2), sum clip(|dz*1000|,0,100),
 *                             #(|dz|>2e-3), #(|dz|>4e-3), #(|dz|>8e-3) };
 * workspace: az_error_metrics_workspace_bytes(B,H,W) bytes. */
int64_t az_error_metrics_workspace_bytes(int64_t B, int64_t H, int64_t W);
int az_error_metrics(const float* disp_gt, const float* depth_gt, const float* disp_pred, const float* depth_pred,
                     const float* focal_length, const float* baseline, const uint8_t* mask, double* out,
                     void* workspace, int64_t B, int64_t H, int64_t W, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* AZ_STEREO_H */
