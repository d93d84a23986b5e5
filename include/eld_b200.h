/* eld_b200.h - C ABI of the B200-native ELD hot path (libeld_b200.so).
 *
 * The reference (Vandermode/ELD) has no FFI layer: its seams are Python duck-typed protocols
 * (SURVEY.md 8b).  This header is what a binding for that seam would call; every entry point
 * names the reference interface it replaces (file:line relative to the reference root).
 *
 * Conventions
 *   - every function returns 0 on success or a negative ELD_E* code; eld_last_error() returns a
 *     thread-local, NUL-terminated description of the last failure on the calling thread;
 *   - the caller owns ALL buffers (device pointers normally come from torch tensors); the library
 *     never frees caller memory and never synchronises the device unless documented;
 *   - `stream` is a cudaStream_t passed as void* (so that this header needs no CUDA include);
 *   - no CPU fallback: without a CUDA device every compute entry point fails with ELD_E_CUDA.
 *   - plain pointers and sizes only - no torch types.
 */
#ifndef ELD_B200_H
#define ELD_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define ELD_OK            0
#define ELD_E_ARG        -1   /* bad argument (null pointer, negative size, unsupported shape) */
#define ELD_E_CUDA       -2   /* CUDA runtime / driver error (text in eld_last_error)          */
#define ELD_E_UNSUPPORTED -3  /* valid request the library does not implement                   */
#define ELD_E_WORKSPACE  -4   /* caller workspace too small                                     */

typedef struct eld_ctx eld_ctx;

/* ABI version of this header; eld_abi_version() must return it. */
#define ELD_ABI_VERSION 1
int         eld_abi_version(void);
const char* eld_last_error(void);

/* One context per (process, device).  Holds the SM count, the TMA encode entry point and cached
 * tensor maps.  Thread-compatible: distinct ctx/stream pairs may be used concurrently. */
int  eld_ctx_create(int device, eld_ctx** out);
void eld_ctx_destroy(eld_ctx* ctx);

/* ------------------------------------------------------------------------------------------------
 * Noise formation model.  Replaces NoiseModelBase.__call__ (noise.py:149-170) + the clip in
 * SynDataset.__getitem__ (dataset/sid_dataset.py:277) + RawPacker.pack_raw_bayer (noise.py:10-20),
 * batched over frames, on the GPU.
 *
 * model_mask bits select the terms; the first three are the reference's released baselines
 * (substring match on the model string, noise.py:158-166), the rest are the paper's full model,
 * which the reference does NOT ship (README.md:41, noise.py:173) - "parity unpinned".
 */
#define ELD_NOISE_P  0x01u  /* 'P'  Poisson shot noise:            z = Poisson(x/K)*K        noise.py:158-159 */
#define ELD_NOISE_p  0x02u  /* 'p'  heteroscedastic Gaussian shot: z = x + n*sqrt(max(Kx,1e-10)) noise.py:160-161 */
#define ELD_NOISE_g  0x04u  /* 'g'  Gaussian read noise:           z += n*max(g_scale,1e-10) noise.py:165-166 */
#define ELD_NOISE_G  0x08u  /* Tukey-lambda read noise  z += TL(G_lambda)*G_scale   [paper-restated] */
#define ELD_NOISE_B  0x10u  /* colour bias              z += color_bias[c]          [paper-restated] */
#define ELD_NOISE_R  0x20u  /* row (banding) noise      z += N(0,R_scale) per SENSOR row [paper-restated] */
#define ELD_NOISE_U  0x40u  /* quantisation             z += U(-q/2, q/2)           [paper-restated] */

/* Per-frame scalars = the tuple NoiseModel._sample_params() returns (noise.py:225) extended with
 * the calibrated-but-unused fields of camera_params/release/ *.npy (SURVEY F2).  Units: DN. */
typedef struct eld_noise_params {
    float K;             /* system gain                                  */
    float g_scale;       /* Gaussian read sigma                          */
    float G_scale;       /* Tukey-lambda scale                           */
    float G_lambda;      /* Tukey-lambda shape                           */
    float R_scale;       /* row-noise sigma                              */
    float q_step;        /* quantisation step                            */
    float saturation;    /* 16383-800 = 15583 (noise.py:205)             */
    float ratio;         /* exposure ratio U(100,300) (noise.py:223)     */
    float color_bias[4]; /* per packed channel (R,G1,B,G2)               */
} eld_noise_params;      /* 48 bytes, no padding */

/* Random stream (identical in the CUDA kernel and in oracle/eld_oracle.c):
 *   Philox4x32-10, key = (seed_lo, seed_hi), counter = (a, (domain<<16)|(c<<8)|d, frame_lo, frame_hi)
 *   with frame = frame_id0 + n the GLOBAL frame id - so the synthetic stream does not depend on
 *   how frames are sharded over GPUs.  See DESIGN.md "random stream".  Normals are Box-Muller on 23-bit
 *   uniforms: |n| <= 5.77 (numpy's polar method is unbounded; the truncated tail has probability 8e-9 per draw).
 *
 * clean/noisy: packed float32 [n][4][h][w] (the layout NoiseModelBase.__call__ receives, SURVEY F3).
 * params: HOST pointer to n entries (copied into the launch; no device sync).
 * clip01 != 0 applies min(max(z,0),1) (sid_dataset.py:277).  clean == noisy (in place) is allowed. */
int eld_noise_packed(eld_ctx* ctx, const float* clean, float* noisy, int n, int h, int w,
                     const eld_noise_params* params, uint32_t model_mask,
                     uint64_t seed, uint64_t frame_id0, int clip01, void* stream);

/* Same model fed by the un-packed Bayer mosaic: fuses RawPacker.pack_raw_bayer (noise.py:10-20,
 * plane order RGBG = (0,0),(0,1),(1,1),(1,0)), the LMDB de-quantisation clip(x/65535,0,1)
 * (dataset/lmdb_dataset.py:38-39) and the noise model.  mosaic: [n][H][W], H and W even;
 * in_dtype ELD_DT_U16 or ELD_DT_F32; y = (m-black)/(white-black).  Writes noisy [n][4][H/2][W/2]
 * and, if clean_out != NULL, the packed clean frame (the training target). */
#define ELD_DT_U16 0
#define ELD_DT_F32 1
#define ELD_DT_BF16 2
int eld_noise_mosaic(eld_ctx* ctx, const void* mosaic, int in_dtype, float black, float white,
                     float* noisy, float* clean_out, int n, int H, int W,
                     const eld_noise_params* params, uint32_t model_mask,
                     uint64_t seed, uint64_t frame_id0, int clip01, void* stream);

/* The LMDB wire format as input (util/lmdb_data.py:184-228, dataset/lmdb_dataset.py:24-39): packed uint16
 * [n][4][h][w], y = clip(v * scale, 0, 1) with scale = 1/65535; only 2 bytes per pixel cross PCIe.  Writes noisy
 * and, if clean_out != NULL, the de-quantised clean frame (the training target).  w % 4 == 0. */
int eld_noise_packed_u16(eld_ctx* ctx, const uint16_t* clean_u16, float scale, float* noisy, float* clean_out,
                         int n, int h, int w, const eld_noise_params* params, uint32_t model_mask,
                         uint64_t seed, uint64_t frame_id0, int clip01, void* stream);

/* Noise fused with ELDTrainDataset's augmentation (dataset/sid_dataset.py:340-356): three independent coin flips per
 * frame - flip rows (np.flip axis 1), flip columns (axis 2), transpose (0,2,1) - applied in that order to BOTH the
 * noisy input and the clean target, then the clip.  The noise of a pixel is keyed by its SOURCE position, so
 *   noisy = aug(eld_noise_packed(clean)),  target_out = aug(clean)   bit for bit, in one pass over the frame.
 * aug_flags: HOST array, one byte per frame: bit 0 rows, bit 1 columns, bit 2 transpose (needs h == w).
 * target_out may be NULL.  Not in place.  w % 4 == 0, 16-byte aligned buffers. */
#define ELD_AUG_FLIP_H     1u
#define ELD_AUG_FLIP_W     2u
#define ELD_AUG_TRANSPOSE  4u
int eld_noise_packed_aug(eld_ctx* ctx, const float* clean, float* noisy, float* target_out, int n, int h, int w,
                         const eld_noise_params* params, uint32_t model_mask, uint64_t seed, uint64_t frame_id0,
                         int clip01, const uint8_t* aug_flags, void* stream);

/* ------------------------------------------------------------------------------------------------
 * Raw -> sRGB rendering of the `--stage_in srgb` branch (train_syn.py:55-58): replaces util/process.py:51-68
 * `process` - apply_gains (:15-19), clip, binning RGBG->RGB (:41-48), apply_ccms (:22-31), clip,
 * gamma_compression (:34-39) or camera_response_function (:71-84) with its 8-bit quantisation - and the clips of
 * ISPDataset.__getitem__ (dataset/sid_dataset.py:309,311), as one elementwise kernel.
 *   packed: device f32 [n][4][h][w] (RGBG planes)   rgb: device f32 [n][3][h][w]
 *   wb: HOST [n][4] white-balance gains   ccm: HOST [n][9] cam2rgb, row-major   gamma: 2.2 in the reference
 *   crf_len == 0: gamma curve.  crf_len >= 2: crf_E device [crf_len] (irradiance grid, ascending),
 *   crf_f device [3][crf_len] (per-channel response) - linear interpolation with torchinterp1d's formula. */
int eld_isp_process(eld_ctx* ctx, const float* packed, float* rgb, int n, int h, int w,
                    const float* wb, const float* ccm, float gamma,
                    const float* crf_E, const float* crf_f, int crf_len, void* stream);

/* ------------------------------------------------------------------------------------------------
 * Metric side of ELDModelBase.eval (models/ELD_model.py:203-243), per frame f of a batch of `n` frames with
 * `per_frame` = C*H*W elements each (f32, any layout, pred and target alike):
 *   correct != 0: IlluminanceCorrect.correct (:156-169): gain = <p,s>/<p,p> over the elements where s != 1,
 *                 p = clamp(pred,0,1); corrected = gain * p (written to `out` if out != NULL, may alias pred)
 *   psnr[f] = 10 log10(255^2 / mean((clip(255 x,0,255) - clip(255 target,0,255))^2)), x = corrected (or pred):
 *             tensor2im (:23-38, no rounding) + skimage's peak_signal_noise_ratio(data_range = 255) (util/index.py:76-79)
 * scratch: device, n * 4 doubles (zeroed here).  psnr, gain (may be NULL): device f32 [n].  No host synchronisation. */
int eld_eval_correct_psnr(eld_ctx* ctx, const float* pred, const float* target, float* out, int n, size_t per_frame,
                          int correct, double* scratch, float* psnr, float* gain, void* stream);

/* SSIM of ELDModelBase.eval: tensor2im (:23-38) + skimage's structural_similarity(data_range = 255,
 * multichannel = True) with its defaults (util/index.py:80), per frame f of x and y, device f32 [n][c][h][w]:
 *   per plane, on a = clip(255 x,0,255), b = clip(255 y,0,255) (no rounding): 7x7 box means ux, uy, uxx, uyy, uxy;
 *   vx = 49/48 (uxx - ux^2), vy = 49/48 (uyy - uy^2), vxy = 49/48 (uxy - ux uy); C1 = (0.01*255)^2, C2 = (0.03*255)^2;
 *   S = (2 ux uy + C1)(2 vxy + C2) / ((ux^2 + uy^2 + C1)(vx + vy + C2)), averaged over the (h-6)(w-6) positions whose
 *   window lies inside the plane (skimage's crop by 3: its reflected border never enters the result);
 *   ssim[f] = mean over the c channels.  Symmetric in x, y up to fp32 rounding.  Window sums in fp32 (of the values
 *   less 127.5), sums over positions in double.
 * h, w >= 7 (skimage's 7x7 window), n, c >= 1; x, y contiguous, with no alignment requirement on them or on w.
 * scratch: device, n * c doubles (zeroed here).  ssim: device f32 [n].  Two launches, no host synchronisation. */
int eld_eval_ssim(eld_ctx* ctx, const float* x, const float* y, int n, int c, int h, int w, double* scratch,
                  float* ssim, void* stream);

/* Number of kernels the library has launched through this ctx since creation (bench.py's
 * gpu_launches evidence). */
int64_t eld_launch_count(const eld_ctx* ctx);

/* ------------------------------------------------------------------------------------------------
 * U-Net (UNetSeeInDark, models/arch/Unet.py:6-91) training step on NHWC bf16 activations with fp32
 * master weights.  Declared in eld_b200_unet.h (included below) to keep this file readable.
 */
#include "eld_b200_unet.h"

#ifdef __cplusplus
}
#endif
#endif /* ELD_B200_H */
