// eval.cu - the metric side of ELDModelBase.eval (reference models/ELD_model.py:203-243) on the device, so that
// Engine.eval (engine.py:75-99, every 20 epochs in train_syn.py:108-113) never pulls frames to the host:
//   IlluminanceCorrect.correct (ELD_model.py:156-169): gain = <p, s> / <p, p> over the elements where s != 1, with
//       p = clamp(predict, 0, 1);  output = gain * p
//   tensor2im (ELD_model.py:23-38): clip(255 * x, 0, 255), no rounding
//   quality_assess -> skimage peak_signal_noise_ratio(data_range = 255) (util/index.py:76-79):
//       PSNR = 10 log10(255^2 / mean((a - b)^2))
//   quality_assess -> skimage structural_similarity(data_range = 255, multichannel = True) (util/index.py:80): SSIM
// Three launches for PSNR (two reductions + a finalise), two for SSIM (tile reduction + finalise), double accumulation,
// no host synchronisation.
#include "common.cuh"

namespace eld {

__device__ __forceinline__ double block_sum(double v, double* sh)
{
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    const int w = threadIdx.x >> 5, l = threadIdx.x & 31;
    __syncthreads();
    if (l == 0) sh[w] = v;
    __syncthreads();
    double t = 0.0;
    if (threadIdx.x < (blockDim.x >> 5)) t = sh[threadIdx.x];
    if (w == 0) {
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) t += __shfl_xor_sync(0xffffffffu, t, o);
    }
    return t;     // valid in thread 0
}

// acc[f][0] += <p, s>, acc[f][1] += <p, p> over s != 1
__global__ void __launch_bounds__(256)
eval_dots_kernel(const float* __restrict__ pred, const float* __restrict__ src, size_t per_frame, double* __restrict__ acc)
{
    __shared__ double sh[8];
    const int f = blockIdx.y;
    const float* p = pred + (size_t)f * per_frame;
    const float* s = src + (size_t)f * per_frame;
    double num = 0.0, den = 0.0;
    for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < per_frame; i += (size_t)gridDim.x * blockDim.x) {
        const float sv = __ldg(s + i);
        const float pv = fminf(fmaxf(__ldg(p + i), 0.0f), 1.0f);
        if (sv != 1.0f) { num += (double)pv * (double)sv; den += (double)pv * (double)pv; }
    }
    const double a = block_sum(num, sh);
    const double b = block_sum(den, sh);
    if (threadIdx.x == 0) { atomicAdd(acc + f * 4 + 0, a); atomicAdd(acc + f * 4 + 1, b); }
}

// out = gain * clamp(p) (correct) or p; acc[f][2] += sum (clip(255 out) - clip(255 s))^2
__global__ void __launch_bounds__(256)
eval_apply_kernel(const float* __restrict__ pred, const float* __restrict__ src, float* __restrict__ out, size_t per_frame,
                  int correct, double* __restrict__ acc)
{
    __shared__ double sh[8];
    const int f = blockIdx.y;
    const float* p = pred + (size_t)f * per_frame;
    const float* s = src + (size_t)f * per_frame;
    float* o = out ? out + (size_t)f * per_frame : nullptr;
    // the reference forms num / den in fp32 (torch.dot) and multiplies in fp32
    const float gain = correct ? (float)acc[f * 4 + 0] / (float)acc[f * 4 + 1] : 1.0f;
    double sq = 0.0;
    for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < per_frame; i += (size_t)gridDim.x * blockDim.x) {
        float v = __ldg(p + i);
        if (correct) v = gain * fminf(fmaxf(v, 0.0f), 1.0f);
        if (o) o[i] = v;
        const float a = fminf(fmaxf(v * 255.0f, 0.0f), 255.0f);
        const float b = fminf(fmaxf(__ldg(s + i) * 255.0f, 0.0f), 255.0f);
        const double d = (double)a - (double)b;
        sq += d * d;
    }
    const double t = block_sum(sq, sh);
    if (threadIdx.x == 0) atomicAdd(acc + f * 4 + 2, t);
}

__global__ void eval_finalize_kernel(const double* __restrict__ acc, size_t per_frame, int n, int correct,
                                     float* __restrict__ psnr, float* __restrict__ gain)
{
    const int f = blockIdx.x * blockDim.x + threadIdx.x;
    if (f >= n) return;
    const double mse = acc[f * 4 + 2] / (double)per_frame;
    psnr[f] = (float)(10.0 * log10(255.0 * 255.0 / mse));
    if (gain) gain[f] = correct ? (float)acc[f * 4 + 0] / (float)acc[f * 4 + 1] : 1.0f;
}

// ---- SSIM: quality_assess -> skimage structural_similarity(data_range = 255, multichannel = True) (util/index.py:80)
// with skimage's defaults: 7x7 uniform window, sample covariance (49/48), K1 = 0.01, K2 = 0.03; the per-position map is
// averaged over the interior (positions whose window lies inside the plane, skimage's crop by 3), then over channels.
// A CTA owns SSIM_TH x SSIM_TW interior outputs of one plane: it stages the tile plus the 6-pixel halo of both planes
// (clip(255 v) applied) in shared memory; each thread owns two adjacent output columns, forms the five 7-tap row sums
// of every staged row and keeps the last 7 in registers for the 7-tap column sums.  Window sums are direct fp32 sums
// in tap order (no running add / subtract), the per-position formula is fp32, partial sums over positions are double.
// The staged values are clip(255 v) - 127.5: the (co)variances do not change under a shift, and halving the magnitude
// quarters the fp32 rounding of the second moments where uxx - ux^2 cancels (bright, flat regions).
constexpr int SSIM_THREADS = 128;
constexpr int SSIM_TW = 2 * SSIM_THREADS;       // output columns per tile
constexpr int SSIM_TH = 16;                     // output rows per tile
constexpr int SSIM_ROWS = SSIM_TH + 6;
constexpr int SSIM_PITCH = SSIM_TW + 8;         // >= SSIM_TW + 6 staged columns, a multiple of 4 (float4 / float2 access)

constexpr float SSIM_SHIFT = 127.5f;

__device__ __forceinline__ float to_im(float v) { return fminf(fmaxf(v * 255.0f, 0.0f), 255.0f) - SSIM_SHIFT; }

__global__ void __launch_bounds__(SSIM_THREADS, 4)
eval_ssim_tile_kernel(const float* __restrict__ x, const float* __restrict__ y, int h, int w, int tiles_x, int tiles_y,
                      int vec4, double* __restrict__ acc)
{
    __shared__ __align__(16) float sx[SSIM_ROWS][SSIM_PITCH];
    __shared__ __align__(16) float sy[SSIM_ROWS][SSIM_PITCH];
    __shared__ double sh[SSIM_THREADS / 32];
    const int tile = blockIdx.x % (tiles_x * tiles_y);
    const int plane = blockIdx.x / (tiles_x * tiles_y);
    const int row0 = (tile / tiles_x) * SSIM_TH, col0 = (tile % tiles_x) * SSIM_TW;
    const size_t base = (size_t)plane * h * w;
    const float* px = x + base;
    const float* py = y + base;

    // stage rows row0 .. row0+21, columns col0 .. col0+SSIM_PITCH-1; outside the plane -> 0 (feeds masked outputs only)
    constexpr int CHUNKS = SSIM_PITCH / 4;
    for (int i = threadIdx.x; i < SSIM_ROWS * CHUNKS; i += SSIM_THREADS) {
        const int r = i / CHUNKS, c = (i % CHUNKS) * 4;
        const int gr = row0 + r, gc = col0 + c;
        float4 a = make_float4(0.f, 0.f, 0.f, 0.f), b = a;
        if (gr < h) {
            const size_t o = (size_t)gr * w + gc;
            if (vec4 && gc + 3 < w) {
                a = __ldg(reinterpret_cast<const float4*>(px + o));
                b = __ldg(reinterpret_cast<const float4*>(py + o));
            } else {
                if (gc + 0 < w) { a.x = __ldg(px + o + 0); b.x = __ldg(py + o + 0); }
                if (gc + 1 < w) { a.y = __ldg(px + o + 1); b.y = __ldg(py + o + 1); }
                if (gc + 2 < w) { a.z = __ldg(px + o + 2); b.z = __ldg(py + o + 2); }
                if (gc + 3 < w) { a.w = __ldg(px + o + 3); b.w = __ldg(py + o + 3); }
            }
        }
        *reinterpret_cast<float4*>(&sx[r][c]) = make_float4(to_im(a.x), to_im(a.y), to_im(a.z), to_im(a.w));
        *reinterpret_cast<float4*>(&sy[r][c]) = make_float4(to_im(b.x), to_im(b.y), to_im(b.z), to_im(b.w));
    }
    __syncthreads();

    const float inv = 1.0f / 49.0f, cov = 49.0f / 48.0f;
    const float C1 = (0.01f * 255.0f) * (0.01f * 255.0f), C2 = (0.03f * 255.0f) * (0.03f * 255.0f);
    const int c0 = 2 * threadIdx.x;
    const int oh = h - 6, ow = w - 6;
    const bool col_ok0 = col0 + c0 < ow, col_ok1 = col0 + c0 + 1 < ow;
    // ring of the last 7 rows' horizontal sums: [row % 7][quantity][column]
    float hs[7][5][2];
    double part = 0.0;
#pragma unroll
    for (int r = 0; r < SSIM_ROWS; ++r) {
        float a[8], b[8];
#pragma unroll
        for (int k = 0; k < 8; k += 2) {
            const float2 va = *reinterpret_cast<const float2*>(&sx[r][c0 + k]);
            const float2 vb = *reinterpret_cast<const float2*>(&sy[r][c0 + k]);
            a[k] = va.x; a[k + 1] = va.y; b[k] = vb.x; b[k + 1] = vb.y;
        }
#pragma unroll
        for (int e = 0; e < 2; ++e) {
            float s0 = a[e], s1 = b[e], s2 = a[e] * a[e], s3 = b[e] * b[e], s4 = a[e] * b[e];
#pragma unroll
            for (int k = 1; k < 7; ++k) {
                const float u = a[e + k], v = b[e + k];
                s0 += u; s1 += v; s2 += u * u; s3 += v * v; s4 += u * v;
            }
            hs[r % 7][0][e] = s0; hs[r % 7][1][e] = s1; hs[r % 7][2][e] = s2; hs[r % 7][3][e] = s3; hs[r % 7][4][e] = s4;
        }
        if (r >= 6) {
            const int o = r - 6;
            const bool row_ok = row0 + o < oh;
#pragma unroll
            for (int e = 0; e < 2; ++e) {
                float m[5];
#pragma unroll
                for (int q = 0; q < 5; ++q) {
                    float s = hs[o % 7][q][e];
#pragma unroll
                    for (int k = 1; k < 7; ++k) s += hs[(o + k) % 7][q][e];
                    m[q] = s * inv;
                }
                const float vx = cov * (m[2] - m[0] * m[0]), vy = cov * (m[3] - m[1] * m[1]), vxy = cov * (m[4] - m[0] * m[1]);
                const float ux = m[0] + SSIM_SHIFT, uy = m[1] + SSIM_SHIFT;
                const float S = ((2.0f * ux * uy + C1) * (2.0f * vxy + C2)) / ((ux * ux + uy * uy + C1) * (vx + vy + C2));
                if (row_ok && (e == 0 ? col_ok0 : col_ok1)) part += (double)S;
            }
        }
    }
    const double t = block_sum(part, sh);
    if (threadIdx.x == 0) atomicAdd(acc + plane, t);
}

// ssim[f] = mean over the c channels of (sum of the plane's map) / ((h-6)(w-6))
__global__ void eval_ssim_finalize_kernel(const double* __restrict__ acc, int n, int c, double count, float* __restrict__ ssim)
{
    const int f = blockIdx.x * blockDim.x + threadIdx.x;
    if (f >= n) return;
    double s = 0.0;
    for (int k = 0; k < c; ++k) s += acc[(size_t)f * c + k] / count;
    ssim[f] = (float)(s / c);
}

}  // namespace eld

using namespace eld;

extern "C" int eld_eval_correct_psnr(eld_ctx* ctx, const float* pred, const float* target, float* out, int n, size_t per_frame,
                                     int correct, double* scratch, float* psnr, float* gain, void* stream)
{
    ELD_REQUIRE(ctx && pred && target && scratch && psnr, "eld_eval_correct_psnr: NULL argument");
    ELD_REQUIRE(n > 0 && per_frame > 0, "eld_eval_correct_psnr: empty batch");
    ELD_CHECK_CUDA(cudaSetDevice(ctx->device));
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    ELD_CHECK_CUDA(cudaMemsetAsync(scratch, 0, (size_t)n * 4 * sizeof(double), st));
    int bx = (int)((per_frame + 256 * 8 - 1) / (256 * 8));
    const int cap = (4 * ctx->num_sms + n - 1) / n;
    if (bx > cap) bx = cap;
    if (bx < 1) bx = 1;
    const dim3 grid((unsigned)bx, (unsigned)n);
    if (correct) {
        eval_dots_kernel<<<grid, 256, 0, st>>>(pred, target, per_frame, scratch);
        count_launch(ctx);
    }
    eval_apply_kernel<<<grid, 256, 0, st>>>(pred, target, out, per_frame, correct, scratch);
    eval_finalize_kernel<<<(n + 63) / 64, 64, 0, st>>>(scratch, per_frame, n, correct, psnr, gain);
    ELD_CHECK_CUDA(cudaGetLastError());
    count_launch(ctx, 2);
    return ELD_OK;
}

extern "C" int eld_eval_ssim(eld_ctx* ctx, const float* x, const float* y, int n, int c, int h, int w, double* scratch,
                             float* ssim, void* stream)
{
    ELD_REQUIRE(ctx && x && y && scratch && ssim, "eld_eval_ssim: NULL argument");
    ELD_REQUIRE(n >= 1 && c >= 1, "eld_eval_ssim: empty batch (n = %d, c = %d)", n, c);
    ELD_REQUIRE(h >= 7 && w >= 7, "eld_eval_ssim: %d x %d plane is smaller than skimage's 7 x 7 SSIM window", h, w);
    const long long tiles_x = (w - 6 + SSIM_TW - 1) / SSIM_TW, tiles_y = (h - 6 + SSIM_TH - 1) / SSIM_TH;
    const long long blocks = tiles_x * tiles_y * n * c;
    ELD_REQUIRE(blocks <= 0x7fffffffLL, "eld_eval_ssim: batch too large (%lld tiles)", blocks);
    ELD_CHECK_CUDA(cudaSetDevice(ctx->device));
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    ELD_CHECK_CUDA(cudaMemsetAsync(scratch, 0, (size_t)n * c * sizeof(double), st));
    // float4 staging needs 16-byte rows: w % 4 == 0 and both planes 16-byte aligned
    const int vec4 = (w % 4 == 0) && ((reinterpret_cast<uintptr_t>(x) | reinterpret_cast<uintptr_t>(y)) % 16 == 0);
    eval_ssim_tile_kernel<<<(unsigned)blocks, SSIM_THREADS, 0, st>>>(x, y, h, w, (int)tiles_x, (int)tiles_y, vec4, scratch);
    eval_ssim_finalize_kernel<<<(n + 63) / 64, 64, 0, st>>>(scratch, n, c, (double)(h - 6) * (double)(w - 6), ssim);
    ELD_CHECK_CUDA(cudaGetLastError());
    count_launch(ctx, 2);
    return ELD_OK;
}
