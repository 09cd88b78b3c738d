// loss.cu -- the image objective of a DSS training step (Trainer.calc_dr_loss, DSS/training/trainer.py:332-376),
// forward and backward, without a host read-back.
//
// The reference selects the rgb pixels with a boolean index (L1Loss, losses.py:130-137) and branches in Python on
// `mask_pred.sum() > 0`; both wait for the device.  Here the forward is one reduction pass over the pixels that
// writes per-block partial sums, followed by one small kernel that combines them in a fixed order (fp64) into the
// per-view sums and the four loss terms; the backward is one elementwise pass that reads those sums and the upstream
// gradient from device memory.  No atomics: results are bit-reproducible.
#include "common.cuh"

namespace dss {

// per-view sums, in this order, in dss_dr_loss_args::partials and ::sums
enum { LS_COUNT = 0, LS_ABS_RGB, LS_ABS_MASK, LS_INTER, LS_UNION, LS_NUM };

static constexpr int LOSS_THREADS = 256;
static constexpr double LOSS_EPS = 1e-17;   // eps_denom default (DSS/utils/mathHelper.py:10-14)

// eps_denom(U) and d eps_denom / dU as torch autograd gives them: the sign is a constant, the clamp passes the
// gradient where |U| >= eps, abs contributes sgn(U) (0 at U == 0)
__device__ __forceinline__ double loss_eps_denom(double u) {
    const double a = fmax(fabs(u), LOSS_EPS);
    return u < 0.0 ? -a : a;
}
__device__ __forceinline__ double loss_eps_denom_grad(double u) {
    return (u != 0.0 && fabs(u) >= LOSS_EPS) ? 1.0 : 0.0;
}
__device__ __forceinline__ float sgnf(float x) { return x > 0.f ? 1.f : (x < 0.f ? -1.f : 0.f); }

// deterministic sum over the block: fixed shuffle tree per warp, then the warps in order
__device__ __forceinline__ void block_sum(double (&v)[LS_NUM], double (*sh)[LS_NUM]) {
#pragma unroll
    for (int k = 0; k < LS_NUM; ++k)
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) v[k] += __shfl_down_sync(0xffffffffu, v[k], o);
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    if (lane == 0)
#pragma unroll
        for (int k = 0; k < LS_NUM; ++k) sh[warp][k] = v[k];
    __syncthreads();
    if (threadIdx.x == 0) {
        for (int w = 1; w < (int)(blockDim.x >> 5); ++w)
#pragma unroll
            for (int k = 0; k < LS_NUM; ++k) sh[0][k] += sh[w][k];
    }
}

// grid (DSS_DR_LOSS_BLOCKS_PER_VIEW, N): block b of view n accumulates pixels b*T + t, stepping by B*T
__global__ void __launch_bounds__(LOSS_THREADS) dr_loss_partials_kernel(
        const float4 *__restrict__ image, const float *__restrict__ img, const float *__restrict__ mask, int64_t SS,
        double *__restrict__ partials) {
    __shared__ double sh[LOSS_THREADS / 32][LS_NUM];
    const int n = blockIdx.y;
    const float4 *im = image + (int64_t)n * SS;
    const float *r = img + (int64_t)n * 3 * SS, *g = r + SS, *b = g + SS;
    const float *mk = mask + (int64_t)n * SS;
    double v[LS_NUM] = {0.0, 0.0, 0.0, 0.0, 0.0};
    for (int64_t p = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; p < SS; p += (int64_t)gridDim.x * blockDim.x) {
        const float4 q = __ldg(im + p);
        const float m = __ldg(mk + p);
        // differences of two floats are exact in fp64
        const double dr = (double)q.x - __ldg(r + p), dg = (double)q.y - __ldg(g + p), db = (double)q.z - __ldg(b + p);
        if (m != 0.f && q.w != 0.f) {
            v[LS_COUNT] += 1.0;
            v[LS_ABS_RGB] += fabs(dr) + fabs(dg) + fabs(db);
        }
        const double md = m, ad = q.w;
        v[LS_ABS_MASK] += fabs(md - ad);
        v[LS_INTER] += md * ad;
        v[LS_UNION] += md + ad - md * ad;
    }
    block_sum(v, sh);
    if (threadIdx.x == 0) {
        double *out = partials + ((int64_t)n * gridDim.x + blockIdx.x) * LS_NUM;
#pragma unroll
        for (int k = 0; k < LS_NUM; ++k) out[k] = sh[0][k];
    }
}

// one block: warp w combines the partials of views w, w + 8, ... (lane-strided, then a fixed shuffle tree); thread 0
// then adds the views in order and evaluates the loss terms
__global__ void __launch_bounds__(LOSS_THREADS) dr_loss_finish_kernel(
        const double *__restrict__ partials, int N, int B, int64_t SS, float lambda_rgb, float lambda_sil,
        float iou_weight, double *__restrict__ sums, float *__restrict__ terms) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    for (int n = warp; n < N; n += blockDim.x >> 5) {
        double v[LS_NUM] = {0.0, 0.0, 0.0, 0.0, 0.0};
        for (int b = lane; b < B; b += 32) {
            const double *pp = partials + ((int64_t)n * B + b) * LS_NUM;
#pragma unroll
            for (int k = 0; k < LS_NUM; ++k) v[k] += pp[k];
        }
#pragma unroll
        for (int k = 0; k < LS_NUM; ++k)
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) v[k] += __shfl_down_sync(0xffffffffu, v[k], o);
        if (lane == 0)
#pragma unroll
            for (int k = 0; k < LS_NUM; ++k) sums[(int64_t)n * LS_NUM + k] = v[k];
    }
    __syncthreads();
    if (threadIdx.x != 0) return;
    double cnt = 0.0, abs_rgb = 0.0, abs_mask = 0.0, iou = 0.0;
    for (int n = 0; n < N; ++n) {
        const double *s = sums + (int64_t)n * LS_NUM;
        cnt += s[LS_COUNT];
        abs_rgb += s[LS_ABS_RGB];
        abs_mask += s[LS_ABS_MASK];
        iou += 1.0 - s[LS_INTER] / loss_eps_denom(s[LS_UNION]);
    }
    // totals row (read by the backward): {M, sum |d rgb|, sum |m - alpha|, sum_n (1 - I_n / U_n), 0}
    double *tot = sums + (int64_t)N * LS_NUM;
    tot[0] = cnt;
    tot[1] = abs_rgb;
    tot[2] = abs_mask;
    tot[3] = iou;
    tot[4] = 0.0;
    const double l_rgb = cnt > 0.0 ? abs_rgb / cnt : 0.0;
    const double l_mask = abs_mask / ((double)N * (double)SS);
    const double l_iou = iou / N;
    const double l_sil = (double)iou_weight * l_iou + l_mask;
    terms[0] = (float)((double)lambda_rgb * l_rgb + (double)lambda_sil * l_sil);
    terms[1] = (float)l_rgb;
    terms[2] = (float)l_sil;
    terms[3] = (float)l_iou;
}

// grid (x, N): elementwise gradient of the loss with respect to the rendered image
__global__ void __launch_bounds__(LOSS_THREADS) dr_loss_backward_kernel(
        const float4 *__restrict__ image, const float *__restrict__ img, const float *__restrict__ mask, int N,
        int64_t SS, const double *__restrict__ sums, const float *__restrict__ grad_loss, float lambda_rgb,
        float lambda_sil, float iou_weight, float4 *__restrict__ grad_image) {
    const int n = blockIdx.y;
    const double g = (double)__ldg(grad_loss);
    const double *tot = sums + (int64_t)N * LS_NUM;
    const double cnt = tot[0];
    // rgb: g lambda_rgb sgn(d) / M on the selected pixels (no term at all when M == 0)
    const float c_rgb = cnt > 0.0 ? (float)(g * (double)lambda_rgb / cnt) : 0.0f;
    // alpha: silhouette L1 + IoU of this view
    const double gs = g * (double)lambda_sil;
    const double c_mask = gs / ((double)N * (double)SS);
    const double I = sums[(int64_t)n * LS_NUM + LS_INTER], U = sums[(int64_t)n * LS_NUM + LS_UNION];
    const double D = loss_eps_denom(U);
    const double c_i = -gs * (double)iou_weight / N / D;                                   // d/dI = -1/D
    const double c_u = gs * (double)iou_weight / N * I / (D * D) * loss_eps_denom_grad(U);   // d/dU = I/D^2 dD/dU
    const float4 *im = image + (int64_t)n * SS;
    const float *r = img + (int64_t)n * 3 * SS, *gg = r + SS, *b = gg + SS;
    const float *mk = mask + (int64_t)n * SS;
    float4 *out = grad_image + (int64_t)n * SS;
    for (int64_t p = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; p < SS; p += (int64_t)gridDim.x * blockDim.x) {
        const float4 q = __ldg(im + p);
        const float m = __ldg(mk + p);
        float4 o;
        if (m != 0.f && q.w != 0.f) {
            o.x = c_rgb * sgnf(q.x - __ldg(r + p));
            o.y = c_rgb * sgnf(q.y - __ldg(gg + p));
            o.z = c_rgb * sgnf(q.z - __ldg(b + p));
        } else {
            o.x = o.y = o.z = 0.0f;
        }
        const double md = m;
        // I = sum m alpha, U = sum (m + alpha - m alpha):  dI/dalpha = m, dU/dalpha = 1 - m
        o.w = (float)(c_mask * (double)sgnf(q.w - m) + c_i * md + c_u * (1.0 - md));
        out[p] = o;
    }
}

static int check_loss_args(const dss_dr_loss_args *a) {
    DSS_REQUIRE(a != nullptr, "args is null");
    DSS_REQUIRE(a->n_views >= 1 && a->image_size >= 1, "n_views and image_size must be positive");
    DSS_REQUIRE(a->image && a->img && a->mask && a->sums, "image, img, mask and sums are required");
    DSS_REQUIRE((reinterpret_cast<uintptr_t>(a->image) & 15) == 0, "image must be 16-byte aligned");
    return DSS_OK;
}

// blocks per view of the backward: one per LOSS_THREADS pixels, at most 256 (4 pixels per thread at 512 x 512)
static unsigned loss_backward_blocks(int64_t SS) {
    const int64_t per_view = (SS + LOSS_THREADS - 1) / LOSS_THREADS;
    return (unsigned)(per_view < 256 ? per_view : 256);
}

}  // namespace dss

extern "C" {

int dss_dr_loss_forward(dss_ctx *ctx, const dss_dr_loss_args *a, void *stream) {
    using namespace dss;
    cudaStream_t st = (cudaStream_t)stream;
    DSS_REQUIRE(ctx != nullptr, "ctx is null");
    int rc = check_loss_args(a);
    if (rc) return rc;
    DSS_REQUIRE(a->partials && a->terms, "forward needs partials and terms");
    const int64_t SS = (int64_t)a->image_size * a->image_size;
    dim3 grid(DSS_DR_LOSS_BLOCKS_PER_VIEW, (unsigned)a->n_views);
    dr_loss_partials_kernel<<<grid, LOSS_THREADS, 0, st>>>(reinterpret_cast<const float4 *>(a->image), a->img, a->mask,
                                                          SS, a->partials);
    DSS_LAUNCH_CHECK(ctx);
    dr_loss_finish_kernel<<<1, LOSS_THREADS, 0, st>>>(a->partials, a->n_views, DSS_DR_LOSS_BLOCKS_PER_VIEW, SS,
                                                      a->lambda_rgb, a->lambda_silhouette, a->iou_weight, a->sums,
                                                      a->terms);
    DSS_LAUNCH_CHECK(ctx);
    return DSS_OK;
}

int dss_dr_loss_backward(dss_ctx *ctx, const dss_dr_loss_args *a, void *stream) {
    using namespace dss;
    cudaStream_t st = (cudaStream_t)stream;
    DSS_REQUIRE(ctx != nullptr, "ctx is null");
    int rc = check_loss_args(a);
    if (rc) return rc;
    DSS_REQUIRE(a->grad_loss && a->grad_image, "backward needs grad_loss and grad_image");
    DSS_REQUIRE((reinterpret_cast<uintptr_t>(a->grad_image) & 15) == 0, "grad_image must be 16-byte aligned");
    const int64_t SS = (int64_t)a->image_size * a->image_size;
    dim3 grid(loss_backward_blocks(SS), (unsigned)a->n_views);
    dr_loss_backward_kernel<<<grid, LOSS_THREADS, 0, st>>>(
        reinterpret_cast<const float4 *>(a->image), a->img, a->mask, a->n_views, SS, a->sums, a->grad_loss,
        a->lambda_rgb, a->lambda_silhouette, a->iou_weight, reinterpret_cast<float4 *>(a->grad_image));
    DSS_LAUNCH_CHECK(ctx);
    return DSS_OK;
}

}  // extern "C"
