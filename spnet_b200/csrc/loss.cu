// Fused YOLO-ellipse loss (value, 5-term breakdown and dL/dy_pred in one launch),
// selective sigmoid, and detection decode.
//
// Follows the reference's custom_loss (spnet/models.py:564-589) and its numpy
// twin my_loss (:594-633); constants from :557-562; column layout from
// spnet/config.py:30-38 (8 variables per predictor:
// cx, cy, a, b, cos2t, sin2t, noobj, rings).
#include "common.cuh"

namespace {

constexpr float kLambdaCenter = 2.0f;
constexpr float kLambdaSize = 1.0f;
constexpr float kLambdaAngle = 3.0f;
constexpr float kLambdaNoobj = 0.3f;
constexpr float kLambdaClass = 5.0f;

constexpr int kLossThreads = 1024;

__device__ __forceinline__ float sigmoidf_(float x) { return 1.0f / (1.0f + expf(-x)); }

// Loss terms of one sample row for the predictors this lane owns (lanes stride over predictors).
// yt may point to global or shared memory. acc = center,size,angle,noobj,class partial sums.
__device__ __forceinline__ void loss_row(const float* yt, const float* __restrict__ yp, float* __restrict__ g, int npred,
                                         int lane, int hybrid, int sel_sigmoid, float c, float (&acc)[5]) {
    for (int p = lane; p < npred; p += 32) {
        float t[8], q[8];
        const float4 t0 = *reinterpret_cast<const float4*>(yt + p * 8);
        const float4 t1 = *reinterpret_cast<const float4*>(yt + p * 8 + 4);
        const float4 q0 = *reinterpret_cast<const float4*>(yp + p * 8);
        const float4 q1 = *reinterpret_cast<const float4*>(yp + p * 8 + 4);
        t[0] = t0.x; t[1] = t0.y; t[2] = t0.z; t[3] = t0.w; t[4] = t1.x; t[5] = t1.y; t[6] = t1.z; t[7] = t1.w;
        q[0] = q0.x; q[1] = q0.y; q[2] = q0.z; q[3] = q0.w; q[4] = q1.x; q[5] = q1.y; q[6] = q1.z; q[7] = q1.w;

        float dsig = 1.0f;  // d(noobj activation)/d(raw)
        if (sel_sigmoid) {
            const float sg = sigmoidf_(q[6]);
            dsig = sg * (1.0f - sg);
            q[6] = sg;
        }
        const float pobj = 1.0f - t[6];
        const float ab = t[2] - t[3];
        const float ab2 = ab * ab;
        float e[8];
#pragma unroll
        for (int i = 0; i < 8; ++i) e[i] = q[i] - t[i];

        acc[0] += pobj * (e[0] * e[0]) + pobj * (e[1] * e[1]);
        acc[1] += pobj * (e[2] * e[2]) + pobj * (e[3] * e[3]);
        acc[2] += pobj * (e[4] * e[4]) * ab2 + pobj * (e[5] * e[5]) * ab2;
        acc[4] += pobj * (e[7] * e[7]);
        float gno;
        if (hybrid) {
            const float z = q[6];
            acc[3] += fmaxf(0.0f, z) - z * t[6] + log1pf(expf(-fabsf(z)));
            gno = kLambdaNoobj * (sigmoidf_(z) - t[6]);
        } else {
            acc[3] += e[6] * e[6];
            gno = 2.0f * kLambdaNoobj * e[6];
        }
        if (g) {
            float4 g0, g1;
            g0.x = 2.0f * kLambdaCenter * pobj * e[0] * c;
            g0.y = 2.0f * kLambdaCenter * pobj * e[1] * c;
            g0.z = 2.0f * kLambdaSize * pobj * e[2] * c;
            g0.w = 2.0f * kLambdaSize * pobj * e[3] * c;
            g1.x = 2.0f * kLambdaAngle * pobj * ab2 * e[4] * c;
            g1.y = 2.0f * kLambdaAngle * pobj * ab2 * e[5] * c;
            g1.z = gno * dsig * c;
            g1.w = 2.0f * kLambdaClass * pobj * e[7] * c;
            *reinterpret_cast<float4*>(g + p * 8) = g0;
            *reinterpret_cast<float4*>(g + p * 8 + 4) = g1;
        }
    }
}

// Fixed-order batch reduction of the per-warp partial sums (bitwise reproducible run to run).
__device__ __forceinline__ void loss_finish(float (&acc)[5], int warp, int lane, int nwarps, float c, float* __restrict__ out6) {
    __shared__ float part[32][5];
#pragma unroll
    for (int i = 0; i < 5; ++i) acc[i] = warp_sum(acc[i]);
    if (lane == 0) {
#pragma unroll
        for (int i = 0; i < 5; ++i) part[warp][i] = acc[i];
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        float tot[5] = {0.f, 0.f, 0.f, 0.f, 0.f};
        for (int w = 0; w < nwarps; ++w)
            for (int i = 0; i < 5; ++i) tot[i] += part[w][i];
        const float lam[5] = {kLambdaCenter, kLambdaSize, kLambdaAngle, kLambdaNoobj, kLambdaClass};
        float total = 0.f;
        for (int i = 0; i < 5; ++i) {
            const float v = lam[i] * tot[i] * c;
            out6[1 + i] = v;
            total += v;
        }
        out6[0] = total;
    }
}

// One warp per sample, lanes stride over predictors. Single CTA so that the
// batch reduction has a fixed order (bitwise reproducible run to run).
// out6 = [total, center, size, angle, noobj, class], each already divided by
// ncols and averaged over the batch, as my_loss returns them.
__global__ void __launch_bounds__(kLossThreads) yolo_ellipse_loss_kernel(
    const float* __restrict__ y_true, const float* __restrict__ y_pred, int batch, int ncols,
    int hybrid, int sel_sigmoid, float* __restrict__ out6, float* __restrict__ grad) {
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, nwarps = blockDim.x >> 5;
    const int npred = ncols >> 3;
    const float c = 1.0f / ((float)ncols * (float)batch);
    float acc[5] = {0.f, 0.f, 0.f, 0.f, 0.f};  // center,size,angle,noobj,class
    for (int s = warp; s < batch; s += nwarps)
        loss_row(y_true + (size_t)s * ncols, y_pred + (size_t)s * ncols, grad ? grad + (size_t)s * ncols : nullptr, npred, lane,
                 hybrid, sel_sigmoid, c, acc);
    loss_finish(acc, warp, lane, nwarps, c, out6);
}

// ---- grid-cell / slot assignment (true_to_pred_grid, spnet/utils.py:191-244) + norm_Y (:179-184) ----
// One image per warp. ann: [n, max_obj, 8] float64 rows [cx,cy,a,b,cos2t,sin2t,noobj,rings] exactly as
// parse_meta_file returns them (already sorted by (cx, cy), :284); counts[n] rows in use. The row of
// antinode j goes to cell ix = int((cx - 40) / xbin), iy = int((cy - 40) / ybin) (float64 divide, truncation
// toward zero, clamped to the grid), slot = number of antinodes this cell already holds; a cell that is
// offered more than `ppc` antinodes trips the reference's assert (:240): here err[image] = 1 + j of the first
// offender and that antinode is dropped (the host wrapper raises AssertionError). Everything not assigned keeps
// the per-cell defaults. Output row = (value cast to fp32 - means) / ranges in fp32, the two roundings numpy does.
__device__ __forceinline__ void assign_row(const double* __restrict__ ann, int cnt, int nx, int ny, int ppc, int xbin, int ybin,
                                           const float* __restrict__ defaults, const float* __restrict__ means,
                                           const float* __restrict__ ranges, float* yrow, unsigned char* cell_count, int lane,
                                           int* err_out) {
    const int ncols = nx * ny * ppc * 8;
    for (int i = lane; i < ncols; i += 32) yrow[i] = __fdiv_rn(__fsub_rn(defaults[i], means[i]), ranges[i]);
    for (int i = lane; i < nx * ny; i += 32) cell_count[i] = 0;
    __syncwarp();
    if (lane == 0) {
        int err = 0;
        for (int j = 0; j < cnt; ++j) {
            const double* row = ann + (size_t)j * 8;
            int ix = (int)((row[0] - 40.0) / (double)xbin);  // C cast = truncation toward zero = python int()
            int iy = (int)((row[1] - 40.0) / (double)ybin);
            ix = min(max(ix, 0), nx - 1);
            iy = min(max(iy, 0), ny - 1);
            const int slot = cell_count[ix * ny + iy];
            if (slot >= ppc) {
                if (!err) err = j + 1;
                continue;
            }
            cell_count[ix * ny + iy] = (unsigned char)(slot + 1);
            const int o = ((ix * ny + iy) * ppc + slot) * 8;
#pragma unroll
            for (int k = 0; k < 8; ++k) yrow[o + k] = __fdiv_rn(__fsub_rn((float)row[k], means[o + k]), ranges[o + k]);
        }
        if (err_out) *err_out = err;
    }
    __syncwarp();
}

__global__ void __launch_bounds__(256) assign_grid_kernel(const double* __restrict__ ann, const int* __restrict__ counts, int n,
                                                          int max_obj, int nx, int ny, int ppc, int xbin, int ybin,
                                                          const float* __restrict__ defaults, const float* __restrict__ means,
                                                          const float* __restrict__ ranges, float* __restrict__ Y, int* __restrict__ err) {
    __shared__ unsigned char cells[8][256];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int img = blockIdx.x * 8 + warp;
    if (img >= n) return;
    const int ncols = nx * ny * ppc * 8;
    assign_row(ann + (size_t)img * max_obj * 8, counts[img], nx, ny, ppc, xbin, ybin, defaults, means, ranges,
               Y + (size_t)img * ncols, cells[warp], lane, err + img);
}

// custom_loss straight from the annotations: every warp first builds its sample's target row in shared memory
// (assignment + normalisation above), then runs the same loss / gradient arithmetic on it - one launch covers
// grid-cell/slot assignment, ellipse and ring-count regression and the (optional) selective sigmoid.
// y_true_out (nullable) receives the rows. Dynamic shared memory: nwarps * (ncols * 4 + 256) bytes.
__global__ void __launch_bounds__(kLossThreads) yolo_ellipse_loss_ann_kernel(
    const double* __restrict__ ann, const int* __restrict__ counts, int max_obj, int nx, int ny, int ppc, int xbin, int ybin,
    const float* __restrict__ defaults, const float* __restrict__ means, const float* __restrict__ ranges,
    const float* __restrict__ y_pred, int batch, int hybrid, int sel_sigmoid, float* __restrict__ y_true_out,
    float* __restrict__ out6, float* __restrict__ grad, int* __restrict__ err) {
    extern __shared__ __align__(16) unsigned char loss_smem[];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, nwarps = blockDim.x >> 5;
    const int ncols = nx * ny * ppc * 8, npred = ncols >> 3;
    float* yrow = reinterpret_cast<float*>(loss_smem) + (size_t)warp * ncols;
    unsigned char* cells = loss_smem + (size_t)nwarps * ncols * 4 + (size_t)warp * 256;
    const float c = 1.0f / ((float)ncols * (float)batch);
    float acc[5] = {0.f, 0.f, 0.f, 0.f, 0.f};
    for (int s = warp; s < batch; s += nwarps) {
        assign_row(ann + (size_t)s * max_obj * 8, counts[s], nx, ny, ppc, xbin, ybin, defaults, means, ranges, yrow, cells, lane,
                   err + s);
        if (y_true_out)
            for (int i = lane; i < ncols; i += 32) y_true_out[(size_t)s * ncols + i] = yrow[i];
        loss_row(yrow, y_pred + (size_t)s * ncols, grad ? grad + (size_t)s * ncols : nullptr, npred, lane, hybrid, sel_sigmoid, c,
                 acc);
        __syncwarp();
    }
    loss_finish(acc, warp, lane, nwarps, c, out6);
}

// (v / 255 - 0.5) * 2 of spnet/utils.py:340-342 for uint8 frames: there are only 256 inputs, so the caller passes the
// 256 results computed by numpy in fp32 - bit-exact by construction - and the kernel is a table look-up at HBM speed.
__global__ void __launch_bounds__(256) normalize_u8_kernel(const uint4* __restrict__ in, const float* __restrict__ lut,
                                                           float4* __restrict__ out, long long n16, const unsigned char* tail_in,
                                                           float* tail_out, int ntail) {
    __shared__ float sl[256];
    sl[threadIdx.x] = lut[threadIdx.x];
    __syncthreads();
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n16; i += (long long)gridDim.x * blockDim.x) {
        const uint4 v = in[i];
        const uint32_t w[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
        for (int k = 0; k < 4; ++k)
            out[i * 4 + k] = make_float4(sl[w[k] & 255u], sl[(w[k] >> 8) & 255u], sl[(w[k] >> 16) & 255u], sl[w[k] >> 24]);
    }
    if (blockIdx.x == 0 && (int)threadIdx.x < ntail) tail_out[threadIdx.x] = sl[tail_in[threadIdx.x]];
}

// y[:, j] = sigmoid(x[:, j]) for j in range(start, end, skip), identity elsewhere
// (SelectiveSigmoid, spnet/models.py:277-298).
__global__ void selective_sigmoid_fwd_kernel(const float* __restrict__ x, float* __restrict__ y,
                                             long long n, int ncols, int start, int end, int skip) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const int j = (int)(i % ncols);
    const bool sel = j >= start && j < end && ((j - start) % skip == 0);
    const float v = x[i];
    y[i] = sel ? sigmoidf_(v) : v;
}

// dx = dy * y(1-y) on the selected columns (y = forward output), dy elsewhere.
__global__ void selective_sigmoid_bwd_kernel(const float* __restrict__ y, const float* __restrict__ dy,
                                             float* __restrict__ dx, long long n, int ncols, int start,
                                             int end, int skip) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const int j = (int)(i % ncols);
    const bool sel = j >= start && j < end && ((j - start) % skip == 0);
    const float yy = y[i];
    dx[i] = sel ? dy[i] * yy * (1.0f - yy) : dy[i];
}

// Decode (denorm_Y + cleanup_antinode_vars' integer part + existence test;
// spnet/utils.py:186-188, :56-64, :109-118). One thread per predictor.
//   denorm  [n, ncols] f32 : y*ranges + means, two roundings exactly as numpy does
//   ints    [n, npred, 5] i32 : round-half-even of cx, cy, a, b, noobj
//   exists  [n, npred] u8  : noobj==0 && rings>0 && a>=0 && b>=0
__global__ void decode_detections_kernel(const float* __restrict__ y, const float* __restrict__ means,
                                         const float* __restrict__ ranges, int n, int ncols,
                                         float* __restrict__ denorm, int* __restrict__ ints,
                                         unsigned char* __restrict__ exists) {
    const int npred = ncols >> 3;
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= (long long)n * npred) return;
    const int p = (int)(i % npred);
    const size_t row = (size_t)(i / npred) * ncols + (size_t)p * 8;
    float v[8];
#pragma unroll
    for (int k = 0; k < 8; ++k) {
        v[k] = __fadd_rn(__fmul_rn(y[row + k], ranges[p * 8 + k]), means[p * 8 + k]);
        denorm[row + k] = v[k];
    }
    const int cx = __float2int_rn(v[0]), cy = __float2int_rn(v[1]);
    const int a = __float2int_rn(v[2]), b = __float2int_rn(v[3]);
    const int noobj = __float2int_rn(v[6]);
    int* o = ints + i * 5;
    o[0] = cx; o[1] = cy; o[2] = a; o[3] = b; o[4] = noobj;
    exists[i] = (noobj == 0 && v[7] > 0.0f && a >= 0 && b >= 0) ? 1 : 0;
}

}  // namespace

extern "C" {

int spnet_yolo_ellipse_loss(const float* y_true, const float* y_pred, int batch, int ncols, int hybrid,
                            int sel_sigmoid, float* out6, float* grad, cudaStream_t stream) {
    SPNET_REQUIRE(y_true && y_pred && out6, "yolo_ellipse_loss: null pointer");
    SPNET_REQUIRE(batch > 0 && ncols > 0 && ncols % 8 == 0, "yolo_ellipse_loss: bad shape %d x %d", batch, ncols);
    yolo_ellipse_loss_kernel<<<1, kLossThreads, 0, stream>>>(y_true, y_pred, batch, ncols, hybrid, sel_sigmoid,
                                                             out6, grad);
    return spnet_check_launch("yolo_ellipse_loss");
}

int spnet_selective_sigmoid_fwd(const float* x, float* y, int rows, int ncols, int start, int end, int skip,
                                cudaStream_t stream) {
    SPNET_REQUIRE(x && y && rows > 0 && ncols > 0 && skip > 0, "selective_sigmoid_fwd: bad args");
    const long long n = (long long)rows * ncols;
    selective_sigmoid_fwd_kernel<<<ceil_div(n, 256), 256, 0, stream>>>(x, y, n, ncols, start, end, skip);
    return spnet_check_launch("selective_sigmoid_fwd");
}

int spnet_selective_sigmoid_bwd(const float* y, const float* dy, float* dx, int rows, int ncols, int start,
                                int end, int skip, cudaStream_t stream) {
    SPNET_REQUIRE(y && dy && dx && rows > 0 && ncols > 0 && skip > 0, "selective_sigmoid_bwd: bad args");
    const long long n = (long long)rows * ncols;
    selective_sigmoid_bwd_kernel<<<ceil_div(n, 256), 256, 0, stream>>>(y, dy, dx, n, ncols, start, end, skip);
    return spnet_check_launch("selective_sigmoid_bwd");
}

int spnet_decode_detections(const float* y, const float* means, const float* ranges, int n, int ncols,
                            float* denorm, int* ints, unsigned char* exists, cudaStream_t stream) {
    SPNET_REQUIRE(y && means && ranges && denorm && ints && exists, "decode_detections: null pointer");
    SPNET_REQUIRE(n > 0 && ncols > 0 && ncols % 8 == 0, "decode_detections: bad shape");
    const long long total = (long long)n * (ncols / 8);
    decode_detections_kernel<<<ceil_div(total, 256), 256, 0, stream>>>(y, means, ranges, n, ncols, denorm, ints,
                                                                       exists);
    return spnet_check_launch("decode_detections");
}

// true_to_pred_grid (spnet/utils.py:191-244) + norm_Y (:179-184) for n images in one launch.
// ann [n, max_obj, 8] float64, counts [n] int32, defaults / means / ranges [nx*ny*ppc*8] fp32 (setup_means_and_ranges,
// :144-176), Y [n, nx*ny*ppc*8] fp32, err [n] int32 (0, or 1 + index of the antinode that overflowed its cell).
int spnet_assign_grid(const double* ann, const int* counts, int n, int max_obj, int nx, int ny, int ppc, const float* defaults,
                      const float* means, const float* ranges, float* Y, int* err, cudaStream_t stream) {
    SPNET_REQUIRE(ann && counts && defaults && means && ranges && Y && err, "assign_grid: null pointer");
    SPNET_REQUIRE(n > 0 && max_obj >= 0 && nx > 0 && ny > 0 && ppc > 0 && nx * ny <= 256 && ppc < 255, "assign_grid: bad shape");
    const int xbin = (470 - 40) / nx, ybin = (350 - 40) / ny;  // int((cx_max - cx_min) / pred_shape[0]) of :151-152
    SPNET_REQUIRE(xbin > 0 && ybin > 0, "assign_grid: grid too fine");
    assign_grid_kernel<<<ceil_div(n, 8), 256, 0, stream>>>(ann, counts, n, max_obj, nx, ny, ppc, xbin, ybin, defaults, means,
                                                           ranges, Y, err);
    return spnet_check_launch("assign_grid");
}

// custom_loss (spnet/models.py:564-589) fed by the raw annotations: assignment + normalisation + loss + gradient in
// ONE launch. y_true_out nullable [batch, ncols]; other arguments as spnet_assign_grid / spnet_yolo_ellipse_loss.
int spnet_yolo_ellipse_loss_ann(const double* ann, const int* counts, int max_obj, int nx, int ny, int ppc, const float* defaults,
                                const float* means, const float* ranges, const float* y_pred, int batch, int hybrid,
                                int sel_sigmoid, float* y_true_out, float* out6, float* grad, int* err, cudaStream_t stream) {
    SPNET_REQUIRE(ann && counts && defaults && means && ranges && y_pred && out6 && err, "yolo_ellipse_loss_ann: null pointer");
    SPNET_REQUIRE(batch > 0 && max_obj >= 0 && nx > 0 && ny > 0 && ppc > 0 && nx * ny <= 256 && ppc < 255,
                  "yolo_ellipse_loss_ann: bad shape");
    const int xbin = (470 - 40) / nx, ybin = (350 - 40) / ny;
    SPNET_REQUIRE(xbin > 0 && ybin > 0, "yolo_ellipse_loss_ann: grid too fine");
    const int ncols = nx * ny * ppc * 8;
    constexpr size_t kSmemMax = 200 * 1024;  // opted in to once; each launch asks for what its columns need
    int nwarps = kLossThreads / 32;
    while (nwarps > 1 && (size_t)nwarps * (ncols * 4 + 256) > kSmemMax) nwarps >>= 1;
    const size_t smem = (size_t)nwarps * (ncols * 4 + 256);
    SPNET_REQUIRE(smem <= kSmemMax, "yolo_ellipse_loss_ann: %d output columns do not fit shared memory", ncols);
    static bool configured[64] = {};
    const int rc = spnet_smem_optin(configured, yolo_ellipse_loss_ann_kernel, kSmemMax, "yolo_ellipse_loss_ann");
    if (rc) return rc;
    yolo_ellipse_loss_ann_kernel<<<1, nwarps * 32, smem, stream>>>(ann, counts, max_obj, nx, ny, ppc, xbin, ybin, defaults, means,
                                                                  ranges, y_pred, batch, hybrid, sel_sigmoid, y_true_out, out6,
                                                                  grad, err);
    return spnet_check_launch("yolo_ellipse_loss_ann");
}

// uint8 frames -> fp32 network input on the device (spnet/utils.py:340-342). lut [256] fp32 = ((v/255)-0.5)*2 as numpy
// computes it in fp32; in / out must be 16-byte aligned.
int spnet_normalize_u8(const unsigned char* in, const float* lut, float* out, long long n, cudaStream_t stream) {
    SPNET_REQUIRE(in && lut && out && n > 0, "normalize_u8: bad args");
    SPNET_REQUIRE(((uintptr_t)in % 16 == 0) && ((uintptr_t)out % 16 == 0), "normalize_u8: pointers must be 16-byte aligned");
    const long long n16 = n / 16;
    const int ntail = (int)(n - n16 * 16);
    long long blocks = (n16 + 255) / 256;
    if (blocks > spnet_num_sms() * 8) blocks = spnet_num_sms() * 8;
    if (blocks < 1) blocks = 1;
    normalize_u8_kernel<<<(unsigned)blocks, 256, 0, stream>>>(reinterpret_cast<const uint4*>(in), lut,
                                                              reinterpret_cast<float4*>(out), n16, in + n16 * 16, out + n16 * 16,
                                                              ntail);
    return spnet_check_launch("normalize_u8");
}

}  // extern "C"
