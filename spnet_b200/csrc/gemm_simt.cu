// Exact-fp32 GEMM on the CUDA cores (FFMA, fp32 accumulate) with arbitrary operand
// strides. It is the fp32-mode engine behind the same layers gemm_tc.cu serves in bf16
// mode (the reference network runs fp32: spnet/config.py:4), so that "fp32 within 1e-4"
// parity can be checked without tensor-core rounding.
//
//   D[M,N] (op)= sum_k A(r,k) * B(n,k),  A(r,k) = A[r*sa_r + k*sa_k],  B(n,k) = B[n*sb_r + k*sb_k]
#include "common.cuh"

namespace {

constexpr int TM = 64, TN = 64, TK = 16, PAD = 4;

enum { OUT_T = 0, OUT_F32 = 1, OUT_ATOMIC_F32 = 2, OUT_SLAB_F32 = 3 };

__global__ void __launch_bounds__(256) gemm_simt_kernel(const float* __restrict__ A, long long sa_r, long long sa_k,
                                                        const float* __restrict__ B, long long sb_r, long long sb_k,
                                                        float* __restrict__ D, long long ldd, long long slab_stride,
                                                        int out_mode, int M, int N, int K, int k_per_split,
                                                        long long* __restrict__ colstats) {
    __shared__ float As[TK][TM + PAD];
    __shared__ float Bs[TK][TN + PAD];
    __shared__ float cs[16][2][TN];  // per thread-row partial column sums, added in row order (run-to-run identical)
    const int tid = threadIdx.x, tx = tid & 15, ty = tid >> 4;
    const int m0 = blockIdx.y * TM, n0 = blockIdx.x * TN;
    const int kbeg = blockIdx.z * k_per_split;
    const int kend = min(K, kbeg + k_per_split);
    const bool a_kfast = (sa_k == 1), b_kfast = (sb_k == 1);

    float acc[4][4];
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[i][j] = 0.f;

    for (int k0 = kbeg; k0 < kend; k0 += TK) {
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            const int e = tid + i * 256;
            int r, k;
            if (a_kfast) { k = e & (TK - 1); r = e >> 4; } else { r = e & (TM - 1); k = e >> 6; }
            float v = 0.f;
            if (m0 + r < M && k0 + k < kend) v = A[(long long)(m0 + r) * sa_r + (long long)(k0 + k) * sa_k];
            As[k][r] = v;
            if (b_kfast) { k = e & (TK - 1); r = e >> 4; } else { r = e & (TN - 1); k = e >> 6; }
            v = 0.f;
            if (n0 + r < N && k0 + k < kend) v = B[(long long)(n0 + r) * sb_r + (long long)(k0 + k) * sb_k];
            Bs[k][r] = v;
        }
        __syncthreads();
#pragma unroll
        for (int kk = 0; kk < TK; ++kk) {
            const float4 a4 = *reinterpret_cast<const float4*>(&As[kk][ty * 4]);
            const float4 b4 = *reinterpret_cast<const float4*>(&Bs[kk][tx * 4]);
            const float a[4] = {a4.x, a4.y, a4.z, a4.w};
            const float b[4] = {b4.x, b4.y, b4.z, b4.w};
#pragma unroll
            for (int i = 0; i < 4; ++i)
#pragma unroll
                for (int j = 0; j < 4; ++j) acc[i][j] = fmaf(a[i], b[j], acc[i][j]);
        }
        __syncthreads();
    }

    float csum[4] = {0.f, 0.f, 0.f, 0.f}, csq[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        const int r = m0 + ty * 4 + i;
        if (r >= M) continue;
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const int c = n0 + tx * 4 + j;
            if (c >= N) continue;
            float v = acc[i][j];
            if (out_mode == OUT_T) {  // D in the operands' type: fp32, the same store as OUT_F32
                D[(long long)r * ldd + c] = v;
            } else if (out_mode == OUT_F32) {
                D[(long long)r * ldd + c] = v;
            } else if (out_mode == OUT_SLAB_F32) {  // split z keeps its partial in its own slab (fixed-order split-K)
                D[(long long)blockIdx.z * slab_stride + (long long)r * ldd + c] = v;
            } else {
                atomicAdd(D + (long long)r * ldd + c, v);
            }
            csum[j] += v;
            csq[j] = fmaf(v, v, csq[j]);
        }
    }
    if (colstats) {
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            cs[ty][0][tx * 4 + j] = csum[j];
            cs[ty][1][tx * 4 + j] = csq[j];
        }
        __syncthreads();
        if (tid < TN && n0 + tid < N) {
            float t0 = 0.f, t1 = 0.f;
            for (int r_ = 0; r_ < 16; ++r_) { t0 += cs[r_][0][tid]; t1 += cs[r_][1][tid]; }
            stat_add(colstats, n0 + tid, (double)t0);
            stat_add(colstats, N + n0 + tid, (double)t1);
        }
    }
}

}  // namespace

extern "C" {

// A, B and D are fp32 in every out_mode.
int spnet_gemm_simt(const float* A, long long sa_r, long long sa_k, const float* B, long long sb_r, long long sb_k,
                    float* D, long long ldd, long long slab_stride, int out_mode, int M, int N, int K, int splits,
                    long long* colstats, cudaStream_t stream) {
    SPNET_REQUIRE(A && B && D, "gemm_simt: null pointer");
    SPNET_REQUIRE(M > 0 && N > 0 && K > 0, "gemm_simt: bad shape %d %d %d", M, N, K);
    SPNET_REQUIRE(out_mode >= 0 && out_mode <= 3, "gemm_simt: bad out_mode");
    SPNET_REQUIRE(splits <= 1 || out_mode == OUT_ATOMIC_F32 || out_mode == OUT_SLAB_F32, "gemm_simt: split-K needs out_mode 2 or 3");
    SPNET_REQUIRE(!(colstats && splits > 1), "gemm_simt: column statistics are not defined for split-K partials");
    if (splits < 1) splits = 1;
    SPNET_REQUIRE(out_mode != OUT_SLAB_F32 || slab_stride > 0, "gemm_simt: out_mode 3 needs slab_stride");
    int kps = ceil_div(ceil_div(K, splits), TK) * TK;
    splits = ceil_div(K, kps);
    dim3 grid(ceil_div(N, TN), ceil_div(M, TM), splits);
    SPNET_REQUIRE(grid.y <= 65535 && grid.z <= 65535, "gemm_simt: grid too large");
    gemm_simt_kernel<<<grid, 256, 0, stream>>>(A, sa_r, sa_k, B, sb_r, sb_k, D, ldd, slab_stride, out_mode, M, N, K, kps,
                                               colstats);
    return spnet_check_launch("gemm_simt");
}

}  // extern "C"
