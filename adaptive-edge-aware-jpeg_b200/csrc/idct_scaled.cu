// idct_scaled.cu -- DCT-domain scaled decode (aeaj_decode_scaled): every leaf of size s decodes straight to (s/m) x (s/m)
// samples of a 1/m plane, m = min(scale, block_min), from the top-left t x t (t = s/m) of its coefficients:
//     V = (1/m) C_t^T Y_t C_t,   Y_t = float(coef * q) over the top-left t x t, q the size-s table,
// C_t the orthonormal t-point DCT-II matrix.  The t-point DC term is t * mean and the s-point one s * mean, so the 1/m keeps each
// leaf's mean.  V / scale + mid (no fma) is stored at (y/m + r, x/m + c) for the rows / columns that cover the leaf's valid
// extent.  Where scale > block_min, k_box_reduce takes the 1/m planes to 1/scale with leaf-aligned box means.
//
//   t = 1       : one thread per leaf, the DC term only (C_1 = 1)
//   t <= 32     : t lanes per leaf, lane r owns row r (the layout of k_dct_rows, without its even / odd folding)
//   t >= 64     : one CTA per leaf, two register-blocked shared-memory GEMMs
// FP32 FMA accumulation in sequential order: the error bound of the full IDCT (DESIGN.md section 2) holds at size t.
#include "aeaj_internal.cuh"

namespace {

// the leaf's t x t input, dequantised: row-major blocks read (r, c) at r * s + c, zigzag-ordered blocks at izz[r * s + c]
__device__ __forceinline__ float scaled_coef(const PlaneDesc& P, const ClassEntry& e, const int* __restrict__ qt,
                                             const int* __restrict__ izz, int s, int r, int c) {
    const int nat = r * s + c;
    const int idx = P.zigzag ? __ldg(izz + nat) : nat;
    return (float)(__ldg(P.coef + (size_t)e.coef_off + idx) * __ldg(qt + nat));
}

// store sample (r, c) of the leaf's scaled block (v = C_t^T Y C_t, before the 1/m) if it covers the leaf's valid extent
__device__ __forceinline__ void scaled_store(const PlaneDesc& P, const ClassEntry& e, int m, float inv_m, int r, int c, float v) {
    const int hs = aeaj_cdiv(P.h, m), ws = aeaj_cdiv(P.w, m);
    const int ys = e.y / m + r, xs = e.x / m + c;
    if (ys < hs && xs < ws) P.layer_f32[(size_t)ys * ws + xs] = __fadd_rn(__fdiv_rn(__fmul_rn(v, inv_m), P.scale), P.mid);
}

// t = 1: V = Y[0][0] / m
__global__ void __launch_bounds__(256) k_idct_scaled_dc(const PlaneDesc* __restrict__ planes, const ClassEntry* __restrict__ list,
                                                        const int* __restrict__ count_ptr, int s, int lg, int m, float inv_m) {
    const int count = *count_ptr;
    for (int li = blockIdx.x * 256 + threadIdx.x; li < count; li += gridDim.x * 256) {
        const ClassEntry e = list[li];
        const PlaneDesc& P = planes[e.plane];
        scaled_store(P, e, m, inv_m, 0, 0, (float)(__ldg(P.coef + (size_t)e.coef_off) * __ldg(P.qtab[lg])));
    }
}

// 2 <= T <= 32: T lanes per leaf, 32 / T leaves per warp, 8 warps per block
template <int T>
__global__ void __launch_bounds__(256) k_idct_scaled_rows(const PlaneDesc* __restrict__ planes, const ClassEntry* __restrict__ list,
                                                          const int* __restrict__ count_ptr, int s, int lg, int m, float inv_m,
                                                          const float* __restrict__ Cg, const int* __restrict__ izz) {
    constexpr int LPW = 32 / T;
    constexpr int TS = (T >= 8) ? T + 1 : T;           // exchange-tile row stride: the column reads of pass 2 spread over banks
    __shared__ float sC[T * T];                        // C_t, row-major: sC[k * T + i] = C[k][i]
    __shared__ float sT[8][LPW * T * TS];
    for (int i = threadIdx.x; i < T * T; i += 256) sC[i] = Cg[i];
    __syncthreads();
    const int count = *count_ptr;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int sub = lane / T, r = lane % T;
    float crow[T];                                     // pass 2 of lane r: C[i][r], i < T
#pragma unroll
    for (int i = 0; i < T; i++) crow[i] = sC[i * T + r];
    const int groups = (count + LPW - 1) / LPW;
    for (int g = blockIdx.x * 8 + warp; g < groups; g += gridDim.x * 8) {
        const int li = g * LPW + sub;
        const bool act = li < count;
        ClassEntry e = {0, 0, 0, 0};
        if (act) e = list[li];
        const PlaneDesc& P = planes[e.plane];
        float in[T];
        if (act) {
            const int* qt = P.qtab[lg];
#pragma unroll
            for (int j = 0; j < T; j++) in[j] = scaled_coef(P, e, qt, izz, s, r, j);
        } else {
#pragma unroll
            for (int j = 0; j < T; j++) in[j] = 0.0f;
        }
        float* X = &sT[warp][sub * T * TS];
        // pass 1: U[r][l] = sum_j Y[r][j] C[j][l]
#pragma unroll
        for (int l = 0; l < T; l++) {
            float acc = 0.0f;
#pragma unroll
            for (int j = 0; j < T; j++) acc = __fmaf_rn(in[j], sC[j * T + l], acc);
            X[r * TS + l] = acc;
        }
        __syncwarp();
        // pass 2: V[r][l] = sum_i C[i][r] U[i][l]
        float out[T];
#pragma unroll
        for (int l = 0; l < T; l++) out[l] = 0.0f;
#pragma unroll
        for (int i = 0; i < T; i++) {
#pragma unroll
            for (int l = 0; l < T; l++) out[l] = __fmaf_rn(crow[i], X[i * TS + l], out[l]);
        }
        __syncwarp();                                  // the next group overwrites the tile
        if (act) {
#pragma unroll
            for (int l = 0; l < T; l++) scaled_store(P, e, m, inv_m, r, l, out[l]);
        }
    }
}

// T in {64, 128}: one CTA per leaf.  sY holds Y, then U = Y C; sC holds C.  256 threads as 16 x 16, each owning the rows
// tr + 16 a and the columns tc + 16 b (a, b < T / 16) of every product.
constexpr size_t scaled_cta_smem(int T) { return (size_t)(T * (T + 1) + T * T) * sizeof(float); }

template <int T>
__global__ void __launch_bounds__(256) k_idct_scaled_cta(const PlaneDesc* __restrict__ planes, const ClassEntry* __restrict__ list,
                                                         const int* __restrict__ count_ptr, int s, int lg, int m, float inv_m,
                                                         const float* __restrict__ Cg, const int* __restrict__ izz) {
    constexpr int N = T / 16, YS = T + 1;              // YS: row stride of Y / U
    extern __shared__ float smem[];
    float* sY = smem;                                  // [T][YS]
    float* sC = smem + T * YS;                         // [T][T]
    const int tid = threadIdx.x, tr = tid >> 4, tc = tid & 15;
    for (int i = tid; i < T * T; i += 256) sC[i] = Cg[i];
    const int count = *count_ptr;
    for (int li = blockIdx.x; li < count; li += gridDim.x) {
        const ClassEntry e = list[li];
        const PlaneDesc& P = planes[e.plane];
        const int* qt = P.qtab[lg];
        __syncthreads();                               // the previous leaf is done with sY (and sC is loaded)
        for (int i = tid; i < T * T; i += 256) {
            const int r = i / T, c = i - r * T;
            sY[r * YS + c] = scaled_coef(P, e, qt, izz, s, r, c);
        }
        __syncthreads();
        float acc[N][N];
#pragma unroll
        for (int a = 0; a < N; a++)
#pragma unroll
            for (int b = 0; b < N; b++) acc[a][b] = 0.0f;
        // pass 1: U[i][l] = sum_j Y[i][j] C[j][l]
        for (int j = 0; j < T; j++) {
            float av[N], bv[N];
#pragma unroll
            for (int a = 0; a < N; a++) av[a] = sY[(tr + 16 * a) * YS + j];
#pragma unroll
            for (int b = 0; b < N; b++) bv[b] = sC[j * T + tc + 16 * b];
#pragma unroll
            for (int a = 0; a < N; a++)
#pragma unroll
                for (int b = 0; b < N; b++) acc[a][b] = __fmaf_rn(av[a], bv[b], acc[a][b]);
        }
        __syncthreads();                               // everyone is done reading Y
#pragma unroll
        for (int a = 0; a < N; a++)
#pragma unroll
            for (int b = 0; b < N; b++) { sY[(tr + 16 * a) * YS + tc + 16 * b] = acc[a][b]; acc[a][b] = 0.0f; }
        __syncthreads();
        // pass 2: V[r][l] = sum_i C[i][r] U[i][l]
        for (int i = 0; i < T; i++) {
            float av[N], bv[N];
#pragma unroll
            for (int a = 0; a < N; a++) av[a] = sC[i * T + tr + 16 * a];
#pragma unroll
            for (int b = 0; b < N; b++) bv[b] = sY[i * YS + tc + 16 * b];
#pragma unroll
            for (int a = 0; a < N; a++)
#pragma unroll
                for (int b = 0; b < N; b++) acc[a][b] = __fmaf_rn(av[a], bv[b], acc[a][b]);
        }
#pragma unroll
        for (int a = 0; a < N; a++)
#pragma unroll
            for (int b = 0; b < N; b++) scaled_store(P, e, m, inv_m, tr + 16 * a, tc + 16 * b, acc[a][b]);
    }
}

// one image's plane [sh][sw] -> [dh][dw], dh = ceil(sh / f), dw = ceil(sw / f): the mean of the in-bounds cells of each
// f x f group, summed in row-major order; grid.y = the image of the batch
__global__ void __launch_bounds__(256) k_box_reduce(const float* __restrict__ src, int sh, int sw, float* __restrict__ dst,
                                                    int dh, int dw, int f) {
    const size_t b = blockIdx.y;
    const float* sp = src + b * sh * sw;
    float* dp = dst + b * dh * dw;
    for (int i = blockIdx.x * 256 + threadIdx.x; i < dh * dw; i += gridDim.x * 256) {
        const int oy = i / dw, ox = i - oy * dw;
        const int y0 = oy * f, x0 = ox * f, y1 = min(y0 + f, sh), x1 = min(x0 + f, sw);
        float acc = 0.0f;
        for (int y = y0; y < y1; y++)
            for (int x = x0; x < x1; x++) acc = __fadd_rn(acc, __ldg(sp + (size_t)y * sw + x));
        dp[i] = __fdiv_rn(acc, (float)((y1 - y0) * (x1 - x0)));
    }
}

template <int T>
int launch_rows_scaled(aeaj_handle* h, const PlaneDesc* planes_dev, const ClassEntry* list, const int* count, int64_t cap,
                       int s, int lg, int m, const int* izz, cudaStream_t st) {
    const int64_t groups = aeaj_cdiv64(cap, 32 / T);
    const int blocks = (int)std::max<int64_t>(1, std::min<int64_t>(aeaj_cdiv64(groups, 8), (int64_t)h->sm_count * 8));
    k_idct_scaled_rows<T><<<blocks, 256, 0, st>>>(planes_dev, list, count, s, lg, m, 1.0f / m, h->dct_dev[ilog2i(T)], izz);
    AEAJ_LAUNCH_CHECK();
    return 0;
}

template <int T>
int launch_cta_scaled(aeaj_handle* h, const PlaneDesc* planes_dev, const ClassEntry* list, const int* count, int64_t cap,
                      int s, int lg, int m, const int* izz, cudaStream_t st) {
    const size_t smem = scaled_cta_smem(T);            // opted in per device by aeaj_idct_scaled_init
    const int per_sm = smem > 110 * 1024 ? 1 : 2;
    const int blocks = (int)std::min<int64_t>(std::max<int64_t>(cap, 1), (int64_t)h->sm_count * per_sm);
    k_idct_scaled_cta<T><<<blocks, 256, smem, st>>>(planes_dev, list, count, s, lg, m, 1.0f / m, h->dct_dev[ilog2i(T)], izz);
    AEAJ_LAUNCH_CHECK();
    return 0;
}

}  // namespace

int aeaj_idct_scaled_init() {
    AEAJ_CUDA(cudaFuncSetAttribute(k_idct_scaled_cta<64>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)scaled_cta_smem(64)));
    AEAJ_CUDA(cudaFuncSetAttribute(k_idct_scaled_cta<128>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)scaled_cta_smem(128)));
    return 0;
}

int launch_idct_scaled(aeaj_handle* h, const PlaneDesc* planes_dev, const ClassEntry* class_lists, const int* class_counts,
                       const int64_t* off, const int64_t* caps, int lg_min, int lg_max, int m, cudaStream_t st, int* launches) {
    for (int lg = lg_min; lg <= lg_max; lg++) {
        if (caps[lg] <= 0) continue;
        const int s = 1 << lg, T = s / m;
        const ClassEntry* list = class_lists + off[lg];
        const int* cnt = class_counts + lg;
        const int* izz = h->izz_dev[lg];
        int rc = 0;
        switch (T) {
            case 1: {
                const int blocks = (int)std::max<int64_t>(1, std::min<int64_t>(aeaj_cdiv64(caps[lg], 256), (int64_t)h->sm_count * 8));
                k_idct_scaled_dc<<<blocks, 256, 0, st>>>(planes_dev, list, cnt, s, lg, m, 1.0f / m);
                AEAJ_LAUNCH_CHECK();
                break;
            }
            case 2: rc = launch_rows_scaled<2>(h, planes_dev, list, cnt, caps[lg], s, lg, m, izz, st); break;
            case 4: rc = launch_rows_scaled<4>(h, planes_dev, list, cnt, caps[lg], s, lg, m, izz, st); break;
            case 8: rc = launch_rows_scaled<8>(h, planes_dev, list, cnt, caps[lg], s, lg, m, izz, st); break;
            case 16: rc = launch_rows_scaled<16>(h, planes_dev, list, cnt, caps[lg], s, lg, m, izz, st); break;
            case 32: rc = launch_rows_scaled<32>(h, planes_dev, list, cnt, caps[lg], s, lg, m, izz, st); break;
            case 64: rc = launch_cta_scaled<64>(h, planes_dev, list, cnt, caps[lg], s, lg, m, izz, st); break;
            case 128: rc = launch_cta_scaled<128>(h, planes_dev, list, cnt, caps[lg], s, lg, m, izz, st); break;
            default: aeaj_set_error("scaled IDCT: output size %d per leaf not supported (1..128)", T); return AEAJ_EINVAL;
        }
        if (rc) return rc;
        if (launches) (*launches)++;
    }
    return 0;
}

int launch_box_reduce(const float* src, int sh, int sw, float* dst, int dh, int dw, int f, int batch, cudaStream_t st) {
    const dim3 grd((unsigned)std::max(1, std::min(aeaj_cdiv(dh * dw, 256), 4096)), (unsigned)batch);
    k_box_reduce<<<grd, 256, 0, st>>>(src, sh, sw, dst, dh, dw, f);
    AEAJ_LAUNCH_CHECK();
    return 0;
}
