// dct.cu -- variable-size 2-D DCT/IDCT with fused (de)normalisation, reflect-padded leaf
// extraction, quantisation and dequantisation (jpeg.py:387-404, 461-529, 410-459) for sm_100a.
//
// Work arrives as per-size-class lists of leaves (quadtree.cu).  Both directions are the same
// product  Out = M . In . M^T  with M = C (forward, cv.dct) or M = C^T (inverse, cv.idct), where
// C[k][i] = sqrt(2/s) cos(pi (2i+1) k / 2s), row 0 scaled by 1/sqrt 2, evaluated in f64 on the host
// and stored as f32.  FP32 FMA accumulation: SURVEY.md App. A5 measured 0 quantiser flips against
// cv.dct for an f32 matrix DCT (tie class T-DCT), which is the parity bar.  Plain TF32 tensor-core tiles do
// not hold that bar; the error-compensated 3xTF32 tcgen05 kernels that do are in dct_tc.cu (the default for the
// size classes they cover) and the kernels of this file serve the small classes and the FP32 reference path.
//
//   s <= 32 : "row" kernel -- s lanes per leaf, lane r owns row r; pass 1 in registers against
//             broadcast reads of M from shared memory, exchange through a per-warp shared tile,
//             pass 2 with the lane's own M row in registers; stores are fully coalesced rows.
//   s >= 64 : "cta" kernel -- one CTA per leaf, two register-blocked shared-memory GEMMs
//             (V = M.In, Out = V.M^T) with the intermediate kept transposed in shared memory.
// Quantise: rint(double(coef)/double(q)) half-even (np.round of an f64 quotient, jpeg.py:501);
// dequantise: float(int32*int32) (jpeg.py:524); normalise (v-m)*s, denormalise n/s+m, no fma.
#include "aeaj_internal.cuh"

namespace {

// quantize(): the exact float32 quantiser, see aeaj_internal.cuh

// ---------------------------------------------------------------------------------------------
// row kernel, S in {2,4,8,16,32}; block = 256 threads = 8 warps; each warp handles 32/S leaves.
// ---------------------------------------------------------------------------------------------
template <int S, bool INVERSE>
__global__ void __launch_bounds__(256) k_dct_rows(const PlaneDesc* __restrict__ planes, const ClassEntry* __restrict__ list,
                                                  const int* __restrict__ count_ptr, const float* __restrict__ Mg, const float* __restrict__ Mtg) {
    constexpr int LPW = 32 / S;                        // leaves per warp
    constexpr int LG = (S == 2) ? 1 : (S == 4) ? 2 : (S == 8) ? 3 : (S == 16) ? 4 : 5;
    __shared__ __align__(16) float sM[S * S];          // M   (row-major)
    __shared__ __align__(16) float sMt[S * S];         // M^T (row-major)
    // exchange tiles: row stride TS (16 B aligned, spreads the pass-1 column stores over banks) and
    // a per-leaf stride GS chosen so that the LPW leaves of a warp start in different bank groups
    constexpr int TS = (S >= 8) ? S + 4 : S;
    constexpr int GS = S * TS + ((LPW > 1) ? ((32 / LPW) - (S * TS) % 32 + 32) % 32 : 0);
    __shared__ __align__(16) float sT[8][LPW * GS + 4];
    for (int i = threadIdx.x; i < S * S; i += 256) { sM[i] = Mg[i]; sMt[i] = Mtg[i]; }
    __syncthreads();
    const int count = *count_ptr;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int sub = lane / S, r = lane % S;            // leaf slot in warp, row in leaf
    // S >= 16 uses the even / odd symmetry of the DCT matrix, C[k][S-1-i] = (-1)^k C[k][i], in both passes: half the FMAs
    // and half the shared-memory reads of the matrix (the passes are bound by shared-memory latency, not by HBM).
    constexpr bool EO = (S >= 16);
    constexpr int Hh = S / 2;
    // pass-2 coefficients of this lane.  plain: M[r][i], i < S.  EO forward (lane = frequency k): C[k][i], i < S/2.
    // EO inverse (lane pair i, S-1-i; the low lane sums the even k, the high lane the odd k): C[2kk+par][min(i, S-1-i)].
    float mrow[EO ? Hh : S];
    if (!EO) {
#pragma unroll
        for (int i = 0; i < S; i++) mrow[i] = sMt[i * S + r];
    } else if (!INVERSE) {
#pragma unroll
        for (int i = 0; i < Hh; i++) mrow[i] = sMt[i * S + r];
    } else {
        const int rlo = min(r, S - 1 - r), par = (r < Hh) ? 0 : 1;
#pragma unroll
        for (int kk = 0; kk < Hh; kk++) mrow[kk] = sMt[(2 * kk + par) * S + rlo];
    }
    const int groups = (count + LPW - 1) / LPW;        // warp-sized groups of leaves
    for (int g = blockIdx.x * 8 + warp; g < groups; g += gridDim.x * 8) {
        const int li = g * LPW + sub;
        bool act = li < count;
        ClassEntry e = {0, 0, 0, 0};
        if (act) e = list[li];
        const PlaneDesc& P = planes[e.plane];
        act = act && e.y >= P.ry0 && e.y < P.ry1;      // halo-split: only the leaves of this call's band
        float in[S];
        if (act) {
            if (!INVERSE) {
                const int bh = min(S, P.h - e.y), bw = min(S, P.w - e.x);
                const float* row = P.layer_f32 + (size_t)(e.y + pad_reflect(r, bh)) * P.w + e.x;
                const float mid = P.mid, sc = P.scale;
                if (bw == S && S >= 4 && ((P.w & 3) == 0)) {
#pragma unroll
                    for (int j = 0; j < S; j += 4) {
                        float4 v = __ldg(reinterpret_cast<const float4*>(row + j));
                        in[j] = v.x; in[j + 1] = v.y; in[j + 2] = v.z; in[j + 3] = v.w;
                    }
                } else {
#pragma unroll
                    for (int j = 0; j < S; j++) in[j] = __ldg(row + pad_reflect(j, bw));
                }
#pragma unroll
                for (int j = 0; j < S; j++) in[j] = __fmul_rn(__fsub_rn(in[j], mid), sc);
            } else if (!P.zigzag) {
                const int* cf = P.coef + (size_t)e.coef_off + r * S;
                const int* qt = P.qtab[LG] + r * S;
                if (S >= 4) {
#pragma unroll
                    for (int j = 0; j < S; j += 4) {
                        int4 cv = __ldg(reinterpret_cast<const int4*>(cf + j)), qv = __ldg(reinterpret_cast<const int4*>(qt + j));
                        in[j] = (float)(cv.x * qv.x); in[j + 1] = (float)(cv.y * qv.y); in[j + 2] = (float)(cv.z * qv.z); in[j + 3] = (float)(cv.w * qv.w);
                    }
                } else {
#pragma unroll
                    for (int j = 0; j < S; j++) in[j] = (float)(__ldg(cf + j) * __ldg(qt + j));
                }
            }
        } else {
#pragma unroll
            for (int j = 0; j < S; j++) in[j] = 0.0f;
        }
        float* T = &sT[warp][sub * GS];
        if (INVERSE && P.zigzag) {
            // zigzag-ordered stream: coalesced read, scatter through the warp tile into row-major, then dequantise
            __syncwarp();
            if (act) {
                const int* cf = P.coef + (size_t)e.coef_off;
                const int* qt = P.qtab[LG];
                const int* zz = P.zz[LG];
#pragma unroll
                for (int k = 0; k < S; k++) {
                    const int idx = r + k * S, nat = __ldg(zz + idx);
                    T[(nat / S) * TS + (nat % S)] = (float)(__ldg(cf + idx) * __ldg(qt + nat));
                }
            }
            __syncwarp();
#pragma unroll
            for (int j = 0; j < S; j++) in[j] = act ? T[r * TS + j] : 0.0f;
            __syncwarp();
        }
        float out[S];
        if (!EO) {
            // pass 1: t[l] = sum_j in[j] * M[l][j]
#pragma unroll
            for (int l = 0; l < S; l++) {
                float acc = 0.0f;
#pragma unroll
                for (int j = 0; j < S; j++) acc = __fmaf_rn(in[j], sM[l * S + j], acc);
                T[r * TS + l] = acc;
            }
            __syncwarp();
            // pass 2: out[l] = sum_i M[r][i] * T[i][l]
#pragma unroll
            for (int l = 0; l < S; l++) out[l] = 0.0f;
#pragma unroll
            for (int i = 0; i < S; i++) {
#pragma unroll
                for (int l = 0; l < S; l++) out[l] = __fmaf_rn(mrow[i], T[i * TS + l], out[l]);
            }
        } else if (!INVERSE) {
            // pass 1 (rows): fold the input, t[2m] = sum_{j<h} (x[j] + x[S-1-j]) C[2m][j], t[2m+1] = sum_{j<h} (x[j] - x[S-1-j]) C[2m+1][j]
            float u[Hh], d[Hh];
#pragma unroll
            for (int j = 0; j < Hh; j++) { u[j] = __fadd_rn(in[j], in[S - 1 - j]); d[j] = __fsub_rn(in[j], in[S - 1 - j]); }
#pragma unroll
            for (int m = 0; m < Hh; m++) {
                float ae = 0.0f, ao = 0.0f;
#pragma unroll
                for (int j = 0; j < Hh; j++) { ae = __fmaf_rn(u[j], sM[(2 * m) * S + j], ae); ao = __fmaf_rn(d[j], sM[(2 * m + 1) * S + j], ao); }
                T[r * TS + 2 * m] = ae; T[r * TS + 2 * m + 1] = ao;
            }
            __syncwarp();
            // fold the rows of the intermediate in place: row i <- T[i] + T[S-1-i], row S-1-i <- T[i] - T[S-1-i]; the two lanes
            // of a row pair take half the columns each
            {
                const int rlo = min(r, S - 1 - r), rhi = S - 1 - rlo, c0 = (r < Hh) ? 0 : Hh;
#pragma unroll
                for (int l = 0; l < Hh; l += 4) {
                    float4 a = *reinterpret_cast<const float4*>(T + rlo * TS + c0 + l), b = *reinterpret_cast<const float4*>(T + rhi * TS + c0 + l);
                    *reinterpret_cast<float4*>(T + rlo * TS + c0 + l) = make_float4(__fadd_rn(a.x, b.x), __fadd_rn(a.y, b.y), __fadd_rn(a.z, b.z), __fadd_rn(a.w, b.w));
                    *reinterpret_cast<float4*>(T + rhi * TS + c0 + l) = make_float4(__fsub_rn(a.x, b.x), __fsub_rn(a.y, b.y), __fsub_rn(a.z, b.z), __fsub_rn(a.w, b.w));
                }
            }
            __syncwarp();
            // pass 2 (columns): lane = frequency k; even k reads the sum rows (0 .. h-1), odd k the difference rows (S-1 .. h)
            const float* Tb = (r & 1) ? (T + (S - 1) * TS) : T;
            const int step = (r & 1) ? -TS : TS;
#pragma unroll
            for (int l = 0; l < S; l++) out[l] = 0.0f;
#pragma unroll
            for (int i = 0; i < Hh; i++) {
#pragma unroll
                for (int l = 0; l < S; l++) out[l] = __fmaf_rn(mrow[i], Tb[i * step + l], out[l]);
            }
        } else {
            // pass 1 (rows): E[l] = sum_{j even} z[j] C[j][l], O[l] = sum_{j odd} z[j] C[j][l] (l < h); t[l] = E + O, t[S-1-l] = E - O
#pragma unroll
            for (int l = 0; l < Hh; l++) {
                float ae = 0.0f, ao = 0.0f;
#pragma unroll
                for (int j = 0; j < S; j += 2) { ae = __fmaf_rn(in[j], sM[l * S + j], ae); ao = __fmaf_rn(in[j + 1], sM[l * S + j + 1], ao); }
                T[r * TS + l] = __fadd_rn(ae, ao); T[r * TS + S - 1 - l] = __fsub_rn(ae, ao);
            }
            __syncwarp();
            // pass 2 (columns): the lane pair (i, S-1-i) shares the work -- the low lane sums the even k, the high lane the odd k
            const int par = (r < Hh) ? 0 : 1;
            float acc[S];
#pragma unroll
            for (int l = 0; l < S; l++) acc[l] = 0.0f;
#pragma unroll
            for (int kk = 0; kk < Hh; kk++) {
                const float* Tk = T + (2 * kk) * TS + par * TS;
#pragma unroll
                for (int l = 0; l < S; l++) acc[l] = __fmaf_rn(mrow[kk], Tk[l], acc[l]);
            }
#pragma unroll
            for (int l = 0; l < S; l++) {
                const float other = __shfl_xor_sync(0xffffffffu, acc[l], S - 1);
                out[l] = par ? __fsub_rn(other, acc[l]) : __fadd_rn(acc[l], other);     // row i: E + O, row S-1-i: E - O
            }
        }
        __syncwarp();
        if (act) {
            if (!INVERSE && P.zigzag) {
                // stage the quantised row in the warp tile, then the S lanes of the leaf write the block in zigzag order
                const int* qt = P.qtab[LG] + r * S;
                int* Ti = reinterpret_cast<int*>(T);
#pragma unroll
                for (int l = 0; l < S; l++) Ti[r * TS + l] = quantize(out[l], __ldg(qt + l));
            } else if (!INVERSE) {
                int* cf = P.coef + (size_t)e.coef_off + r * S;
                const int* qt = P.qtab[LG] + r * S;
                if (S >= 4) {
#pragma unroll
                    for (int l = 0; l < S; l += 4) {
                        int4 qv = __ldg(reinterpret_cast<const int4*>(qt + l));
                        *reinterpret_cast<int4*>(cf + l) = make_int4(quantize(out[l], qv.x), quantize(out[l + 1], qv.y), quantize(out[l + 2], qv.z), quantize(out[l + 3], qv.w));
                    }
                } else {
#pragma unroll
                    for (int l = 0; l < S; l++) cf[l] = quantize(out[l], __ldg(qt + l));
                }
            } else {
                const int y = e.y + r;
                if (y < P.h) {
                    float* row = P.layer_f32 + (size_t)y * P.w + e.x;
                    const int bw = min(S, P.w - e.x);
                    const float mid = P.mid, sc = P.scale;
                    if (bw == S && S >= 4 && ((P.w & 3) == 0)) {
#pragma unroll
                        for (int l = 0; l < S; l += 4)
                            *reinterpret_cast<float4*>(row + l) = make_float4(__fadd_rn(__fdiv_rn(out[l], sc), mid), __fadd_rn(__fdiv_rn(out[l + 1], sc), mid),
                                                                              __fadd_rn(__fdiv_rn(out[l + 2], sc), mid), __fadd_rn(__fdiv_rn(out[l + 3], sc), mid));
                    } else {
#pragma unroll
                        for (int l = 0; l < S; l++)
                            if (l < bw) row[l] = __fadd_rn(__fdiv_rn(out[l], sc), mid);
                    }
                }
            }
        }
        if (!INVERSE && P.zigzag) {
            __syncwarp();
            if (act) {
                int* cf = P.coef + (size_t)e.coef_off;
                const int* zz = P.zz[LG];
                const int* Ti = reinterpret_cast<const int*>(T);
#pragma unroll
                for (int k = 0; k < S; k++) {
                    const int idx = r + k * S, nat = __ldg(zz + idx);
                    cf[idx] = Ti[(nat / S) * TS + (nat % S)];
                }
            }
            __syncwarp();
        }
    }
}

// ---------------------------------------------------------------------------------------------
// CTA kernel, S in {64,128}: one CTA (256 threads) per leaf, FP32 FMA, using the even/odd symmetry of
// the DCT matrix, C[k][N-1-i] = (-1)^k C[k][i]: with Ce[m][i] = C[2m][i], Co[m][i] = C[2m+1][i]
// (m, i < h = N/2) every 1-D transform is two h x h products on folded data -- half the FLOPs.
//
//   forward  (cv.dct):  U = X[i]+X[N-1-i], D = X[i]-X[N-1-i] (fold rows while loading);
//                       V[2m] = Ce.U, V[2m+1] = Co.D; fold V's columns in registers;
//                       Out[k][2m] = sum_j P[k][j] Ce[m][j], Out[k][2m+1] = sum_j Q[k][j] Co[m][j]
//   inverse  (cv.idct): E = Ce^T.Z[even rows], O = Co^T.Z[odd rows]; V[i] = E+O, V[N-1-i] = E-O;
//                       E' = V[:, even].Ce, O' = V[:, odd].Co; X[i][j] = E'+O', X[i][N-1-j] = E'-O'
//
// Thread t: parity g = t & 1 (even / odd half), pair p = t >> 1.  The two lanes of a pair hold the even
// and the odd partial results for the same tile and exchange them with __shfl_xor(.., 1).
// Shared memory: sA = [Ae | Ao] (2 x h x h: the half matrices in the orientation the pass needs),
// sB = N x N staging (folded input, then the transposed intermediate).  1.5 N^2 floats = 96 KB at N=128.
// ---------------------------------------------------------------------------------------------
template <int S, bool INVERSE>
__global__ void __launch_bounds__(256) k_dct_cta(const PlaneDesc* __restrict__ planes, const ClassEntry* __restrict__ list,
                                                 const int* __restrict__ count_ptr, const float* __restrict__ half_tab) {
    constexpr int N = S, Hh = S / 2;
    constexpr int LG = (S == 64) ? 6 : 7;
    constexpr int T = S / 16;                          // tile edge per thread: 8 (N=128) or 4 (N=64)
    constexpr int RC = T / 4;                          // number of 4-wide chunks along the "4-chunk" axis
    constexpr int CW = T / 2;                          // width of the two mirrored column chunks (forward pass 1)
    // Bank-conflict avoidance: the odd halves start 16 floats later than a multiple of 32 (the even / odd lanes
    // of a pair read the same offsets of the two halves), and staging rows are NS = N + 4 floats apart (the
    // transposed stores walk down a column).
    constexpr int NS = N + 4, PAD = 16;
    extern __shared__ __align__(16) float smem[];
    float* sA = smem;                                  // even half matrix [Hh][Hh]
    float* sAo = sA + Hh * Hh + PAD;                   // odd half matrix
    float* sB = sAo + Hh * Hh + PAD;                   // staging, first Hh rows  [Hh][NS]
    float* sBo = sB + Hh * NS + PAD;                   // staging, second Hh rows [Hh][NS]
    const int tid = threadIdx.x, g = tid & 1, p = tid >> 1;
    for (int i = tid; i < Hh * Hh / 4; i += 256) {
        reinterpret_cast<float4*>(sA)[i] = __ldg(reinterpret_cast<const float4*>(half_tab) + i);
        reinterpret_cast<float4*>(sAo)[i] = __ldg(reinterpret_cast<const float4*>(half_tab + Hh * Hh) + i);
    }
    const float* sAg = g ? sAo : sA;
    const int count = *count_ptr;
    // pass-1 tile: rows (h of them) in chunks of 4 at stride 32, columns (N of them)
    const int tr = p / 16, tc = p % 16;
    // pass-2 tile: rows (N of them) in chunks of 4 at stride 64, columns (h of them) in chunks of 4 at stride 32
    const int tr2 = p / 8, tc2 = p % 8;
    for (int li = blockIdx.x; li < count; li += gridDim.x) {
        const ClassEntry e = list[li];
        const PlaneDesc& P = planes[e.plane];
        if (e.y < P.ry0 || e.y >= P.ry1) continue;     // halo-split: only the leaves of this call's band (uniform per CTA)
        __syncthreads();                               // previous leaf done with sB
        if (!INVERSE) {
            // load X, fold rows: sB[i][j] = X[i][j] + X[N-1-i][j] (i < h), sB[h+i][j] = X[i][j] - X[N-1-i][j]
            const int bh = min(N, P.h - e.y), bw = min(N, P.w - e.x);
            const float mid = P.mid, sc = P.scale;
            if (bh == N && bw == N && (P.w & 3) == 0) {
                // full leaf: 128-bit loads of rows rr and N-1-rr
                for (int i = tid; i < Hh * N / 4; i += 256) {
                    const int rr = (i * 4) / N, cc = (i * 4) - rr * N;
                    const float4 a = __ldg(reinterpret_cast<const float4*>(P.layer_f32 + (size_t)(e.y + rr) * P.w + e.x + cc));
                    const float4 b = __ldg(reinterpret_cast<const float4*>(P.layer_f32 + (size_t)(e.y + N - 1 - rr) * P.w + e.x + cc));
                    const float a0 = __fmul_rn(__fsub_rn(a.x, mid), sc), a1 = __fmul_rn(__fsub_rn(a.y, mid), sc), a2 = __fmul_rn(__fsub_rn(a.z, mid), sc), a3 = __fmul_rn(__fsub_rn(a.w, mid), sc);
                    const float b0 = __fmul_rn(__fsub_rn(b.x, mid), sc), b1 = __fmul_rn(__fsub_rn(b.y, mid), sc), b2 = __fmul_rn(__fsub_rn(b.z, mid), sc), b3 = __fmul_rn(__fsub_rn(b.w, mid), sc);
                    *reinterpret_cast<float4*>(sB + rr * NS + cc) = make_float4(__fadd_rn(a0, b0), __fadd_rn(a1, b1), __fadd_rn(a2, b2), __fadd_rn(a3, b3));
                    *reinterpret_cast<float4*>(sBo + rr * NS + cc) = make_float4(__fsub_rn(a0, b0), __fsub_rn(a1, b1), __fsub_rn(a2, b2), __fsub_rn(a3, b3));
                }
            } else {
                for (int i = tid; i < Hh * N; i += 256) {
                    const int rr = i / N, cc = i - rr * N;
                    const int xx = e.x + pad_reflect(cc, bw);
                    float a = __ldg(P.layer_f32 + (size_t)(e.y + pad_reflect(rr, bh)) * P.w + xx);
                    float b = __ldg(P.layer_f32 + (size_t)(e.y + pad_reflect(N - 1 - rr, bh)) * P.w + xx);
                    a = __fmul_rn(__fsub_rn(a, mid), sc); b = __fmul_rn(__fsub_rn(b, mid), sc);
                    sB[rr * NS + cc] = __fadd_rn(a, b); sBo[rr * NS + cc] = __fsub_rn(a, b);
                }
            }
        } else {
            // load Z dequantised, rows in split order: even rows first, then odd rows
            const int* cf = P.coef + (size_t)e.coef_off;
            const int* qt = P.qtab[LG];
            if (P.zigzag) {
                const int* zz = P.zz[LG];
                for (int i = tid; i < N * N; i += 256) {
                    const int nat = __ldg(zz + i), k = nat / N, l = nat - k * N;
                    (((k & 1) ? sBo : sB) + (k >> 1) * NS)[l] = (float)(__ldg(cf + i) * __ldg(qt + nat));
                }
            } else {
                for (int i = tid; i < N * N / 4; i += 256) {
                    const int k = (i * 4) / N, l = (i * 4) - k * N;
                    int4 cv = __ldg(reinterpret_cast<const int4*>(cf) + i), qv = __ldg(reinterpret_cast<const int4*>(qt) + i);
                    *reinterpret_cast<float4*>(((k & 1) ? sBo : sB) + (k >> 1) * NS + l) =
                        make_float4((float)(cv.x * qv.x), (float)(cv.y * qv.y), (float)(cv.z * qv.z), (float)(cv.w * qv.w));
                }
            }
        }
        __syncthreads();
        float acc[T][T];
#pragma unroll
        for (int a = 0; a < T; a++)
#pragma unroll
            for (int b = 0; b < T; b++) acc[a][b] = 0.0f;
        const float* sBg = g ? sBo : sB;
        if (!INVERSE) {
            // pass 1: Vg[m][j] = sum_i Cg[m][i] * Fg[i][j]; sAg[i][m] = Cg[m][i]; columns = two mirrored chunks
            for (int i = 0; i < Hh; i++) {
                float av[T], bv[T];
#pragma unroll
                for (int c = 0; c < RC; c++) { float4 t = *reinterpret_cast<const float4*>(sAg + i * Hh + tr * 4 + c * 32); av[4 * c] = t.x; av[4 * c + 1] = t.y; av[4 * c + 2] = t.z; av[4 * c + 3] = t.w; }
                if (CW == 4) {
                    float4 t = *reinterpret_cast<const float4*>(sBg + i * NS + tc * 4);
                    float4 u = *reinterpret_cast<const float4*>(sBg + i * NS + N - 4 - tc * 4);
                    bv[0] = t.x; bv[1] = t.y; bv[2] = t.z; bv[3] = t.w; bv[4] = u.w; bv[5] = u.z; bv[6] = u.y; bv[7] = u.x;
                } else {
                    float2 t = *reinterpret_cast<const float2*>(sBg + i * NS + tc * 2);
                    float2 u = *reinterpret_cast<const float2*>(sBg + i * NS + N - 2 - tc * 2);
                    bv[0] = t.x; bv[1] = t.y; bv[2] = u.y; bv[3] = u.x;
                }
#pragma unroll
                for (int a = 0; a < T; a++)
#pragma unroll
                    for (int b = 0; b < T; b++) acc[a][b] = __fmaf_rn(av[a], bv[b], acc[a][b]);
            }
            __syncthreads();                           // everyone finished reading the folded input
            // fold V's columns in registers and store transposed, rows in split order k' = g*h + m:
            //   sB[j][k']       = P[k][j] = V[k][j] + V[k][N-1-j]      (j < h)
            //   sB[h + j][k']   = Q[k][j] = V[k][j] - V[k][N-1-j]
#pragma unroll
            for (int b = 0; b < CW; b++) {
                const int j = tc * CW + b;
#pragma unroll
                for (int c = 0; c < RC; c++) {
                    float pv[4], qv[4];
#pragma unroll
                    for (int a = 0; a < 4; a++) { pv[a] = __fadd_rn(acc[4 * c + a][b], acc[4 * c + a][b + CW]); qv[a] = __fsub_rn(acc[4 * c + a][b], acc[4 * c + a][b + CW]); }
                    const int kk = g * Hh + tr * 4 + c * 32;
                    *reinterpret_cast<float4*>(sB + j * NS + kk) = make_float4(pv[0], pv[1], pv[2], pv[3]);
                    *reinterpret_cast<float4*>(sBo + j * NS + kk) = make_float4(qv[0], qv[1], qv[2], qv[3]);
                }
            }
            __syncthreads();
#pragma unroll
            for (int a = 0; a < T; a++)
#pragma unroll
                for (int b = 0; b < T; b++) acc[a][b] = 0.0f;
            // pass 2: Out[k'][2m+g] = sum_j F2g[j][k'] * Cg[m][j]   (F2e = P, F2o = Q; sAg[j][m] = Cg[m][j])
            for (int j = 0; j < Hh; j++) {
                float av[T], bv[T];
#pragma unroll
                for (int c = 0; c < RC; c++) { float4 t = *reinterpret_cast<const float4*>(sBg + j * NS + tr2 * 4 + c * 64); av[4 * c] = t.x; av[4 * c + 1] = t.y; av[4 * c + 2] = t.z; av[4 * c + 3] = t.w; }
#pragma unroll
                for (int c = 0; c < RC; c++) { float4 t = *reinterpret_cast<const float4*>(sAg + j * Hh + tc2 * 4 + c * 32); bv[4 * c] = t.x; bv[4 * c + 1] = t.y; bv[4 * c + 2] = t.z; bv[4 * c + 3] = t.w; }
#pragma unroll
                for (int a = 0; a < T; a++)
#pragma unroll
                    for (int b = 0; b < T; b++) acc[a][b] = __fmaf_rn(av[a], bv[b], acc[a][b]);
            }
            // quantise, interleave even/odd columns with the pair lane, store int4
            int* cf = P.coef + (size_t)e.coef_off;
            const int* qt = P.qtab[LG];
            const bool zig = P.zigzag != 0;
            int* stage = reinterpret_cast<int*>(sB);              // row-major staging for the zigzag gather (stride N)
            if (zig) __syncthreads();                              // everyone finished reading sB / sBo in pass 2
#pragma unroll
            for (int a = 0; a < T; a++) {
                const int kp = tr2 * 4 + (a & 3) + (a >> 2) * 64;           // split-order row
                const int k = (kp < Hh) ? 2 * kp : 2 * (kp - Hh) + 1;       // natural row
#pragma unroll
                for (int c = 0; c < RC; c++) {
                    const int m0 = tc2 * 4 + c * 32;
                    int qv[4];
#pragma unroll
                    for (int b = 0; b < 4; b++) qv[b] = quantize(acc[a][4 * c + b], __ldg(qt + k * N + 2 * (m0 + b) + g));
                    const int x0 = g ? qv[0] : qv[2], x1 = g ? qv[1] : qv[3];
                    const int r0 = __shfl_xor_sync(0xffffffffu, x0, 1), r1 = __shfl_xor_sync(0xffffffffu, x1, 1);
                    const int4 o = g ? make_int4(r0, qv[2], r1, qv[3]) : make_int4(qv[0], r0, qv[1], r1);
                    *reinterpret_cast<int4*>((zig ? stage : cf) + k * N + 2 * m0 + 4 * g) = o;
                }
            }
            if (zig) {
                __syncthreads();
                const int* zz = P.zz[LG];
                for (int i = tid; i < N * N; i += 256) cf[i] = stage[__ldg(zz + i)];
            }
        } else {
            // pass 1: Rg[i][l] = sum_m Cg[m][i] * Zg[m][l]; sAg[m][i] = Cg[m][i]; columns l natural in chunks of 4
            for (int m = 0; m < Hh; m++) {
                float av[T], bv[T];
#pragma unroll
                for (int c = 0; c < RC; c++) { float4 t = *reinterpret_cast<const float4*>(sAg + m * Hh + tr * 4 + c * 32); av[4 * c] = t.x; av[4 * c + 1] = t.y; av[4 * c + 2] = t.z; av[4 * c + 3] = t.w; }
#pragma unroll
                for (int c = 0; c < RC; c++) { float4 t = *reinterpret_cast<const float4*>(sBg + m * NS + tc * 4 + c * 64); bv[4 * c] = t.x; bv[4 * c + 1] = t.y; bv[4 * c + 2] = t.z; bv[4 * c + 3] = t.w; }
#pragma unroll
                for (int a = 0; a < T; a++)
#pragma unroll
                    for (int b = 0; b < T; b++) acc[a][b] = __fmaf_rn(av[a], bv[b], acc[a][b]);
            }
            __syncthreads();                           // everyone finished reading Z
            // V[i][l] = E + O (even lane), V[N-1-i][l] = E - O (odd lane); store transposed with the columns in
            // split order: sB[(l&1)*h + (l>>1)][row]
#pragma unroll
            for (int b = 0; b < T; b++) {
                const int l = tc * 4 + (b & 3) + (b >> 2) * 64;
                float* vrow = ((l & 1) ? sBo : sB) + (l >> 1) * NS;
#pragma unroll
                for (int c = 0; c < RC; c++) {
                    float v[4];
#pragma unroll
                    for (int a = 0; a < 4; a++) {
                        const float mine = acc[4 * c + a][b];
                        const float other = __shfl_xor_sync(0xffffffffu, mine, 1);
                        v[a] = g ? __fsub_rn(other, mine) : __fadd_rn(mine, other);     // g=0: E+O ; g=1: E-O
                    }
                    const int i0 = tr * 4 + c * 32;
                    if (!g) *reinterpret_cast<float4*>(vrow + i0) = make_float4(v[0], v[1], v[2], v[3]);
                    else *reinterpret_cast<float4*>(vrow + (N - 4 - i0)) = make_float4(v[3], v[2], v[1], v[0]);
                }
            }
            __syncthreads();
#pragma unroll
            for (int a = 0; a < T; a++)
#pragma unroll
                for (int b = 0; b < T; b++) acc[a][b] = 0.0f;
            // pass 2: R2g[i'][j] = sum_m V[i'][2m+g] * Cg[m][j] = sum_m sBg[m][i'] * sAg[m][j]
            for (int m = 0; m < Hh; m++) {
                float av[T], bv[T];
#pragma unroll
                for (int c = 0; c < RC; c++) { float4 t = *reinterpret_cast<const float4*>(sBg + m * NS + tr2 * 4 + c * 64); av[4 * c] = t.x; av[4 * c + 1] = t.y; av[4 * c + 2] = t.z; av[4 * c + 3] = t.w; }
#pragma unroll
                for (int c = 0; c < RC; c++) { float4 t = *reinterpret_cast<const float4*>(sAg + m * Hh + tc2 * 4 + c * 32); bv[4 * c] = t.x; bv[4 * c + 1] = t.y; bv[4 * c + 2] = t.z; bv[4 * c + 3] = t.w; }
#pragma unroll
                for (int a = 0; a < T; a++)
#pragma unroll
                    for (int b = 0; b < T; b++) acc[a][b] = __fmaf_rn(av[a], bv[b], acc[a][b]);
            }
            // X[i'][j] = E' + O' (even lane), X[i'][N-1-j] = E' - O' (odd lane); denormalise, crop, store
            const float mid = P.mid, sc = P.scale;
            const bool vec_ok = ((P.w & 3) == 0);
#pragma unroll
            for (int a = 0; a < T; a++) {
                const int y = e.y + tr2 * 4 + (a & 3) + (a >> 2) * 64;
#pragma unroll
                for (int c = 0; c < RC; c++) {
                    float v[4];
#pragma unroll
                    for (int b = 0; b < 4; b++) {
                        const float mine = acc[a][4 * c + b];
                        const float other = __shfl_xor_sync(0xffffffffu, mine, 1);
                        const float x = g ? __fsub_rn(other, mine) : __fadd_rn(mine, other);
                        v[b] = __fadd_rn(__fdiv_rn(x, sc), mid);
                    }
                    const int j0 = tc2 * 4 + c * 32;
                    const int xs = e.x + (g ? (N - 4 - j0) : j0);
                    if (y < P.h) {
                        float* row = P.layer_f32 + (size_t)y * P.w;
                        const float4 o = g ? make_float4(v[3], v[2], v[1], v[0]) : make_float4(v[0], v[1], v[2], v[3]);
                        if (vec_ok && xs + 3 < P.w) *reinterpret_cast<float4*>(row + xs) = o;
                        else {
                            if (xs < P.w) row[xs] = o.x;
                            if (xs + 1 < P.w) row[xs + 1] = o.y;
                            if (xs + 2 < P.w) row[xs + 2] = o.z;
                            if (xs + 3 < P.w) row[xs + 3] = o.w;
                        }
                    }
                }
            }
        }
    }
}

template <int S, bool INV>
int launch_rows(aeaj_handle* h, const PlaneDesc* planes_dev, const ClassEntry* list, const int* count, int64_t cap, cudaStream_t st) {
    constexpr int LPW = 32 / S;
    int64_t groups = aeaj_cdiv64(cap, LPW);
    int blocks = (int)std::min<int64_t>(aeaj_cdiv64(groups, 8), (int64_t)h->sm_count * 8);
    if (blocks < 1) blocks = 1;
    const int lg = ilog2i(S);
    k_dct_rows<S, INV><<<blocks, 256, 0, st>>>(planes_dev, list, count, INV ? h->dct_dev[lg] + S * S : h->dct_dev[lg],
                                               INV ? h->dct_dev[lg] : h->dct_dev[lg] + S * S);
    AEAJ_LAUNCH_CHECK();
    return 0;
}
constexpr size_t cta_smem_bytes(int S) { return (size_t)(S * S / 2 + S * (S + 4) + 3 * 16) * sizeof(float); }

template <int S, bool INV>
int launch_cta(aeaj_handle* h, const PlaneDesc* planes_dev, const ClassEntry* list, const int* count, int64_t cap, cudaStream_t st) {
    const size_t smem = cta_smem_bytes(S);             // opted in per device by aeaj_dct_init
    int per_sm = (smem > 110 * 1024) ? 1 : ((smem > 56 * 1024) ? 2 : 4);
    int blocks = (int)std::min<int64_t>(std::max<int64_t>(cap, 1), (int64_t)h->sm_count * per_sm);
    const int lg = ilog2i(S);
    // half tables [Ae | Ao]: forward needs Cg^T (sAg[i][m] = Cg[m][i]), inverse needs Cg (sAg[m][i] = Cg[m][i])
    k_dct_cta<S, INV><<<blocks, 256, smem, st>>>(planes_dev, list, count, h->dct_half_dev[lg] + (INV ? (S * S / 2) : 0));
    AEAJ_LAUNCH_CHECK();
    return 0;
}

// ---------------------------------------------------------------------------------------------
// 256 x 256 leaves.  Only the reference's GUI sliders reach this size (gui/main_frame.py:44-45), so this is a plain,
// untuned kernel: one CTA per leaf, two tiled FP32 GEMMs (64 x 64 output tiles, K chunks of 16) through a per-CTA
// global scratch tile; sequential-k FMA accumulation like the other FP32 kernels, the same fused load / store epilogues.
// ---------------------------------------------------------------------------------------------
constexpr int D256_CTAS = 64;
template <class FA, class FB, class FS>
__device__ __forceinline__ void gemm256(FA a_of, FB b_of, FS store) {           // Out[r][c] = sum_k A(r,k) * B(k,c), all 256 x 256
    constexpr int N = 256, TM = 64, TK = 16;
    __shared__ float sAt[TK][TM + 4];                                             // A tile transposed: [k][r]
    __shared__ float sBt[TK][TM + 4];                                             // B tile: [k][c]
    const int tid = threadIdx.x, tr = tid >> 4, tc = tid & 15;                    // 16 x 16 threads, 4 x 4 outputs each
    for (int r0 = 0; r0 < N; r0 += TM)
        for (int c0 = 0; c0 < N; c0 += TM) {
            float acc[4][4];
#pragma unroll
            for (int i = 0; i < 4; i++)
#pragma unroll
                for (int j = 0; j < 4; j++) acc[i][j] = 0.0f;
            for (int k0 = 0; k0 < N; k0 += TK) {
                __syncthreads();
                for (int i = tid; i < TM * TK; i += 256) {
                    const int rr = i / TK, kk = i - rr * TK;                      // A: consecutive threads walk k (row-major A)
                    sAt[kk][rr] = a_of(r0 + rr, k0 + kk);
                    const int k2 = i / TM, cc = i - k2 * TM;                      // B: consecutive threads walk c
                    sBt[k2][cc] = b_of(k0 + k2, c0 + cc);
                }
                __syncthreads();
#pragma unroll
                for (int kk = 0; kk < TK; kk++) {
                    const float4 av = *reinterpret_cast<const float4*>(&sAt[kk][tr * 4]);
                    const float4 bv = *reinterpret_cast<const float4*>(&sBt[kk][tc * 4]);
                    const float a[4] = {av.x, av.y, av.z, av.w}, b[4] = {bv.x, bv.y, bv.z, bv.w};
#pragma unroll
                    for (int i = 0; i < 4; i++)
#pragma unroll
                        for (int j = 0; j < 4; j++) acc[i][j] = __fmaf_rn(a[i], b[j], acc[i][j]);
                }
            }
#pragma unroll
            for (int i = 0; i < 4; i++)
#pragma unroll
                for (int j = 0; j < 4; j++) store(r0 + tr * 4 + i, c0 + tc * 4 + j, acc[i][j]);
        }
}

template <bool INVERSE>
__global__ void __launch_bounds__(256) k_dct256(const PlaneDesc* __restrict__ planes, const ClassEntry* __restrict__ list, const int* __restrict__ count_ptr,
                                                const float* __restrict__ Cm, const float* __restrict__ Ct, const int* __restrict__ izz,
                                                float* __restrict__ scratch) {
    constexpr int N = 256;
    float* Wt = scratch + (size_t)blockIdx.x * N * N;
    const int count = *count_ptr;
    for (int li = blockIdx.x; li < count; li += gridDim.x) {
        const ClassEntry e = list[li];
        const PlaneDesc& P = planes[e.plane];
        if (e.y < P.ry0 || e.y >= P.ry1) continue;
        const int bh = min(N, P.h - e.y), bw = min(N, P.w - e.x);
        const float mid = P.mid, sc = P.scale;
        int* cf = P.coef + (size_t)e.coef_off;
        const int* qt = P.qtab[8];
        const bool zig = P.zigzag != 0;
        float* lay = P.layer_f32 + (size_t)e.y * P.w + e.x;
        const int w = P.w;
        if (!INVERSE) {
            // W = C . X   (X: normalised, reflect-padded samples)
            gemm256([&](int r, int k) { return __ldg(Cm + r * N + k); },
                    [&](int k, int c) { return __fmul_rn(__fsub_rn(__ldg(lay + (size_t)pad_reflect(k, bh) * w + pad_reflect(c, bw)), mid), sc); },
                    [&](int r, int c, float v) { Wt[r * N + c] = v; });
            __syncthreads();
            // Out = W . C^T, quantised
            gemm256([&](int r, int k) { return Wt[r * N + k]; },
                    [&](int k, int c) { return __ldg(Ct + k * N + c); },
                    [&](int r, int c, float v) { const int nat = r * N + c; cf[zig ? __ldg(izz + nat) : nat] = quantize(v, __ldg(qt + nat)); });
        } else {
            // V = C^T . Z   (Z: dequantised coefficients, jpeg.py:524)
            gemm256([&](int r, int k) { return __ldg(Ct + r * N + k); },
                    [&](int k, int c) { const int nat = k * N + c; return (float)(__ldg(cf + (zig ? __ldg(izz + nat) : nat)) * __ldg(qt + nat)); },
                    [&](int r, int c, float v) { Wt[r * N + c] = v; });
            __syncthreads();
            // X = V . C, de-normalised and cropped
            gemm256([&](int r, int k) { return Wt[r * N + k]; },
                    [&](int k, int c) { return __ldg(Cm + k * N + c); },
                    [&](int r, int c, float v) { if (r < bh && c < bw) lay[(size_t)r * w + c] = __fadd_rn(__fdiv_rn(v, sc), mid); });
        }
        __syncthreads();
    }
}

template <bool INV>
int launch_256(aeaj_handle* h, const PlaneDesc* planes_dev, const ClassEntry* list, const int* count, int64_t cap, float* scratch, cudaStream_t st) {
    AEAJ_REQUIRE(scratch, "256 x 256 leaves need the per-call scratch tiles (aeaj_dct256_scratch_floats)");
    const int blocks = (int)std::min<int64_t>(std::max<int64_t>(cap, 1), D256_CTAS);
    k_dct256<INV><<<blocks, 256, 0, st>>>(planes_dev, list, count, h->dct_dev[8], h->dct_dev[8] + 256 * 256, h->izz256_dev, scratch);
    AEAJ_LAUNCH_CHECK();
    return 0;
}

template <bool INV>
int launch_all(aeaj_handle* h, const PlaneDesc* planes_dev, const ClassEntry* class_lists, const int* class_counts,
               const int64_t* off, const int64_t* caps, int lg_min, int lg_max, cudaStream_t st, int* launches,
               void (*mark)(void*, const char*), void* mark_ctx, int tensor_dct, float* scratch256) {
    static const char* fwd_names[9] = {"", "dct_quant_2", "dct_quant_4", "dct_quant_8", "dct_quant_16", "dct_quant_32", "dct_quant_64", "dct_quant_128", "dct_quant_256"};
    static const char* inv_names[9] = {"", "dequant_idct_2", "dequant_idct_4", "dequant_idct_8", "dequant_idct_16", "dequant_idct_32", "dequant_idct_64", "dequant_idct_128", "dequant_idct_256"};
    for (int lg = lg_min; lg <= lg_max; lg++) {
        if (caps[lg] <= 0) continue;
        const ClassEntry* list = class_lists + off[lg];
        const int* cnt = class_counts + lg;
        int rc = 0;
        switch (lg) {
            case 1: rc = launch_rows<2, INV>(h, planes_dev, list, cnt, caps[lg], st); break;
            case 2: rc = launch_rows<4, INV>(h, planes_dev, list, cnt, caps[lg], st); break;
            case 3: rc = launch_rows<8, INV>(h, planes_dev, list, cnt, caps[lg], st); break;
            // tensor_dct bit k: size class 16 << k runs on the tcgen05 kernels of dct_tc.cu, else on the FP32 kernels of this file
            case 4: rc = (tensor_dct & 1) ? launch_dct_tc(h, 16, planes_dev, list, cnt, caps[lg], INV ? 1 : 0, st)
                                          : launch_rows<16, INV>(h, planes_dev, list, cnt, caps[lg], st); break;
            case 5: rc = (tensor_dct & 2) ? launch_dct_tc(h, 32, planes_dev, list, cnt, caps[lg], INV ? 1 : 0, st)
                                          : launch_rows<32, INV>(h, planes_dev, list, cnt, caps[lg], st); break;
            case 6: rc = (tensor_dct & 4) ? launch_dct_tc(h, 64, planes_dev, list, cnt, caps[lg], INV ? 1 : 0, st)
                                          : launch_cta<64, INV>(h, planes_dev, list, cnt, caps[lg], st); break;
            case 7: rc = (tensor_dct & 8) ? launch_dct_tc(h, 128, planes_dev, list, cnt, caps[lg], INV ? 1 : 0, st)
                                          : launch_cta<128, INV>(h, planes_dev, list, cnt, caps[lg], st); break;
            case 8: rc = launch_256<INV>(h, planes_dev, list, cnt, caps[lg], scratch256, st); break;
            default: aeaj_set_error("block size %d not supported (2..256)", 1 << lg); return AEAJ_EINVAL;
        }
        if (rc) return rc;
        if (launches) (*launches)++;
        if (mark) mark(mark_ctx, INV ? inv_names[lg] : fwd_names[lg]);
    }
    return 0;
}

}  // namespace

// DCT-II matrices C and C^T per size, f64 on the host, stored f32: table for size s at dct_dev[log2 s],
// layout [C (s*s)][C^T (s*s)].
size_t aeaj_dct256_scratch_floats() { return (size_t)D256_CTAS * 256 * 256; }

int aeaj_dct_init(aeaj_handle* h) {
    // function attributes are per device: set them for the device of every new handle (aeaj_create selected it)
    AEAJ_CUDA(cudaFuncSetAttribute(k_dct_cta<64, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)cta_smem_bytes(64)));
    AEAJ_CUDA(cudaFuncSetAttribute(k_dct_cta<64, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)cta_smem_bytes(64)));
    AEAJ_CUDA(cudaFuncSetAttribute(k_dct_cta<128, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)cta_smem_bytes(128)));
    AEAJ_CUDA(cudaFuncSetAttribute(k_dct_cta<128, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)cta_smem_bytes(128)));
    size_t total = 0;
    for (int lg = 1; lg <= 8; lg++) total += 2 * ((size_t)1 << (2 * lg));
    float* host = (float*)malloc(total * sizeof(float));
    if (!host) return AEAJ_ENOMEM;
    AEAJ_CUDA(cudaMalloc(&h->dct_all_dev, total * sizeof(float)));
    size_t o = 0;
    for (int lg = 1; lg <= 8; lg++) {
        const int s = 1 << lg;
        for (int k = 0; k < s; k++)
            for (int i = 0; i < s; i++) {
                double v = sqrt(2.0 / s) * cos(M_PI * (2 * i + 1) * k / (2.0 * s));
                if (k == 0) v *= sqrt(0.5);
                host[o + (size_t)k * s + i] = (float)v;
                host[o + (size_t)s * s + (size_t)i * s + k] = (float)v;
            }
        h->dct_dev[lg] = h->dct_all_dev + o;
        o += 2 * (size_t)s * s;
    }
    h->dct_dev[0] = nullptr;
    AEAJ_CUDA(cudaMemcpy(h->dct_all_dev, host, total * sizeof(float), cudaMemcpyHostToDevice));
    free(host);
    // half tables for the even/odd CTA kernels (sizes 64, 128):
    //   [Ce^T | Co^T] (forward)  then  [Ce | Co] (inverse), each h x h row-major, Cg[m][i] = C[2m+g][i], i < h
    size_t htotal = 0;
    for (int lg = 6; lg <= 7; lg++) htotal += (size_t)1 << (2 * lg);
    float* hh = (float*)malloc(htotal * sizeof(float));
    if (!hh) return AEAJ_ENOMEM;
    AEAJ_CUDA(cudaMalloc(&h->dct_half_all_dev, htotal * sizeof(float)));
    size_t ho = 0;
    for (int k = 0; k < 9; k++) h->dct_half_dev[k] = nullptr;
    for (int lg = 6; lg <= 7; lg++) {
        const int s = 1 << lg, hf = s / 2;
        float* fwd = hh + ho;                       // [2][hf][hf] transposed halves
        float* inv = hh + ho + (size_t)s * s / 2;   // [2][hf][hf] plain halves
        for (int g = 0; g < 2; g++)
            for (int m = 0; m < hf; m++)
                for (int i = 0; i < hf; i++) {
                    const int k = 2 * m + g;
                    double v = sqrt(2.0 / s) * cos(M_PI * (2 * i + 1) * k / (2.0 * s));
                    if (k == 0) v *= sqrt(0.5);
                    fwd[(size_t)g * hf * hf + (size_t)i * hf + m] = (float)v;
                    inv[(size_t)g * hf * hf + (size_t)m * hf + i] = (float)v;
                }
        h->dct_half_dev[lg] = h->dct_half_all_dev + ho;
        ho += (size_t)s * s;
    }
    AEAJ_CUDA(cudaMemcpy(h->dct_half_all_dev, hh, htotal * sizeof(float), cudaMemcpyHostToDevice));
    free(hh);
    // zigzag tables: the standard JPEG walk generalised to s x s (jpeg.py:743-766)
    size_t ztotal = 0;
    for (int lg = 1; lg <= 8; lg++) ztotal += (size_t)1 << (2 * lg);
    int32_t* zh = (int32_t*)malloc(ztotal * sizeof(int32_t));
    if (!zh) return AEAJ_ENOMEM;
    AEAJ_CUDA(cudaMalloc(&h->zz_all_dev, ztotal * sizeof(int32_t)));
    size_t zo = 0;
    for (int k = 0; k < 9; k++) h->zz_dev[k] = nullptr;
    for (int lg = 1; lg <= 8; lg++) {
        const int s = 1 << lg;
        int row = 0, col = 0;
        for (int i = 0; i < s * s; i++) {
            zh[zo + i] = row * s + col;
            if (((row + col) & 1) == 0) {
                if (col == s - 1) row++; else if (row == 0) col++; else { row--; col++; }
            } else {
                if (row == s - 1) col++; else if (col == 0) row++; else { row++; col--; }
            }
        }
        h->zz_dev[lg] = h->zz_all_dev + zo;
        zo += (size_t)s * s;
    }
    {   // inverse permutations (row-major index -> stream position), same layout: k_dct256 and the scaled IDCT (idct_scaled.cu)
        std::vector<int32_t> inv(ztotal);
        for (int lg = 1; lg <= 8; lg++) {
            const size_t o = h->zz_dev[lg] - h->zz_all_dev;
            for (int i = 0; i < (1 << (2 * lg)); i++) inv[o + zh[o + i]] = i;
        }
        AEAJ_CUDA(cudaMalloc(&h->izz_all_dev, ztotal * sizeof(int32_t)));
        AEAJ_CUDA(cudaMemcpy(h->izz_all_dev, inv.data(), ztotal * sizeof(int32_t), cudaMemcpyHostToDevice));
        for (int k = 0; k < 9; k++) h->izz_dev[k] = k ? h->izz_all_dev + (h->zz_dev[k] - h->zz_all_dev) : nullptr;
        h->izz256_dev = h->izz_dev[8];
    }
    AEAJ_CUDA(cudaMemcpy(h->zz_all_dev, zh, ztotal * sizeof(int32_t), cudaMemcpyHostToDevice));
    free(zh);
    return 0;
}

int launch_dct_quant(aeaj_handle* h, const PlaneDesc* planes_dev, const ClassEntry* class_lists, const int* class_counts,
                     const int64_t* off, const int64_t* caps, int lg_min, int lg_max, cudaStream_t st, int* launches,
                     void (*mark)(void*, const char*), void* mark_ctx, int tensor_dct, float* scratch256) {
    return launch_all<false>(h, planes_dev, class_lists, class_counts, off, caps, lg_min, lg_max, st, launches, mark, mark_ctx, tensor_dct, scratch256);
}
int launch_dequant_idct(aeaj_handle* h, const PlaneDesc* planes_dev, const ClassEntry* class_lists, const int* class_counts,
                        const int64_t* off, const int64_t* caps, int lg_min, int lg_max, cudaStream_t st, int* launches,
                        void (*mark)(void*, const char*), void* mark_ctx, int tensor_dct, float* scratch256) {
    return launch_all<true>(h, planes_dev, class_lists, class_counts, off, caps, lg_min, lg_max, st, launches, mark, mark_ctx, tensor_dct, scratch256);
}
