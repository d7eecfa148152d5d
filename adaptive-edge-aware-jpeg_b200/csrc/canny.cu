// canny.cu -- EdgeDetection.canny (edge_detection.py:28-86) for sm_100a.
//
//   u8 cast (color.cu) -> CLAHE tile histograms -> CLAHE LUTs -> [CLAHE apply + Gaussian 3x3 +
//   bilateral 5x5] fused, shared-memory tiled with halo staging -> 256-bin histogram -> percentile
//   thresholds -> Sobel/magnitude/NMS/double threshold -> bit-packed strong/weak maps (warp ballot)
//   -> hysteresis by bitmap frontier propagation (persistent CTAs, tile-local convergence in shared
//   memory, dirty neighbour tiles re-queued through a global work queue; no grid-wide barriers).
//
// Integer / u8 work.  Measured, the stencil kernels are bound by instruction issue and the shared-memory pipe, not by HBM
// (DESIGN.md 4); the layout (bit-packed maps, u8 planes, one pass per stage) keeps the traffic at its algorithmic minimum.
// Arithmetic follows SURVEY.md App. A3 as validated by the CPU oracle against the reference.
#include "aeaj_internal.cuh"

namespace {

// bilateral tables: cv.bilateralFilter(d=5, sigmaColor=75, sigmaSpace=75) -- OpenCV builds them with
// std::exp in double and stores float; done on the host with the same libm (aeaj_create).
__constant__ float c_bil_color[256];
__constant__ float c_bil_space[13];
__constant__ int c_bil_dy[13];
__constant__ int c_bil_dx[13];

// ---------------------------------------------------------------------------------------------
// CLAHE (OpenCV imgproc/clahe.cpp), clip 0.75, 4x4 tiles
// ---------------------------------------------------------------------------------------------
struct ClaheGeom { int th, tw, clip; float lutScale, inv_th, inv_tw; };
__host__ __device__ inline ClaheGeom clahe_geom(int h, int w) {
    int eh = h, ew = w;
    if ((w % 4) != 0 || (h % 4) != 0) { eh = h + (4 - h % 4); ew = w + (4 - w % 4); }
    ClaheGeom g;
    g.th = eh / 4; g.tw = ew / 4;
    int area = g.th * g.tw;
    g.lutScale = 255.0f / (float)area;
    int clip = (int)(0.75 * area / 256);
    g.clip = clip < 1 ? 1 : clip;
    g.inv_th = 1.0f / (float)g.th; g.inv_tw = 1.0f / (float)g.tw;
    return g;
}

constexpr int HIST_ROWS = 32;   // rows of one CLAHE tile handled by one block
// 16 consecutive pixels from one 128-bit load, equal neighbours merged into one shared-memory atomic
__device__ __forceinline__ void hist_add16(unsigned int* wh, uint4 q) {
    const unsigned w[4] = {q.x, q.y, q.z, q.w};
    int prev = w[0] & 0xff, cnt = 0;
#pragma unroll
    for (int k = 0; k < 16; k++) {
        const int v = (w[k >> 2] >> (8 * (k & 3))) & 0xff;
        if (v == prev) cnt++;
        else { atomicAdd(&wh[prev], (unsigned)cnt); prev = v; cnt = 1; }
    }
    atomicAdd(&wh[prev], (unsigned)cnt);
}
// grid: (row chunks, 16 tiles, planes).  Each warp walks rows of the tile with 128-bit loads over the
// 16-byte-aligned middle of the row segment; head / tail / reflected padding go byte by byte.
__global__ void __launch_bounds__(256) k_clahe_hist(const PlaneDesc* __restrict__ planes) {
    const PlaneDesc& P = planes[blockIdx.z];
    ClaheGeom g = clahe_geom(P.h, P.w);
    const int tile = blockIdx.y, ty = tile >> 2, tx = tile & 3;
    const int r0 = blockIdx.x * HIST_ROWS;
    if (r0 >= g.th) return;
    __shared__ unsigned int wh[8][256];
    for (int i = threadIdx.x; i < 8 * 256; i += 256) (&wh[0][0])[i] = 0;
    __syncthreads();
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int r1 = min(r0 + HIST_ROWS, g.th);
    const uint8_t* src = P.u8a;
    unsigned int* my = wh[warp];
    const int cx0 = tx * g.tw, cx1 = cx0 + g.tw;
    // halo-split bands: this call owns padded rows [ry0, ry1), the band that ends at h also owns the reflected padding
    const int band_hi = (P.ry1 >= P.h) ? 4 * g.th : P.ry1;
    for (int r = r0 + warp; r < r1; r += 8) {
        const int gy = ty * g.th + r;
        if (gy < P.ry0 || gy >= band_hi) continue;
        const int sy = reflect101(gy, P.h);
        const uint8_t* rowp = src + (size_t)sy * P.w;
        const int xa = cx0, xb = min(cx1, P.w);
        if (xa < xb) {
            const int head = min((int)((16 - ((uintptr_t)(rowp + xa) & 15)) & 15), xb - xa);
            const int nvec = (xb - xa - head) >> 4;
            const int tail0 = xa + head + nvec * 16;
            for (int x = xa + lane; x < xa + head; x += 32) atomicAdd(&my[rowp[x]], 1u);
            for (int x = tail0 + lane; x < xb; x += 32) atomicAdd(&my[rowp[x]], 1u);
            const uint4* vp = reinterpret_cast<const uint4*>(rowp + xa + head);
            for (int c = lane; c < nvec; c += 32) hist_add16(my, __ldg(vp + c));
        }
        for (int x = max(cx0, P.w) + lane; x < cx1; x += 32) atomicAdd(&my[rowp[reflect101(x, P.w)]], 1u);
    }
    __syncthreads();
    unsigned s = 0;
#pragma unroll
    for (int k = 0; k < 8; k++) s += wh[k][threadIdx.x];
    if (s) atomicAdd(&P.clahe_hist[tile * 256 + threadIdx.x], s);
}

// grid: (16 tiles, planes), 256 threads = bins
// sum over the ranks of a halo-split (world == 1: just this GPU's counters); peer counters are read uncached
__device__ __forceinline__ unsigned peer_sum(const unsigned int* mine, const PeerSet& peers) {
    unsigned s = 0;
    for (int r = 0; r < peers.world; r++)
        s += (r == peers.rank) ? *mine : __ldcv(reinterpret_cast<const unsigned int*>(reinterpret_cast<const char*>(mine) + peers.delta[r]));
    return s;
}

__global__ void __launch_bounds__(256) k_clahe_lut(const PlaneDesc* __restrict__ planes, const __grid_constant__ PeerSet peers) {
    const PlaneDesc& P = planes[blockIdx.y];
    ClaheGeom g = clahe_geom(P.h, P.w);
    const int tile = blockIdx.x, i = threadIdx.x;
    __shared__ int red[256];
    int hv = (int)peer_sum(&P.clahe_hist[tile * 256 + i], peers);
    int excess = hv > g.clip ? hv - g.clip : 0;
    hv = hv > g.clip ? g.clip : hv;
    red[i] = excess;
    __syncthreads();
    for (int s = 128; s > 0; s >>= 1) { if (i < s) red[i] += red[i + s]; __syncthreads(); }
    int clipped = red[0];
    __syncthreads();
    int redist = clipped / 256, residual = clipped - redist * 256;
    hv += redist;
    if (residual != 0) {
        int step = 256 / residual; if (step < 1) step = 1;
        if ((i % step) == 0 && (i / step) < residual) hv++;
    }
    // inclusive scan
    red[i] = hv;
    __syncthreads();
    for (int off = 1; off < 256; off <<= 1) {
        int t = (i >= off) ? red[i - off] : 0;
        __syncthreads();
        red[i] += t;
        __syncthreads();
    }
    int v = __float2int_rn(__fmul_rn((float)red[i], g.lutScale));
    P.clahe_lut[tile * 256 + i] = (uint8_t)(v < 0 ? 0 : (v > 255 ? 255 : v));
}

// ---------------------------------------------------------------------------------------------
// fused pre-filter: [CLAHE apply] -> [Gaussian 3x3] -> [bilateral d=5] on a 64x32 tile.
// Halo cells hold the value at the REFLECT_101-folded coordinate, so each stage sees exactly the
// border OpenCV builds for it (proof sketch in DESIGN.md: the fold is a local isometry and the
// Gaussian is symmetric; the bilateral is evaluated at in-image pixels only).
// stages: bit0 CLAHE apply, bit1 Gaussian, bit2 bilateral.   grid: (tiles x, tiles y, planes)
// ---------------------------------------------------------------------------------------------
constexpr int PF_TW = 128, PF_TH = 64;
constexpr int PF_CG = PF_TW / 4;                     // 4-px groups per output row (stage C)
constexpr int PF_CR = 2 * (256 / PF_CG);             // output rows per stage-C pass
constexpr int PF_AS = PF_TW + 8;                     // row stride of both staging tiles (4-byte aligned rows)
constexpr int PF_AG = PF_AS / 4;                     // 4-column groups per staging row
// tap k of the 13-tap bilateral window in raster order -> (dy, dx, weight class r^2 in {0,1,2,4} -> 0..3)
#define BIL_TAPS_UP(X) X(0,-2,0,3) X(1,-1,-1,2) X(2,-1,0,1) X(3,-1,1,2) X(4,0,-2,3) X(5,0,-1,1)
#define BIL_TAPS_DN(X) X(7,0,1,1) X(8,0,2,3) X(9,1,-1,2) X(10,1,0,1) X(11,1,1,2) X(12,2,0,3)

// Instruction budget (the kernel is issue bound, ~250 -> ~200 thread instructions per sample):
//  * stage A works on 4-column groups (one 16-byte read of the folded coordinates / weights, one word store) and, when
//    the whole tile interpolates between the same four CLAHE tiles (all but the tiles that straddle a CLAHE tile centre
//    line), reads the four LUT bytes of a pixel with ONE shared load from a per-block table of packed quadruples;
//  * stage B stores 4 x the Gaussian result as u16, so that |a - b| of two window elements IS the byte offset into the
//    float weight table (no shift / LEA per tap); the sums are carried scaled by 4, which commutes with every rounding
//    (sum4 = 4 sum exactly, (4 s) / w = 4 (s / w)), and the centre tap needs no table lookup;
//  * stage C gives a thread 4 px of two ADJACENT rows: the 6 x 8 window is extracted / converted once for 8 px.
__global__ void __launch_bounds__(256, 4) k_prefilter(const PlaneDesc* __restrict__ planes, const __grid_constant__ TileMap tm, int stages, int do_hist) {
    int plane_i, txi, tyi;
    tile_decode(tm, blockIdx.x, plane_i, txi, tyi);
    const PlaneDesc& P = planes[plane_i];
    const int X0 = txi * PF_TW, Y0 = tyi * PF_TH;
    if (Y0 < P.ry0 || Y0 >= P.ry1) return;             // halo-split bands are multiples of the tile height
    __shared__ __align__(16) uint8_t sA[PF_TH + 6][PF_AS];     // CLAHE output (or source), halo 3
    __shared__ __align__(16) uint16_t sG[PF_TH + 4][PF_AS];    // 4 x Gaussian output, halo 2
    __shared__ __align__(16) uint8_t sLut[16][256];            // general path only (tiny planes: > 2 CLAHE tile pairs per axis)
    __shared__ uint32_t sQuad[4][256];                         // packed path: the four LUT bytes of value v in one word, per
                                                               // (row regime, column regime); a tile straddles at most one CLAHE
                                                               // tile-centre line per axis unless the plane is tiny
    __shared__ float sW[4][256];                               // space weight (r^2 = 0,1,2,4) x colour weight, rounded product
    __shared__ unsigned int sHist[256];
    __shared__ __align__(16) float sXa[PF_AS];                 // CLAHE interpolation weights per tile column / row
    __shared__ float sYa[PF_TH + 6];
    __shared__ uint8_t sTx[PF_AS][2], sTy[PF_TH + 6][2];       // CLAHE tile indices per tile column / row
    __shared__ __align__(16) int sFx[PF_AS];                   // REFLECT_101-folded source coordinates
    __shared__ long long sRow[PF_TH + 6];                      // byte offset of the (folded) source row from P.u8a; rows outside this
                                                               // call's band (multi-GPU halo-split) point into the neighbour rank's copy
    __shared__ __align__(16) int sCo[PF_AS];                   // byte offset of the column's regime table inside sQuad (0 / 1024)
    __shared__ int sRo[PF_TH + 6];                             // same for the row regime (0 / 2048)
    const int tid = threadIdx.x;
    const ClaheGeom g = clahe_geom(P.h, P.w);
    auto tile_of = [](int coord, float inv, float& frac, int& t_lo, int& t_hi) {
        const float tf = __fsub_rn(__fmul_rn((float)coord, inv), 0.5f);
        const int t1 = (int)floorf(tf);
        frac = __fsub_rn(tf, (float)t1);
        t_lo = max(t1, 0); t_hi = min(t1 + 1, 3);
    };
    // regime 0 = the tile pair of column / row 0, regime 1 = the pair of the last column / row; anything else -> general path
    int two_ok = 1;
    if (tid < PF_AS) {
        const int x = reflect101(X0 + tid - 3, P.w);
        sFx[tid] = x;
        float fr, fr0; int lo, hi, lo0, hi0, loL, hiL;
        tile_of(x, g.inv_tw, fr, lo, hi);
        tile_of(reflect101(X0 - 3, P.w), g.inv_tw, fr0, lo0, hi0);
        tile_of(reflect101(X0 + PF_AS - 4, P.w), g.inv_tw, fr0, loL, hiL);
        sXa[tid] = fr;
        sTx[tid][0] = (uint8_t)lo; sTx[tid][1] = (uint8_t)hi;
        const bool r0 = (lo == lo0 && hi == hi0), r1 = (lo == loL && hi == hiL);
        sCo[tid] = r0 ? 0 : 1024;
        two_ok = r0 || r1;
    } else if (tid >= PF_AS && tid < PF_AS + PF_TH + 6) {
        const int r = tid - PF_AS;
        const int y = reflect101(Y0 + r - 3, P.h);
        sRow[r] = ((y < P.ry0) ? P.peer_up : ((y >= P.ry1) ? P.peer_dn : 0ll)) + (long long)y * P.w;
        float fr, fr0; int lo, hi, lo0, hi0, loL, hiL;
        tile_of(y, g.inv_th, fr, lo, hi);
        tile_of(reflect101(Y0 - 3, P.h), g.inv_th, fr0, lo0, hi0);
        tile_of(reflect101(Y0 + PF_TH + 2, P.h), g.inv_th, fr0, loL, hiL);
        sYa[r] = fr;
        sTy[r][0] = (uint8_t)(lo * 4); sTy[r][1] = (uint8_t)(hi * 4);
        const bool r0 = (lo == lo0 && hi == hi0), r1 = (lo == loL && hi == hiL);
        sRo[r] = r0 ? 0 : 2048;
        two_ok = r0 || r1;
    }
    {
        float cw = c_bil_color[tid];
        sW[0][tid] = cw;                                       // centre tap: space weight exp(0) = 1
        sW[1][tid] = __fmul_rn(c_bil_space[2], cw);            // r^2 = 1
        sW[2][tid] = __fmul_rn(c_bil_space[1], cw);            // r^2 = 2
        sW[3][tid] = __fmul_rn(c_bil_space[0], cw);            // r^2 = 4
        sHist[tid] = 0;
    }
    const bool uniform = __syncthreads_and(two_ok) != 0;       // packed path usable (also publishes the tables above)
    const bool clahe = (stages & 1) != 0;
    if (clahe) {
        if (uniform) {
            const uint8_t* l = P.clahe_lut;
            const int rr[2] = {sTy[0][0] * 256, sTy[PF_TH + 5][0] * 256}, rh[2] = {sTy[0][1] * 256, sTy[PF_TH + 5][1] * 256};
            const int cl[2] = {sTx[0][0] * 256, sTx[PF_AS - 1][0] * 256}, ch[2] = {sTx[0][1] * 256, sTx[PF_AS - 1][1] * 256};
            const int nry = (sRo[PF_TH + 5] != 0) ? 2 : 1, ncx = (sCo[PF_AS - 1] != 0) ? 2 : 1;
            for (int ry = 0; ry < nry; ry++)
                for (int cx = 0; cx < ncx; cx++)
                    sQuad[ry * 2 + cx][tid] = (uint32_t)l[rr[ry] + cl[cx] + tid] | ((uint32_t)l[rr[ry] + ch[cx] + tid] << 8) |
                                              ((uint32_t)l[rh[ry] + cl[cx] + tid] << 16) | ((uint32_t)l[rh[ry] + ch[cx] + tid] << 24);
        } else {
            for (int i = tid; i < 16 * 256 / 4; i += 256) reinterpret_cast<uint32_t*>(&sLut[0][0])[i] = reinterpret_cast<const uint32_t*>(P.clahe_lut)[i];
        }
        __syncthreads();
    }
    const uint8_t* src = P.u8a;
    // tiles that touch rows of a neighbour rank read the source with ld.cv (never a stale line); everybody else plain loads
    const bool tile_remote = (Y0 - 3 < P.ry0 && P.peer_up != 0) || (Y0 + PF_TH + 3 > P.ry1 && P.peer_dn != 0);
    // stage A: source (folded coordinates) -> CLAHE; the staging region is PF_TH + 6 rows x 72 columns (2 spare
    // columns keep the index arithmetic to shifts; they hold valid folded pixels and are never read)
    auto stage_a = [&](auto remote_tag) {
        constexpr bool REMOTE = decltype(remote_tag)::value;
        auto ld8 = [](const uint8_t* p) -> int { return REMOTE ? (int)__ldcv(p) : (int)*p; };
        if (!clahe || uniform) {
            // a thread keeps its 4-column group and walks down the rows (7 x 34 = 238 threads busy, 10 rows each): no index
            // division, and everything that depends on the column only -- folded coordinates, interpolation weights, regime
            // table offsets -- is loaded once.  Groups whose 8 surrounding bytes lie inside the row fetch two aligned words
            // instead of four bytes.
            static_assert((PF_TH + 6) % (256 / PF_AG) == 0, "stage A row walk");
            constexpr int RSTEP = 256 / PF_AG;
            if (tid < RSTEP * PF_AG) {
                const int gx = (tid % PF_AG) * 4;
                const int4 fx = *reinterpret_cast<const int4*>(&sFx[gx]);
                const float4 xa4 = *reinterpret_cast<const float4*>(&sXa[gx]);
                const float xav[4] = {xa4.x, xa4.y, xa4.z, xa4.w};
                const float xa1v[4] = {__fsub_rn(1.0f, xa4.x), __fsub_rn(1.0f, xa4.y), __fsub_rn(1.0f, xa4.z), __fsub_rn(1.0f, xa4.w)};
                const int4 co4 = *reinterpret_cast<const int4*>(&sCo[gx]);
                const char* qbase = reinterpret_cast<const char*>(&sQuad[0][0]);
                const int xw = X0 - 4 + gx;                                  // the aligned word that holds column X0 - 3 + gx in byte 1
                const bool words = xw >= 0 && xw + 8 <= P.w && (P.w & 3) == 0 && fx.x == xw + 1 && fx.w == xw + 4;
#pragma unroll 2
                for (int ry = tid / PF_AG; ry < PF_TH + 6; ry += RSTEP) {
                    const uint8_t* srow = src + sRow[ry];
                    int v[4];
                    if (words) {
                        const uint32_t* wp = reinterpret_cast<const uint32_t*>(srow + xw);
                        const uint32_t w0 = REMOTE ? __ldcv(wp) : __ldg(wp), w1 = REMOTE ? __ldcv(wp + 1) : __ldg(wp + 1);
                        v[0] = (w0 >> 8) & 0xff; v[1] = (w0 >> 16) & 0xff; v[2] = w0 >> 24; v[3] = w1 & 0xff;
                    } else {
                        v[0] = ld8(srow + fx.x); v[1] = ld8(srow + fx.y); v[2] = ld8(srow + fx.z); v[3] = ld8(srow + fx.w);
                    }
                    uint32_t packed;
                    if (clahe) {
                        int o[4];
                        const float ya = sYa[ry], ya1 = __fsub_rn(1.0f, ya);
                        const int ro = sRo[ry];
                        const int cov[4] = {co4.x + ro, co4.y + ro, co4.z + ro, co4.w + ro};
#pragma unroll
                        for (int k = 0; k < 4; k++) {
                            const uint32_t q = *reinterpret_cast<const uint32_t*>(qbase + cov[k] + v[k] * 4);
                            const float xa = xav[k], xa1 = xa1v[k];
                            const float a = __fmul_rn((float)(q & 0xffu), xa1), b = __fmul_rn((float)((q >> 8) & 0xffu), xa);
                            const float c = __fmul_rn((float)((q >> 16) & 0xffu), xa1), d = __fmul_rn((float)(q >> 24), xa);
                            // a convex combination of bytes: within rounding noise of [0, 255], so cvRound needs no saturation
                            o[k] = __float2int_rn(__fadd_rn(__fmul_rn(__fadd_rn(a, b), ya1), __fmul_rn(__fadd_rn(c, d), ya)));
                        }
                        packed = __byte_perm(__byte_perm(o[0], o[1], 0x0040), __byte_perm(o[2], o[3], 0x0040), 0x5410);
                    } else {
                        packed = __byte_perm(__byte_perm(v[0], v[1], 0x0040), __byte_perm(v[2], v[3], 0x0040), 0x5410);
                    }
                    *reinterpret_cast<uint32_t*>(&sA[ry][gx]) = packed;
                }
            }
        } else {
            for (int i = tid; i < (PF_TH + 6) * PF_AS; i += 256) {
                const int ry = i / PF_AS, rx = i - ry * PF_AS;
                const int v = ld8(src + sRow[ry] + sFx[rx]);
                const float xa = sXa[rx], xa1 = __fsub_rn(1.0f, xa), ya = sYa[ry], ya1 = __fsub_rn(1.0f, ya);
                const uint8_t* l0 = &sLut[sTy[ry][0]][v];
                const uint8_t* l1 = &sLut[sTy[ry][1]][v];
                const int c0 = sTx[rx][0] * 256, c1 = sTx[rx][1] * 256;
                const float a = __fmul_rn((float)l0[c0], xa1), b = __fmul_rn((float)l0[c1], xa);
                const float c = __fmul_rn((float)l1[c0], xa1), d = __fmul_rn((float)l1[c1], xa);
                const float r = __fadd_rn(__fmul_rn(__fadd_rn(a, b), ya1), __fmul_rn(__fadd_rn(c, d), ya));
                sA[ry][rx] = (uint8_t)min(max(__float2int_rn(r), 0), 255);
            }
        }
    };
    if (tile_remote) stage_a(std::true_type{});
    else stage_a(std::false_type{});
    __syncthreads();
    // stage B: Gaussian [1 2 1]x[1 2 1], 4 outputs per thread sharing the 6 column sums; stored as 4 * value (u16)
    for (int i = tid; i < (PF_TH + 4) * (PF_CG + 1); i += 256) {
        const int ry = i / (PF_CG + 1), gx = (i - ry * (PF_CG + 1)) * 4;            // output cells (ry, gx..gx+3) of the halo-2 region
        if (stages & 2) {
            // two 16-bit lanes per register: (c0,c1), (c2,c3), (c4,c5) of each of the three rows -> column sums -> row sums
            uint32_t cs[3];
            {
                uint32_t p[3][3];
#pragma unroll
                for (int r = 0; r < 3; r++) {
                    const uint32_t w0 = *reinterpret_cast<const uint32_t*>(&sA[ry + r][gx]), w1 = *reinterpret_cast<const uint32_t*>(&sA[ry + r][gx + 4]);
                    p[r][0] = __byte_perm(w0, 0, 0x4140); p[r][1] = __byte_perm(w0, 0, 0x4342); p[r][2] = __byte_perm(w1, 0, 0x4140);
                }
#pragma unroll
                for (int j = 0; j < 3; j++) cs[j] = p[0][j] + 2 * p[1][j] + p[2][j];          // <= 1020 per lane
            }
            const uint32_t s1 = __byte_perm(cs[0], cs[1], 0x5432), s3 = __byte_perm(cs[1], cs[2], 0x5432);   // (c1,c2), (c3,c4)
            const uint32_t o01 = cs[0] + cs[1] + 0x00080008u + 2 * s1, o23 = cs[1] + cs[2] + 0x00080008u + 2 * s3;   // sum + 8, <= 4088
            // ((x >> 4) << 2) per lane: the two bits that cross the lane boundary are masked away
            *reinterpret_cast<uint2*>(&sG[ry][gx]) = make_uint2((o01 >> 2) & 0x03fc03fcu, (o23 >> 2) & 0x03fc03fcu);
        } else {
            int o[4];
#pragma unroll
            for (int k = 0; k < 4; k++) o[k] = sA[ry + 1][gx + 1 + k];
            *reinterpret_cast<uint2*>(&sG[ry][gx]) = make_uint2((uint32_t)(o[0] << 2) | ((uint32_t)(o[1] << 2) << 16), (uint32_t)(o[2] << 2) | ((uint32_t)(o[3] << 2) << 16));
        }
    }
    __syncthreads();
    // stage C: bilateral, thread -> 4 consecutive px in rows 2*(tid/16) and 2*(tid/16) + 1 of each 32-row half of the tile
    uint8_t* dst = P.u8b;
    const int tx = (tid % PF_CG) * 4;
#pragma unroll 1
    for (int half = 0; half < PF_TH / PF_CR; half++) {
    const int ty0 = (tid / PF_CG) * 2 + PF_CR * half;
    uint32_t outw[2] = {0, 0};
    {
        // 6 rows x 8 elements window: rows ty0..ty0+5, cols tx..tx+7 of sG (each element = 4 * pixel)
        int wi[6][8];
#pragma unroll
        for (int r = 0; r < 6; r++) {
            const uint2 a = *reinterpret_cast<const uint2*>(&sG[ty0 + r][tx]);
            const uint2 b = *reinterpret_cast<const uint2*>(&sG[ty0 + r][tx + 4]);
            wi[r][0] = a.x & 0xffffu; wi[r][1] = a.x >> 16; wi[r][2] = a.y & 0xffffu; wi[r][3] = a.y >> 16;
            wi[r][4] = b.x & 0xffffu; wi[r][5] = b.x >> 16; wi[r][6] = b.y & 0xffffu; wi[r][7] = b.y >> 16;
        }
        if (stages & 4) {
            const float w_c = sW[0][0];
            const char* wbase = reinterpret_cast<const char*>(&sW[0][0]);
#define BIL_ONE(idx, dy, dx, cls) { const int v = wi[rr + 2 + (dy)][k + 2 + (dx)]; \
                                    const float wgt = *reinterpret_cast<const float*>(wbase + (cls) * 1024 + __sad(v, v0, 0u)); \
                                    sum = __fmaf_rn((float)v, wgt, sum); wsum = __fadd_rn(wsum, wgt); }
#define BIL_PIXEL { const int v0 = wi[rr + 2][k + 2]; \
                    sum = 0.0f; wsum = 0.0f; \
                    BIL_TAPS_UP(BIL_ONE) \
                    sum = __fmaf_rn((float)v0, w_c, sum); wsum = __fadd_rn(wsum, w_c); \
                    BIL_TAPS_DN(BIL_ONE) }
#pragma unroll
            for (int rr = 0; rr < 2; rr++) {
                // cvRound(sum / wsum): an approximate quotient decides unless it is within 1e-3 of a .5 tie (its error is
                // < 1e-4 on values <= 255).  The test is made once per 4 px; the rare row that fails it (< 1 %) is redone
                // with the correctly rounded division, so the common case carries neither a branch per pixel nor the sums.
                // A weighted mean of bytes needs no saturation.
                constexpr unsigned ins[4] = {0x3214u, 0x3240u, 0x3410u, 0x4210u};      // byte k of the word <- low byte of the result
                uint32_t word = 0;
                float worst = 0.0f;
#pragma unroll
                for (int k = 0; k < 4; k++) {
                    float sum, wsum, rw;
                    BIL_PIXEL
                    asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(rw) : "f"(wsum));
                    const float q0 = __fmul_rn(__fmul_rn(sum, rw), 0.25f);
                    const float kf = rintf(q0);
                    word = __byte_perm(word, (uint32_t)(int)kf, ins[k]);
                    worst = fmaxf(worst, fabsf(__fsub_rn(q0, kf)));
                }
                if (worst > 0.499f) {
#pragma unroll
                    for (int k = 0; k < 4; k++) {
                        float sum, wsum;
                        BIL_PIXEL
                        word = __byte_perm(word, (uint32_t)__float2int_rn(__fmul_rn(__fdiv_rn(sum, wsum), 0.25f)), ins[k]);
                    }
                }
                outw[rr] = word;
            }
#undef BIL_PIXEL
#undef BIL_ONE
        } else {
#pragma unroll
            for (int rr = 0; rr < 2; rr++)
#pragma unroll
                for (int k = 0; k < 4; k++) outw[rr] |= (uint32_t)(wi[rr + 2][k + 2] >> 2) << (8 * k);
        }
    }
    const int x = X0 + tx;
#pragma unroll
    for (int rr = 0; rr < 2; rr++) {
        const int y = Y0 + ty0 + rr;
        if (y >= P.h) continue;
        uint8_t* drow = dst + (size_t)y * P.w;
        if (x + 3 < P.w && ((P.w & 3) == 0)) *reinterpret_cast<uint32_t*>(drow + x) = outw[rr];
        else {
#pragma unroll
            for (int k = 0; k < 4; k++) if (x + k < P.w) drow[x + k] = (uint8_t)(outw[rr] >> (8 * k));
        }
        if (do_hist) {
            // shared-memory atomics; four equal px (flat areas, where same-address conflicts would serialise) -> one add of 4
            const uint32_t w = outw[rr], b0 = w & 0xffu;
            if ((x + 3 < P.w) && (w == b0 * 0x01010101u)) {
                atomicAdd(&sHist[b0], 4u);
            } else {
#pragma unroll
                for (int k = 0; k < 4; k++)
                    if (x + k < P.w) atomicAdd(&sHist[(w >> (8 * k)) & 0xffu], 1u);
            }
        }
    }
    }
    if (do_hist) {
        __syncthreads();
        if (sHist[tid]) atomicAdd(&P.hist[tid], sHist[tid]);
    }
}

// plain 256-bin histogram of a u8 plane (stage API: aeaj_percentile_thresholds on its own)
__global__ void __launch_bounds__(256) k_hist_u8(const uint8_t* __restrict__ src, size_t n, unsigned int* __restrict__ hist) {
    __shared__ unsigned int sh[256];
    sh[threadIdx.x] = 0;
    __syncthreads();
    for (size_t i = (size_t)blockIdx.x * 256 + threadIdx.x; i < n; i += (size_t)gridDim.x * 256) atomicAdd(&sh[src[i]], 1u);
    __syncthreads();
    if (sh[threadIdx.x]) atomicAdd(&hist[threadIdx.x], sh[threadIdx.x]);
}

// np.percentile(img, 10 / 30) (method 'linear') from the histogram, then cv.Canny's threshold prep
// (imgproc/canny.cpp: L2gradient -> squared, clamped to 32767, floor); the order statistics are located in k_thresholds.
__device__ void canny_prepare_thresholds(double lo, double hi, int* thr) {
    if (lo > hi) { double t = lo; lo = hi; hi = t; }
    lo = fmin(32767.0, lo); hi = fmin(32767.0, hi);
    if (lo > 0) lo *= lo;
    if (hi > 0) hi *= hi;
    thr[0] = (int)floor(lo); thr[1] = (int)floor(hi);
}
// one warp per plane: lane i owns bins 8i..8i+7; warp-shuffle prefix sums locate the order statistics
__device__ __forceinline__ int first_bin_above(const unsigned long long* cum8, unsigned long long target, int lane) {
    // smallest bin whose inclusive cumulative count exceeds `target`
    const unsigned m = __ballot_sync(0xffffffffu, cum8[7] > target);
    const int src = __ffs(m) - 1;
    int bin = 0;
#pragma unroll
    for (int k = 7; k >= 0; k--) if (cum8[k] > target) bin = 8 * lane + k;
    return __shfl_sync(0xffffffffu, bin, src < 0 ? 31 : src);
}
__device__ __forceinline__ double percentile_warp(const unsigned long long* cum8, unsigned long long n, double q, int lane) {
    const double v = (double)(n - 1) * q;
    const double lo = floor(v), gfrac = v - lo;
    const unsigned long long ilo = (unsigned long long)lo, ihi = ilo + 1 < n ? ilo + 1 : n - 1;
    const int a = first_bin_above(cum8, ilo, lane), b = first_bin_above(cum8, ihi, lane);
    const double d = (double)(b - a);
    return gfrac < 0.5 ? (double)a + d * gfrac : (double)b - d * (1.0 - gfrac);
}
__global__ void __launch_bounds__(128) k_thresholds(const PlaneDesc* __restrict__ planes, int nplanes, const __grid_constant__ PeerSet peers) {
    const int p = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5), lane = threadIdx.x & 31;
    if (p >= nplanes) return;
    const PlaneDesc& P = planes[p];
    unsigned long long cum8[8];
    unsigned long long run = 0;
#pragma unroll
    for (int k = 0; k < 8; k++) { run += peer_sum(&P.hist[8 * lane + k], peers); cum8[k] = run; }
    unsigned long long inc = run;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) { const unsigned long long t = __shfl_up_sync(0xffffffffu, inc, o); if (lane >= o) inc += t; }
    const unsigned long long off = inc - run;
#pragma unroll
    for (int k = 0; k < 8; k++) cum8[k] += off;
    const unsigned long long n = (unsigned long long)P.h * P.w;
    const double lo = percentile_warp(cum8, n, 10.0 / 100.0, lane), hi = percentile_warp(cum8, n, 30.0 / 100.0, lane);
    if (lane == 0) {
        if (P.thr_d) { P.thr_d[0] = lo; P.thr_d[1] = hi; }
        canny_prepare_thresholds(lo, hi, P.thr);
    }
}
__global__ void k_thresholds_from_double(const double* thr_d, int* thr) { canny_prepare_thresholds(thr_d[0], thr_d[1], thr); }

// ---------------------------------------------------------------------------------------------
// Sobel 3x3 (BORDER_REPLICATE) + L2 magnitude + NMS + double threshold -> strong/weak bitmaps.
// tile 64x32, 8 warps; each warp classifies 32 consecutive pixels of a row and ballots them into
// one bitmap word.   grid: (tiles x, tiles y, planes)
// ---------------------------------------------------------------------------------------------
constexpr int NM_TW = 64, NM_TH = 64;
constexpr int NM_SS = NM_TW + 8;                      // source tile: 72 columns starting at X0-4 (4-byte aligned)
constexpr int NM_MS = NM_TW + 4;                      // magnitude tile: 68 columns starting at X0-1
// unsigned bytes of a . signed bytes of b + c
__device__ __forceinline__ int dp4a_us(uint32_t a, uint32_t b, int c) {
    int d;
    asm("dp4a.u32.s32 %0, %1, %2, %3;" : "=r"(d) : "r"(a), "r"(b), "r"(c));
    return d;
}

// c != 0 ? a : b as one SEL (written as a ?: chain the compiler builds branches that every warp then walks through entirely)
__device__ __forceinline__ int selnz(int a, int b, int c) {
    int r;
    asm("{.reg .pred p; setp.ne.s32 p, %3, 0; selp.s32 %0, %1, %2, p;}" : "=r"(r) : "r"(a), "r"(b), "r"(c));
    return r;
}

__global__ void __launch_bounds__(256) k_canny_nms(const PlaneDesc* __restrict__ planes, const __grid_constant__ TileMap tm) {
    int plane_i, txi, tyi;
    tile_decode(tm, blockIdx.x, plane_i, txi, tyi);
    const PlaneDesc& P = planes[plane_i];
    const int X0 = txi * NM_TW, Y0 = tyi * NM_TH;
    if (Y0 < P.ry0 || Y0 >= P.ry1) return;
    __shared__ __align__(16) uint8_t sS[NM_TH + 4][NM_SS];       // rows Y0-2.., cols X0-4.. (BORDER_REPLICATE)
    // 4 x squared magnitude + direction class of the gradient (0 horizontal, 1 vertical, 2 / 3 the diagonals); rows Y0-1..,
    // cols X0-1.. (magnitude 0 outside the image).  One word per cell: with c = 4 m + d,  m > m'  <=>  (c & ~3) > c'  and
    // m >= m'  <=>  (c | 3) >= c', so the neighbours are compared as loaded and the direction never has to be recomputed.
    __shared__ __align__(16) int sM[NM_TH + 2][NM_MS];
    const int tid = threadIdx.x;
    const uint8_t* src = P.u8b;
    // halo-split: the (at most 2) source rows outside this call's band live in the neighbour rank's copy of the plane; tiles
    // that touch them read with ld.cv (never a stale line)
    const int ph = P.h, pw = P.w, ry0 = P.ry0, ry1 = P.ry1;
    const long long up = P.peer_up, dn = P.peer_dn;
    const bool tile_remote = (Y0 - 2 < ry0 && up != 0) || (Y0 + NM_TH + 2 > ry1 && dn != 0);
    auto src_row = [&](int y) -> const uint8_t* {
        return src + ((y < ry0) ? up : ((y >= ry1) ? dn : 0ll)) + (size_t)y * pw;
    };
    // stage 1: source tile.  Interior tiles of 4-aligned planes use 32-bit loads.
    if (X0 >= 4 && X0 + NM_SS - 4 <= pw && (pw & 3) == 0) {
        if (!tile_remote) {
            for (int i = tid; i < (NM_TH + 4) * (NM_SS / 4); i += 256) {
                const int ry = i / (NM_SS / 4), rw = i - ry * (NM_SS / 4);
                reinterpret_cast<uint32_t*>(&sS[ry][0])[rw] =
                    __ldg(reinterpret_cast<const uint32_t*>(src + (size_t)clampi(Y0 + ry - 2, 0, ph - 1) * pw + X0 - 4) + rw);
            }
        } else {
            for (int i = tid; i < (NM_TH + 4) * (NM_SS / 4); i += 256) {
                const int ry = i / (NM_SS / 4), rw = i - ry * (NM_SS / 4);
                reinterpret_cast<uint32_t*>(&sS[ry][0])[rw] = __ldcv(reinterpret_cast<const uint32_t*>(src_row(clampi(Y0 + ry - 2, 0, ph - 1)) + X0 - 4) + rw);
            }
        }
    } else {
        for (int i = tid; i < (NM_TH + 4) * NM_SS; i += 256) {
            const int ry = i / NM_SS, rx = i - ry * NM_SS;
            const uint8_t* p = src_row(clampi(Y0 + ry - 2, 0, ph - 1)) + clampi(X0 + rx - 4, 0, pw - 1);
            sS[ry][rx] = tile_remote ? __ldcv(p) : *p;
        }
    }
    __syncthreads();
    // stage 2: Sobel + L2 magnitude + direction class for 4 cells per task; cell (ry, c) <-> pixel (Y0-1+ry, X0-1+c),
    // its 3x3 window starts at source tile row ry, column c+2.  Tiles whose cells all lie inside the image (all but the
    // border tiles) skip the per-cell bounds selects.
    auto sobel = [&](auto interior_tag) {
        constexpr bool INTERIOR = decltype(interior_tag)::value;
        for (int i = tid; i < (NM_TH + 2) * (NM_MS / 4); i += 256) {
            const int ry = i / (NM_MS / 4), c0 = (i - ry * (NM_MS / 4)) * 4;
            // columns c0 .. c0+7 of the three source rows as two aligned words each; cell k reads bytes k+2 .. k+4.  The Sobel
            // sums are byte dot products (dp4a, unsigned pixels x signed taps): gx = rows (1,2,1) x (-1,0,1), gy = (bottom - top) x (1,2,1)
            uint32_t wa[3], wb[3];
#pragma unroll
            for (int k = 0; k < 3; k++) {
                wa[k] = *reinterpret_cast<const uint32_t*>(&sS[ry + k][c0]);
                wb[k] = *reinterpret_cast<const uint32_t*>(&sS[ry + k][c0 + 4]);
            }
            int m[4];
            const int y = Y0 - 1 + ry;
            const bool yin = (y >= 0 && y < P.h);
#pragma unroll
            for (int k = 0; k < 4; k++) {
                constexpr unsigned sel[4] = {0x5432u, 0x6543u, 0x7654u, 0x7765u};
                const uint32_t t = __byte_perm(wa[0], wb[0], sel[k]), c = __byte_perm(wa[1], wb[1], sel[k]), b = __byte_perm(wa[2], wb[2], sel[k]);
                const int gx = dp4a_us(b, 0x000100ffu, dp4a_us(c, 0x000200feu, dp4a_us(t, 0x000100ffu, 0)));
                const int gy = dp4a_us(b, 0x00010201u, dp4a_us(t, 0x00fffeffu, 0));
                // direction (cv.Canny, L2gradient: tan 22.5 = 13573 / 2^15): |gy| < |gx| tan 22.5 -> horizontal neighbours,
                // |gy| > |gx| tan 67.5 -> vertical, else the diagonal on which gx and gy have the same / opposite sign
                const int ax = abs(gx), ay = abs(gy) << 15;
                const int tg22x = ax * 13573, tg67x = tg22x + (ax << 16);
                const int nh = ay >= tg22x, dg = nh && !(ay > tg67x), pos = dg && ((gx ^ gy) >= 0);
                int v = ((gx * gx + gy * gy) << 2) + nh + dg + pos;
                if (!INTERIOR) {
                    const int x = X0 - 1 + c0 + k;
                    v = (yin && x >= 0 && x < P.w) ? v : 0;
                }
                m[k] = v;
            }
            *reinterpret_cast<int4*>(&sM[ry][c0]) = make_int4(m[0], m[1], m[2], m[3]);
        }
    };
    if (X0 >= 1 && X0 + NM_MS - 1 <= P.w && Y0 >= 1 && Y0 + NM_TH + 1 <= P.h) sobel(std::true_type{});
    else sobel(std::false_type{});
    __syncthreads();
    // stage 3: NMS + double threshold, 4 px per thread; a warp covers 2 rows x 64 px = 4 bitmap words.  Branch-free: the two
    // neighbours along the gradient are picked with selects on the direction class.  m < 2^21, so thresholds above 2^22 are
    // equivalent to 2^22 and 4 thr + 3 cannot overflow; c > 4 thr + 3  <=>  m > thr.
    const int low4 = min(P.thr[0], 1 << 22) * 4 + 3, high4 = min(P.thr[1], 1 << 22) * 4 + 3;
    const int lane = tid & 31;
    const int gx4 = (tid & 15) * 4;                                // first of the 4 px inside the tile row
#pragma unroll 2
    for (int half = 0; half < NM_TH / 16; half++) {
        const int ty = (tid >> 4) + half * 16;
        const int y = Y0 + ty;
        // rows ty, ty+1, ty+2 of sM (pixel rows y-1, y, y+1), columns gx4 .. gx4+5 (pixel x-1 .. x+4)
        int mg[3][6];
#pragma unroll
        for (int k = 0; k < 3; k++) {
            const int4 a = *reinterpret_cast<const int4*>(&sM[ty + k][gx4]);
            const int2 b = *reinterpret_cast<const int2*>(&sM[ty + k][gx4 + 4]);
            mg[k][0] = a.x; mg[k][1] = a.y; mg[k][2] = a.z; mg[k][3] = a.w; mg[k][4] = b.x; mg[k][5] = b.y;
        }
        unsigned sb = 0, wb = 0;
#pragma unroll
        for (int k = 0; k < 4; k++) {
            const int c = mg[1][k + 1];
            const int d = c & 3;
            // d = 0: left / right, 1: up / down, 2: up-right / down-left (gx, gy of opposite sign), 3: up-left / down-right
            const int d1 = d & 1, d2 = d & 2;
            const int n1 = selnz(selnz(mg[0][k], mg[0][k + 2], d1), selnz(mg[0][k + 1], mg[1][k], d1), d2);
            const int n2 = selnz(selnz(mg[2][k + 2], mg[2][k], d1), selnz(mg[2][k + 1], mg[1][k + 2], d1), d2);
            // m > m(n1), and m >= m(n2) along the axes / m > m(n2) on the diagonals (the asymmetry of cv.Canny's NMS)
            const int c_gt = c & ~3;
            const int c2 = selnz(c_gt - 1, c | 3, d2);
            const int keep = (c > low4) & (c_gt > n1) & (c2 >= n2);
            const int strong = keep & (c > high4);
            sb |= (unsigned)strong << k;
            wb |= (unsigned)(keep ^ strong) << k;
        }
        // OR the nibbles of 8 neighbouring lanes into one 32-bit word
        sb <<= 4 * (lane & 7); wb <<= 4 * (lane & 7);
#pragma unroll
        for (int o = 1; o < 8; o <<= 1) { sb |= __shfl_xor_sync(0xffffffffu, sb, o); wb |= __shfl_xor_sync(0xffffffffu, wb, o); }
        const int word = (X0 + gx4) >> 5;
        if ((lane & 7) == 0 && y < P.h && word < P.wpr) {
            P.strong[(size_t)y * P.wpr + word] = sb;
            P.weak[(size_t)y * P.wpr + word] = wb;
        }
    }
}

// ---------------------------------------------------------------------------------------------
// hysteresis: strong |= weak pixels 8-connected (through weak pixels) to a strong pixel.
// Bit-packed frontier propagation without grid-wide barriers.  A tile is 8 words x 32 rows (256 x 32 px), one
// word per thread; a CTA takes a tile to local convergence in shared memory (word-parallel 3x3 spread + in-word
// flood), ORs the new bits into the global bitmap and -- if bits on the tile's border changed -- pushes the (up to
// 8) neighbour tiles that can see them onto a global work queue.  One persistent kernel; a CTA that needs work
// takes a re-visit from the queue if there is one (they sit on the critical path), else the next tile that has not
// had its first pass, else it exits -- nobody ever waits for anybody: a push is always followed by its own CTA
// looking at the queue again, so the queue drains, and idle CTAs leave the SMs to whatever else is running.
// The result is the fixed point reach(strong) through weak pixels, which does not depend on the order of the
// passes (reach(S u T) = reach(S) u reach(T), bits are only ever set, stores are atomic ORs), so asynchronous
// propagation is bit-identical to the round-synchronous version it replaces.
//
// flags[t] != 0: tile t is queued or has not had its first pass (its next pass will load after any store that
// precedes a push attempt, so the push can be dropped).  ring: tile ids, -1 = empty slot, capacity >= 2 x tiles.
// ctrl (one 128-byte line each): [0] head  [32] tail  [64] next first-pass tile  [96] abort  [128] published entries not yet
// claimed (a counting semaphore: a pop is one atomicSub + one atomicAdd, never a compare-and-swap retry loop -- with a
// thousand CTAs looking for work at once, CAS retries on one word were 98 % of the first version's run time)
// ---------------------------------------------------------------------------------------------
constexpr int HY_WW = 8, HY_TR = 32;
constexpr int HY_THREADS = HY_WW * HY_TR;
constexpr int HY_SS = HY_WW + 3;                      // smem row stride (odd: lanes that differ in the row hit different banks)
constexpr int HY_HEAD = 0, HY_TAIL = 32, HY_NEXT = 64, HY_ABORT = 96, HY_AVAIL = 128, HY_CTRL_INTS = 160;
constexpr long long HY_SPIN_LIMIT = 20000000;         // a slot that is never published must not hang the GPU

struct HystQueue { int* flags; int* ring; int* ctrl; int ring_mask; int ntiles; };

__device__ __forceinline__ unsigned spread3(unsigned L, unsigned Cw, unsigned R) {
    return Cw | (Cw << 1) | (Cw >> 1) | (L >> 31) | (R << 31);
}
__device__ __forceinline__ int ld_gpu(const int* p) {                     // one L2 read, gpu scope (a plain volatile load is system scope)
    int v;
    asm volatile("ld.relaxed.gpu.global.s32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}

// one pass over one tile: local convergence, atomic write-back, neighbour pushes
__device__ __forceinline__ void hyst_process_tile(const PlaneDesc* __restrict__ planes, const TileMap& tm, int tile, const HystQueue& q,
                                                  unsigned (*sS)[HY_SS], int* sNbr) {
    const int tid = threadIdx.x, tr = tid & 31, tc = tid >> 5;     // warp = word column, lane = row
    int plane_i, txi, tyi;
    tile_decode(tm, tile, plane_i, txi, tyi);
    const PlaneDesc& P = planes[plane_i];
    const int ntx = aeaj_cdiv(P.wpr, HY_WW);
    const int gy0 = tyi * HY_TR, gw0 = txi * HY_WW;
    __syncthreads();                                               // the previous pass is done with sS / sNbr
    if (tid == 0) *sNbr = 0;
    for (int i = tid; i < (HY_TR + 2) * (HY_WW + 2); i += HY_THREADS) {
        const int ry = i / (HY_WW + 2), rw = i - ry * (HY_WW + 2);
        const int gy = gy0 + ry - 1, gw = gw0 + rw - 1;
        unsigned v = 0;
        if (gy >= 0 && gy < P.h && gw >= 0 && gw < P.wpr) v = __ldcg(P.strong + (size_t)gy * P.wpr + gw);
        sS[ry][rw] = v;
    }
    const int gw = gw0 + tc, gy = gy0 + tr;
    const bool inb = (gy < P.h && gw < P.wpr);
    const unsigned wk = inb ? __ldg(P.weak + (size_t)gy * P.wpr + gw) : 0u;
    __syncthreads();
    const unsigned s_init = sS[tr + 1][tc + 1];
    unsigned s = s_init;
    for (;;) {
        const unsigned n = spread3(sS[tr][tc], sS[tr][tc + 1], sS[tr][tc + 2]) |
                           spread3(sS[tr + 1][tc], s, sS[tr + 1][tc + 2]) |
                           spread3(sS[tr + 2][tc], sS[tr + 2][tc + 1], sS[tr + 2][tc + 2]);
        unsigned add = wk & ~s & n;
        unsigned t = s | add;
        while (add) { add = wk & ~t & ((t << 1) | (t >> 1)); t |= add; }       // flood along the row inside the word
        const int ch = (t != s);
        __syncthreads();
        if (ch) { s = t; sS[tr + 1][tc + 1] = s; }
        if (!__syncthreads_or(ch)) break;
    }
    unsigned nb = 0;
    if (inb && s != s_init) {
        atomicOr(P.strong + (size_t)gy * P.wpr + gw, s);
        // which of the 8 neighbours can see the new bits (bit index = (dy+1)*3 + (dx+1))
        const unsigned diff = s ^ s_init;
        const bool L = (tc == 0) && (diff & 1u), R = (tc == HY_WW - 1) && (diff >> 31);
        if (tr == 0) nb |= 2u | (L ? 1u : 0u) | (R ? 4u : 0u);
        if (tr == HY_TR - 1) nb |= 128u | (L ? 64u : 0u) | (R ? 256u : 0u);
        if (L) nb |= 8u;
        if (R) nb |= 32u;
    }
    if (nb) atomicOr(sNbr, (int)nb);
    __syncthreads();
    if (*sNbr == 0) return;                                                    // nothing a neighbour could see (uniform)
    // ONE gpu-scope fence per pass that pushes (a fence invalidates the SM's L1, so not one per thread): it orders the
    // atomic ORs of all threads of the CTA (observed through the barrier above) before the pushes below
    if (tid == 0) __threadfence();
    __syncthreads();
    if (tid < 9 && tid != 4 && ((*sNbr >> tid) & 1)) {
        const int dy = tid / 3 - 1, dx = tid % 3 - 1;
        const int nx = txi + dx, ny = tyi + dy;
        if (nx >= 0 && nx < ntx && ny >= 0 && ny * HY_TR < P.h) {
            const int nt = tile + dy * ntx + dx;                               // tiles of a plane are consecutive, row-major
            if (atomicExch(&q.flags[nt], 1) == 0) {                            // processed before and not queued: queue a re-visit
                const int slot = atomicAdd(&q.ctrl[HY_TAIL], 1) & q.ring_mask;
                long long spins = 0;
                while (atomicCAS(&q.ring[slot], -1, nt) != -1)                 // the slot's previous ticket has not been read yet
                    if (++spins > HY_SPIN_LIMIT) { atomicExch(&q.ctrl[HY_ABORT], 1); break; }
                // published (the CAS above has returned): one more entry may be claimed.  The value-returning form makes the
                // increment complete before this CTA looks at the counter again after the barrier.
                if (atomicAdd(&q.ctrl[HY_AVAIL], 1) == 0x7fffffff) atomicExch(&q.ctrl[HY_ABORT], 1);
            }
        }
    }
}

__global__ void __launch_bounds__(HY_THREADS) k_hysteresis(const PlaneDesc* __restrict__ planes, const __grid_constant__ TileMap tm, HystQueue q,
                                                           int* __restrict__ status) {
    __shared__ unsigned sS[HY_TR + 2][HY_SS];
    __shared__ int sNbr, sTile;
    const int tid = threadIdx.x;
    for (;;) {
        __syncthreads();                                                       // pushes of the previous pass are out; sTile is free
        if (tid == 0) {
            int t = -1;
            if (ld_gpu(&q.ctrl[HY_AVAIL]) > 0) {                               // 1. a queued re-visit
                if (atomicSub(&q.ctrl[HY_AVAIL], 1) > 0) {                     // claimed one published entry: the ticket below exists
                    const int slot = atomicAdd(&q.ctrl[HY_HEAD], 1) & q.ring_mask;
                    long long spins = 0;
                    while ((t = ld_gpu(&q.ring[slot])) == -1)                  // (an earlier ticket whose pusher is between its two atomics)
                        if (++spins > HY_SPIN_LIMIT) { atomicExch(&q.ctrl[HY_ABORT], 1); break; }
                    if (t >= 0) atomicExch(&q.ring[slot], -1);
                } else atomicAdd(&q.ctrl[HY_AVAIL], 1);                        // lost the race for the last entry: give the count back
            }
            if (t < 0 && ld_gpu(&q.ctrl[HY_NEXT]) < q.ntiles) {           // 2. a tile that has not had its first pass
                const int f = atomicAdd(&q.ctrl[HY_NEXT], 1);
                if (f < q.ntiles) t = f;
            }
            // from here on a neighbour's new bits need a new push.  No fence: the loads of the pass read L2 (ld.cg) and are issued
            // after this atomic has returned (barrier below), so they see every store that preceded a dropped push
            if (t >= 0 && atomicExch(&q.flags[t], 0) == 0x7fffffff) t = -1;    // (never true: forces the value-returning form)
            sTile = t;
        }
        __syncthreads();
        const int tile = sTile;
        if (tile < 0) break;                                                   // 3. nothing to do: leave (whoever pushes later pops later)
        hyst_process_tile(planes, tm, tile, q, sS, &sNbr);
    }
    if (tid == 0 && status) {                                                  // the last CTAs to leave write the final values
        status[0] = ld_gpu(&q.ctrl[HY_TAIL]);                             // tile re-visits in total
        status[1] = ld_gpu(&q.ctrl[HY_ABORT]) ? 0 : 1;                    // converged
    }
}

// final strong bitmap -> uint8 {0,1} map (API / taps) and the reverse (stage API)
__global__ void __launch_bounds__(256) k_bitmap_to_u8(const PlaneDesc* __restrict__ planes) {
    const PlaneDesc& P = planes[blockIdx.z];
    uint8_t* out = P.tap_edge;
    int x = blockIdx.x * 256 + threadIdx.x, y = blockIdx.y;
    if (!out || y >= P.h || x >= P.w) return;
    out[(size_t)y * P.w + x] = (P.strong[(size_t)y * P.wpr + (x >> 5)] >> (x & 31)) & 1u;
}
__global__ void __launch_bounds__(256) k_u8_to_bitmap(const uint8_t* __restrict__ edge, int h, int w, int wpr, uint32_t* __restrict__ bits) {
    int word = blockIdx.x * 8 + (threadIdx.x >> 5), y = blockIdx.y, lane = threadIdx.x & 31;
    if (word >= wpr) return;
    int x = word * 32 + lane;
    unsigned b = __ballot_sync(0xffffffffu, x < w && edge[(size_t)y * w + x] == 1);
    if (lane == 0) bits[(size_t)y * wpr + word] = b;
}

int max_dim(const PlaneDesc* P, int n, bool width) {
    int m = 0;
    for (int i = 0; i < n; i++) m = std::max(m, width ? P[i].w : P[i].h);
    return m;
}

}  // namespace

int aeaj_canny_init_constants() {
    float color[256], space[13];
    int dy[13], dx[13];
    double cc = -0.5 / (75.0 * 75.0), sc = -0.5 / (75.0 * 75.0);
    for (int i = 0; i < 256; i++) color[i] = (float)exp((double)(i * i) * cc);
    int k = 0;
    for (int i = -2; i <= 2; i++)
        for (int j = -2; j <= 2; j++) {
            double r = sqrt((double)i * i + (double)j * j);
            if (r > 2) continue;
            space[k] = (float)exp(r * r * sc); dy[k] = i; dx[k] = j; k++;
        }
    AEAJ_CUDA(cudaMemcpyToSymbol(c_bil_color, color, sizeof color));
    AEAJ_CUDA(cudaMemcpyToSymbol(c_bil_space, space, sizeof space));
    AEAJ_CUDA(cudaMemcpyToSymbol(c_bil_dy, dy, sizeof dy));
    AEAJ_CUDA(cudaMemcpyToSymbol(c_bil_dx, dx, sizeof dx));
    return 0;
}

int launch_clahe_hist(const PlaneDesc* planes_dev, const PlaneDesc* P, int nplanes, cudaStream_t st) {
    int maxth = 0;
    for (int i = 0; i < nplanes; i++) maxth = std::max(maxth, clahe_geom(P[i].h, P[i].w).th);
    dim3 grd(aeaj_cdiv(maxth, HIST_ROWS), 16, nplanes);
    k_clahe_hist<<<grd, 256, 0, st>>>(planes_dev);
    AEAJ_LAUNCH_CHECK();
    return 0;
}
int launch_clahe_lut(const PlaneDesc* planes_dev, int nplanes, const PeerSet& peers, cudaStream_t st) {
    k_clahe_lut<<<dim3(16, nplanes), 256, 0, st>>>(planes_dev, peers);
    AEAJ_LAUNCH_CHECK();
    return 0;
}
int launch_prefilter(const PlaneDesc* planes_dev, const PlaneDesc* P, int nplanes, int stages, int do_hist, cudaStream_t st) {
    const TileMap tm = make_tile_map(P, nplanes, PF_TW, PF_TH);
    k_prefilter<<<tile_map_total(tm, nplanes), 256, 0, st>>>(planes_dev, tm, stages, do_hist);
    AEAJ_LAUNCH_CHECK();
    return 0;
}
int launch_hist_u8(const uint8_t* src, size_t n, unsigned int* hist, cudaStream_t st) {
    int blocks = (int)std::min<size_t>((n + 4095) / 4096, 148 * 8);
    k_hist_u8<<<std::max(blocks, 1), 256, 0, st>>>(src, n, hist);
    AEAJ_LAUNCH_CHECK();
    return 0;
}
int launch_thresholds(const PlaneDesc* planes_dev, int nplanes, const PeerSet& peers, cudaStream_t st) {
    k_thresholds<<<aeaj_cdiv(nplanes, 4), 128, 0, st>>>(planes_dev, nplanes, peers);
    AEAJ_LAUNCH_CHECK();
    return 0;
}
int launch_thresholds_from_double(const double* thr_d, int* thr, cudaStream_t st) {
    k_thresholds_from_double<<<1, 1, 0, st>>>(thr_d, thr);
    AEAJ_LAUNCH_CHECK();
    return 0;
}
int launch_canny_nms(const PlaneDesc* planes_dev, const PlaneDesc* P, int nplanes, cudaStream_t st) {
    const TileMap tm = make_tile_map(P, nplanes, NM_TW, NM_TH);
    k_canny_nms<<<tile_map_total(tm, nplanes), 256, 0, st>>>(planes_dev, tm);
    AEAJ_LAUNCH_CHECK();
    return 0;
}

// number of hysteresis tiles of a batch (the tile index space of make_tile_map(.., 256, 32)) and the ring capacity
int hysteresis_tiles(PlaneDesc* P, int nplanes, int* ring_cap) {
    const TileMap tm = make_tile_map(P, nplanes, HY_WW * 32, HY_TR);
    const int ns = tile_map_total(tm, nplanes);
    int cap = 64;
    while (cap < 2 * ns) cap *= 2;
    *ring_cap = cap;
    return ns;
}
int hysteresis_ctrl_ints() { return HY_CTRL_INTS; }

int aeaj_canny_init(aeaj_handle* h) {
    int rc = aeaj_canny_init_constants(); if (rc) return rc;
    AEAJ_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&h->hyst_blocks_per_sm, k_hysteresis, HY_THREADS, 0));
    if (h->hyst_blocks_per_sm < 1) { aeaj_set_error("hysteresis kernel cannot be resident"); return AEAJ_EINVAL; }
    return 0;
}

// flags: int[ntiles]; ring: int[ring_cap]; ctrl: int[hysteresis_ctrl_ints()]
int launch_hysteresis(aeaj_handle* h, const PlaneDesc* planes_dev, const PlaneDesc* planes_host, int nplanes, int ntiles, int ring_cap,
                      int* flags, int* ring, int* ctrl, int* status, cudaStream_t st) {
    AEAJ_CUDA(cudaMemsetAsync(flags, 1, sizeof(int) * (size_t)ntiles, st));
    AEAJ_CUDA(cudaMemsetAsync(ring, 0xff, sizeof(int) * (size_t)ring_cap, st));
    AEAJ_CUDA(cudaMemsetAsync(ctrl, 0, sizeof(int) * HY_CTRL_INTS, st));
    HystQueue q;
    q.flags = flags; q.ring = ring; q.ctrl = ctrl; q.ring_mask = ring_cap - 1; q.ntiles = ntiles;
    const TileMap tm = make_tile_map(planes_host, nplanes, HY_WW * 32, HY_TR);
    const int grid = std::max(1, std::min(ntiles, h->hyst_blocks_per_sm * h->sm_count));
    k_hysteresis<<<grid, HY_THREADS, 0, st>>>(planes_dev, tm, q, status);
    AEAJ_LAUNCH_CHECK();
    return 0;
}

int launch_bitmap_to_u8(const PlaneDesc* planes_dev, const PlaneDesc* P, int nplanes, cudaStream_t st) {
    dim3 grd(aeaj_cdiv(max_dim(P, nplanes, true), 256), max_dim(P, nplanes, false), nplanes);
    k_bitmap_to_u8<<<grd, 256, 0, st>>>(planes_dev);
    AEAJ_LAUNCH_CHECK();
    return 0;
}
int launch_u8_to_bitmap(const uint8_t* edge, int h, int w, uint32_t* bits, cudaStream_t st) {
    int wpr = aeaj_cdiv(w, 32);
    k_u8_to_bitmap<<<dim3(aeaj_cdiv(wpr, 8), h), 256, 0, st>>>(edge, h, w, wpr, bits);
    AEAJ_LAUNCH_CHECK();
    return 0;
}
