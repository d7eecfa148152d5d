// aeaj_internal.cuh -- shared declarations for libaeaj.so (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include "pqfast.h"
#include <stdint.h>
#include <stdio.h>
#include <algorithm>
#include <type_traits>
#include <vector>
#include <string.h>
#include "../../include/aeaj.h"

// ---------------------------------------------------------------------------------------------
// error plumbing
// ---------------------------------------------------------------------------------------------
void aeaj_set_error(const char* fmt, ...);
#define AEAJ_CUDA(call)                                                                     \
    do {                                                                                    \
        cudaError_t e_ = (call);                                                            \
        if (e_ != cudaSuccess) {                                                            \
            aeaj_set_error("%s failed at %s:%d: %s", #call, __FILE__, __LINE__,             \
                           cudaGetErrorString(e_));                                         \
            return (int)e_;                                                                 \
        }                                                                                   \
    } while (0)
#define AEAJ_LAUNCH_CHECK()                                                                 \
    do {                                                                                    \
        cudaError_t e_ = cudaGetLastError();                                                \
        if (e_ != cudaSuccess) {                                                            \
            aeaj_set_error("kernel launch failed at %s:%d: %s", __FILE__, __LINE__,         \
                           cudaGetErrorString(e_));                                         \
            return (int)e_;                                                                 \
        }                                                                                   \
    } while (0)
#define AEAJ_REQUIRE(cond, msg)                                                             \
    do {                                                                                    \
        if (!(cond)) { aeaj_set_error("%s (%s:%d)", msg, __FILE__, __LINE__); return AEAJ_EINVAL; } \
    } while (0)

// ---------------------------------------------------------------------------------------------
// geometry shared by host and device
// ---------------------------------------------------------------------------------------------
struct ColorConsts {          // per colour space; passed to the kernels by value (kernel parameters)
    float fwd1[9], fwd2[9];   // forward: XYZ->LMS, LMS'->space   (linear spaces: fwd1 = the 3x3)
    float inv1[9], inv2[9];   // inverse: space->LMS', LMS->XYZ   (linear spaces: inv1 = the 3x3)
    float mid[3], scale[3];   // normalisation (MIDPOINTS / SCALE_FACTORS)
    int fast;                 // 1: try the table-driven transfer functions first (pqfast.h), 0: exact float64 path only
    PqTabs pq;                // views over the handle's device tables
};

// one image over several GPUs (peer.cu): ranks share their plan workspaces; a buffer of rank r is reached by adding
// delta[r] (bytes) to the address of this rank's copy
#define AEAJ_MAX_PEERS 8
struct PeerSeg { const void* src; void* dst; long long bytes; };
struct PeerSet { int world, rank; long long delta[AEAJ_MAX_PEERS]; };

// one "plane" = one layer of one image
struct PlaneGeom {
    int h, w;          // layer size
    int wpr;           // bitmap words per row = ceil(w/32)
    int root;          // quadtree root size
    int top;           // top block size T = min(max_block, root)
    int ntx, nty;      // in-bounds top blocks per axis
};

static inline __host__ __device__ int aeaj_cdiv(int a, int b) { return (a + b - 1) / b; }
static inline __host__ __device__ int64_t aeaj_cdiv64(int64_t a, int64_t b) { return (a + b - 1) / b; }

// BORDER_REFLECT_101 with OpenCV's loop (valid for any p, any len >= 1)
static inline __host__ __device__ int reflect101(int p, int len) {
    if (len == 1) return 0;
    while (p < 0 || p >= len) { if (p < 0) p = -p; else p = 2 * (len - 1) - p; }
    return p;
}
static inline __host__ __device__ int clampi(int p, int lo, int hi) { return p < lo ? lo : (p > hi ? hi : p); }
// np.pad(mode='reflect') index for position p >= 0 in a length-n axis (n==1 replicates)
static inline __host__ __device__ int pad_reflect(int p, int n) {
    if (n == 1) return 0;
    int period = 2 * (n - 1);
    p %= period;
    return p < n ? p : period - p;
}

#ifdef __CUDACC__
// np.round(block / qmatrix) (jpeg.py:501): the quotient is formed in float64 and rounded half-to-even.
// A float32 z is never closer than 2^-24 (relative) to a half-integer multiple of q without being exactly on
// it, so rounding the float64 quotient equals rounding the exact quotient -- which is computed here without any
// float64: k = rint(z * ~1/q) is within one of the answer (an approximate MUFU.RCP reciprocal is enough), the
// residual r = z - k*q is exact in one fma (except for k = +-1 chosen when |z/q| is just below 1/2, where either
// rounding of r leads to the same decision), and comparing 2|r| with q -- ties to even -- repairs k.
// The comparison runs on the bit patterns (positive floats order like integers): 2|r| is |r| + one exponent step,
// and adding the parity of k turns "greater" into "greater or equal" exactly when the tie must move to the even side.
// Branch-free, 13 instructions.  Checked against the float64 formula on 30 M values incl. ties and neighbours.
__device__ __forceinline__ int quantize_f(float z, float fq) {
    float rq;
    asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(rq) : "f"(fq));
    const int ki = __float2int_rn(__fmul_rn(z, rq));
    const int rb = __float_as_int(__fmaf_rn(-(float)ki, fq, z));
    const int c = (rb & 0x7fffffff) + (ki & 1) + 0x00800000;
    const int s = (rb >> 31) | 1;
    return ki + ((c > __float_as_int(fq)) ? s : 0);
}
__device__ __forceinline__ int quantize(float z, int q) { return quantize_f(z, (float)q); }
#endif

static inline __host__ __device__ int ilog2i(int v) { int l = 0; while ((1 << l) < v) l++; return l; }

// utils.py:24-41 + quadtree.py:89-90
static inline __host__ __device__ int aeaj_root_size(int h, int w) {
    int n = h > w ? h : w;
    if (n <= 2) return n * 2;
    int p = 1;
    while (p * 2 < n) p *= 2;
    return p * 2;
}

// Morton helpers: z = interleave(y,x), x in even bits (TL,TR,BL,BR child order)
static inline __host__ __device__ uint32_t compact1by1(uint32_t v) {
    v &= 0x55555555u;
    v = (v | (v >> 1)) & 0x33333333u;
    v = (v | (v >> 2)) & 0x0f0f0f0fu;
    v = (v | (v >> 4)) & 0x00ff00ffu;
    v = (v | (v >> 8)) & 0x0000ffffu;
    return v;
}
static inline __host__ __device__ uint32_t part1by1(uint32_t v) {
    v &= 0x0000ffffu;
    v = (v | (v << 8)) & 0x00ff00ffu;
    v = (v | (v << 4)) & 0x0f0f0f0fu;
    v = (v | (v << 2)) & 0x33333333u;
    v = (v | (v << 1)) & 0x55555555u;
    return v;
}

// ---------------------------------------------------------------------------------------------
// handle / plan
// ---------------------------------------------------------------------------------------------
struct aeaj_handle {
    int device;
    int sm_count;
    int hyst_blocks_per_sm;       // occupancy of k_hysteresis on this device (aeaj_canny_init)
    ColorConsts colors_host[8];
    ColorConsts* colors_dev;      // [8]
    double* pq_tabs_dev;          // the fixed-exponent power tables of pqfast.h (one allocation; colors_host[*].pq points into it)
    double pq_worst_eps;          // largest error bound among them (diagnostic)
    float* srgb_lut_dev;          // 256 floats, 0 until aeaj_set_srgb_lut
    int has_srgb_lut;
    float* dct_dev[9];            // DCT-II matrices C (s x s, row-major) for s = 2^k, k = 1..8
    float* dct_all_dev;
    float* dct_half_dev[9];       // even/odd half tables for the CTA kernels (sizes 64, 128)
    float* dct_half_all_dev;
    int32_t* zz_dev[9];           // zigzag tables per log2(size), device
    int32_t* zz_all_dev;
    int32_t* izz_dev[9];          // inverse zigzag permutations per log2(size): row-major index -> stream position
    int32_t* izz_all_dev;
    int32_t* izz256_dev;          // izz_dev[8] (k_dct256)
    int32_t* tc_izz_dev[4];       // inverse zigzag permutations for 16 .. 128 (tensor-core kernels)
    int32_t* tc_izz_all_dev;
    float* dct_tc_tiles_dev;      // [size class 16..128][fwd, inv][Ah | Al]: block-diagonal DCT matrices for the tcgen05 path
    int* tc_err_dev;              // set by the tcgen05 kernel if a barrier wait timed out
};

// device-side description of every plane of a batch; lives in the plan's device memory
struct PlaneDesc {
    int h, w, wpr, root, top, ntx, nty, layer;
    int ry0, ry1;                     // rows of this plane the current call works on (halo-split bands); default [0, h)
    long long peer_up, peer_dn;       // byte deltas to the workspaces of the ranks that own the rows above ry0 / from ry1 on (0: this GPU)
    float mid, scale;
    float* layer_f32;        // downsampled un-normalised layer
    uint8_t* u8a;            // cast / stage ping
    uint8_t* u8b;            // stage pong (post-bilateral)
    uint32_t* strong;        // bitmaps [h][wpr]
    uint32_t* weak;
    uint32_t* clahe_hist;    // [16][256]
    uint8_t* clahe_lut;      // [16][256]
    uint32_t* hist;          // [256] post-bilateral histogram
    int* thr;                // low, high (ints, squared)
    double* thr_d;           // percentile values (float64) for the stage API
    int32_t* leaves;         // [cap][4]
    uint8_t* states;
    int32_t* coef;
    int32_t* counts;         // n_leaves, n_states, n_coef, root
    int2* tb_tot;            // per in-bounds top block: (n_states, n_leaves)
    int* tb_coef;            // per in-bounds top block: n_coef
    int4* tb_base;           // per in-bounds top block: state base, leaf base, coef base, -
    const int32_t* qtab[9];  // per log2(size)
    const float* qtabf[9];   // the same tables as float (tensor-core epilogue); null in single-plane stage calls
    const int32_t* zz[9];    // zigzag order per log2(size): stream index -> row-major index (jpeg.py:726-766)
    int zigzag;              // 1: coefficient streams are stored zigzag-ordered per block (the .ajpg layout)
    uint8_t* packed_states;  // optional: 2-bit MSB-first packing of `states` (jpeg.py:563-571)
    int64_t cap_leaves, cap_states, cap_coef;
    uint8_t* tap_edge;       // optional: the final edge map as uint8 {0,1} [h][w] (encode taps, Canny stage calls)
};

struct ClassEntry { int x, y, plane, coef_off; };

// exact 1-D grids over the tiles of all planes of a batch (no empty blocks for the smaller chroma planes):
// planes are ordered image-major with `nl` layers per image and identical geometry per layer.
struct TileMap { int per_image, nl; int cum[4]; int ntx[3]; };
static inline TileMap make_tile_map(const PlaneDesc* P, int nplanes, int tw, int th, bool square_top = false) {
    TileMap m;
    m.nl = nplanes >= 3 && (nplanes % 3) == 0 && P[0].layer == 0 && P[1].layer == 1 ? 3 : 1;
    int c = 0;
    for (int l = 0; l < 3; l++) {
        m.cum[l] = c;
        if (l < m.nl) {
            int nx = square_top ? P[l].ntx : aeaj_cdiv(P[l].w, tw), ny = square_top ? P[l].nty : aeaj_cdiv(P[l].h, th);
            m.ntx[l] = nx; c += nx * ny;
        } else m.ntx[l] = 1;
    }
    m.cum[3] = c; m.per_image = c;
    return m;
}
static inline int tile_map_total(const TileMap& m, int nplanes) { return m.per_image * (nplanes / m.nl); }
static inline __device__ void tile_decode(const TileMap& m, int bid, int& plane, int& tx, int& ty) {
    const int b = bid / m.per_image, r = bid - b * m.per_image;
    const int l = (r >= m.cum[2] && m.nl > 2) ? 2 : ((r >= m.cum[1] && m.nl > 1) ? 1 : 0);
    const int t = r - m.cum[l];
    ty = t / m.ntx[l]; tx = t - ty * m.ntx[l];
    plane = b * m.nl + l;
}

// one plane's coefficient stream in packed form (pack.cu)
struct PackPlane {
    const int32_t* coef;      // pack: in, unpack: out
    uint32_t* mask;           // [ceil(n / 32)]
    int16_t* vals;            // [nnz]
    const int32_t* n_coef;    // device: number of coefficients of this plane
    int32_t* pk_counts;       // device int32[4]: nnz, n_coef, overflow flag, mask words
    int* chunk_sums;          // scratch: per-chunk nnz, then exclusive offsets
    int64_t cap_coef;         // capacity of the stream buffers
};
size_t aeaj_pack_scratch_ints(int64_t cap_coef);
int launch_pack(const PackPlane* planes_dev, int nplanes, int64_t max_cap_coef, int unpack, cudaStream_t st);

// one plane's zlib stream (deflate.cu, deflate_core.h)
struct DeflatePlane {
    const uint8_t* in;        // the plane's int32 coefficient stream, as bytes
    const int32_t* n_coef;    // device: number of coefficients of this plane
    int64_t cap_coef;         // capacity of the coefficient buffer
    uint8_t* out;             // [cap_out]: the zlib stream
    int64_t cap_out;
    int32_t* length;          // device: bytes of `out` written (0 if the stream did not fit)
    int32_t* status;          // optional device counter of planes whose stream did not fit
    uint8_t* slots;           // scratch [chunks][DF_CHUNK_BOUND]: each chunk's deflate output
    uint16_t* tok;            // scratch [chunks][DF_CHUNK]: each chunk's tokens
    int32_t* chunk_len;       // scratch [chunks]
    uint32_t* chunk_adler;    // scratch [chunks]
    int64_t* chunk_off;       // scratch [chunks]
};
int aeaj_deflate_init();
int launch_deflate(const DeflatePlane* planes_dev, int nplanes, int max_chunks, cudaStream_t st);

// one plane's zlib stream -> its coefficient buffer (inflate.cu, inflate_core.h)
struct InflatePlane {
    const int64_t* offset;    // device: the stream's first byte in the input buffer
    const int64_t* length;    // device: its bytes
    const int32_t* n_coef;    // device: coefficients the stream must inflate to (4 bytes each)
    uint8_t* out;             // the plane's coefficient buffer, as bytes
    int64_t cap_bytes;
    int32_t* status;          // device: IF_* of inflate_core.h
    int64_t* out_bytes;       // device: bytes written
    int32_t* segments;        // device: merged segments decoded independently
};
struct IfSeg;
struct IfStream;
struct InflateArgs {
    const uint8_t* in;        // the input buffer
    int64_t in_bytes;
    int nplanes, cap_segs;    // candidate list: the planes' first segments, then up to cap_segs - nplanes sync points
    int* counters;            // [0] sync points found, [1] / [2] next candidate of the speculative / output pass
    IfStream* streams;        // [nplanes]
    IfSeg* segs;              // [cap_segs]
    int32_t* map;             // [in_bytes / 4 + 1]: input position >> 2 -> candidate index (-1: list full)
};
int launch_inflate(const InflatePlane* planes_dev, const InflateArgs& a, int sm_count, cudaStream_t st);

// kernels' host launchers (defined in the .cu files)
int aeaj_canny_init(aeaj_handle* h);
int aeaj_dct_init(aeaj_handle* h);

int launch_color_forward_planar(aeaj_handle* h, int space, const float* rgb, const uint8_t* rgb_u8, int B, int H, int W,
                                const PlaneDesc* planes_dev, const PlaneDesc* planes_host,
                                float* full_c1, float* full_c2, cudaStream_t st, int* launches, int band0 = 0, int band1 = -1);
int launch_color_pixels(aeaj_handle* h, int space, int inverse, const float* in, float* out, size_t n, cudaStream_t st);
int launch_normalize(const float* in, float* out, size_t n, float mid, float scale, int inverse, cudaStream_t st);
int launch_area(const float* src, int H, int W, float* dst, int dh, int dw, uint8_t* u8_out, int planes,
                size_t src_stride, size_t dst_stride, cudaStream_t st);
int launch_resize_linear(const float* src, int sh, int sw, float* dst, int H, int W, cudaStream_t st);
int launch_upsample_color_inverse(aeaj_handle* h, int space, const PlaneDesc* planes_host, int B, int H, int W,
                                  float* rgb, uint8_t* rgb_u8, cudaStream_t st, int band0 = 0, int band1 = -1);
int launch_peer_barrier(int* const* flags_host, int rank, int world, int epoch, int* err_dev, cudaStream_t st);
int aeaj_color_init(aeaj_handle* h);
int launch_peer_gather(const PeerSeg* segs_dev, int nseg, long long max_bytes, cudaStream_t st);
constexpr int AEAJ_SEGS_BY_PARAM = 64;
int launch_copy_segments_param(const PeerSeg* segs_host, int nseg, long long max_bytes, cudaStream_t st);
int launch_cast_u8(const float* in, uint8_t* out, size_t n, cudaStream_t st);

int launch_clahe_hist(const PlaneDesc* planes_dev, const PlaneDesc* planes_host, int nplanes, cudaStream_t st);
int launch_clahe_lut(const PlaneDesc* planes_dev, int nplanes, const PeerSet& peers, cudaStream_t st);
int launch_prefilter(const PlaneDesc* planes_dev, const PlaneDesc* planes_host, int nplanes, int stages, int do_hist, cudaStream_t st);
int launch_hist_u8(const uint8_t* src, size_t n, unsigned int* hist, cudaStream_t st);
int launch_thresholds(const PlaneDesc* planes_dev, int nplanes, const PeerSet& peers, cudaStream_t st);
int launch_thresholds_from_double(const double* thr_d, int* thr, cudaStream_t st);
int launch_canny_nms(const PlaneDesc* planes_dev, const PlaneDesc* planes_host, int nplanes, cudaStream_t st);
int hysteresis_tiles(PlaneDesc* planes_host, int nplanes, int* ring_cap);
int hysteresis_ctrl_ints();
int launch_hysteresis(aeaj_handle* h, const PlaneDesc* planes_dev, const PlaneDesc* planes_host, int nplanes, int ntiles, int ring_cap,
                      int* flags, int* ring, int* ctrl, int* status, cudaStream_t st);
int launch_bitmap_to_u8(const PlaneDesc* planes_dev, const PlaneDesc* planes_host, int nplanes, cudaStream_t st);
int launch_u8_to_bitmap(const uint8_t* edge, int h, int w, uint32_t* bits, cudaStream_t st);

int launch_quadtree(const PlaneDesc* planes_dev, const PlaneDesc* planes_host, int nplanes, int min_size, int max_size,
                    ClassEntry* class_lists, int* class_counts, const long long* class_offsets_dev, cudaStream_t st,
                    int* launches, int parts = 7);      // parts: 1 count per top block, 2 scan, 4 emit
int launch_pack_states(const PlaneDesc* planes_dev, const PlaneDesc* planes_host, int nplanes, cudaStream_t st);
int launch_bucket_leaves(const PlaneDesc* planes_dev, const PlaneDesc* planes_host, int nplanes, ClassEntry* class_lists,
                         int* class_counts, const long long* class_offsets_dev, int lg_min, int lg_max, cudaStream_t st);
int launch_dct_quant(aeaj_handle* h, const PlaneDesc* planes_dev, const ClassEntry* class_lists, const int* class_counts,
                     const int64_t* class_offsets_host, const int64_t* class_caps_host, int lg_min, int lg_max,
                     cudaStream_t st, int* launches, void (*mark)(void*, const char*), void* mark_ctx, int tensor_dct, float* scratch256);
size_t aeaj_dct256_scratch_floats();
int aeaj_dct_tc_init(aeaj_handle* h);
int launch_dct_tc(aeaj_handle* h, int size, const PlaneDesc* planes_dev, const ClassEntry* list, const int* count, int64_t cap, int inverse, cudaStream_t st);
int launch_dequant_idct(aeaj_handle* h, const PlaneDesc* planes_dev, const ClassEntry* class_lists, const int* class_counts,
                        const int64_t* class_offsets_host, const int64_t* class_caps_host, int lg_min, int lg_max,
                        cudaStream_t st, int* launches, void (*mark)(void*, const char*), void* mark_ctx, int tensor_dct, float* scratch256);
// scaled decode (idct_scaled.cu): the leaves of every class to the 1/m planes (the descriptors' layer_f32, ceil(h/m) x ceil(w/m)),
// and the box reduce of one layer's batch of planes [batch][sh][sw] by f
int aeaj_idct_scaled_init();
int launch_idct_scaled(aeaj_handle* h, const PlaneDesc* planes_dev, const ClassEntry* class_lists, const int* class_counts,
                       const int64_t* class_offsets_host, const int64_t* class_caps_host, int lg_min, int lg_max, int m,
                       cudaStream_t st, int* launches);
int launch_box_reduce(const float* src, int sh, int sw, float* dst, int dh, int dw, int f, int batch, cudaStream_t st);
