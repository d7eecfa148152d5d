// pack.cu -- lossless device-side packing of the quantised coefficient streams for the trip over PCIe (sm_100a).
//
// Once the hot path runs on the GPU, moving the int32 coefficient streams to the host-side entropy coder
// (jpeg.py:573-590) and back (jpeg.py:655-672) is two thirds of all bytes on the bus, and most of those bytes are
// zeros: quantisation leaves 10-20 % of the coefficients non-zero, and a coefficient of an orthonormal DCT of samples
// in [-127, 127] is bounded by 127 * size <= 32512, so it fits 16 bits.  Packed form of one plane's stream of n
// coefficients (any block layout -- row-major or zigzag):
//     mask : uint32[ceil(n / 32)]   bit i of word j set  <=>  coefficient 32 j + i is non-zero
//     vals : int16[nnz]             the non-zero coefficients in stream order
// 1/8 + 2 * nnz / n bytes per coefficient instead of 4.  A value outside int16 raises the plane's overflow flag
// and the caller moves that plane as int32 instead (never observed with the reference's normalisation).
//
// Three small HBM-bound kernels per direction: per-chunk popcounts, one scan per plane, emit.
#include "aeaj_internal.cuh"

namespace {

constexpr int PK_THREADS = 256;
constexpr int PK_CHUNK = PK_THREADS * 32;             // coefficients per CTA: every warp owns 32 mask words

__device__ __forceinline__ int plane_n(const PackPlane& P) { return (int)min((long long)max(*P.n_coef, 0), (long long)P.cap_coef); }

__device__ __forceinline__ int warp_sum(int v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

// block-wide exclusive scan of one int per warp (8 warps) -> offset of this warp, total
__device__ __forceinline__ int warp_offsets(int warp_total, int* smem, int& block_total) {
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    __syncthreads();
    if (lane == 0) smem[warp] = warp_total;
    __syncthreads();
    int off = 0, tot = 0;
#pragma unroll
    for (int k = 0; k < PK_THREADS / 32; k++) { const int t = smem[k]; if (k < warp) off += t; tot += t; }
    block_total = tot;
    return off;
}

// pass 1 (pack): mask words + per-chunk non-zero counts.   grid: (chunks, planes)
__global__ void __launch_bounds__(PK_THREADS) k_pack_count(const PackPlane* __restrict__ planes) {
    const PackPlane P = planes[blockIdx.y];
    const int n = plane_n(P);
    const long long base = (long long)blockIdx.x * PK_CHUNK;
    if (base >= n) return;
    __shared__ int s_w[PK_THREADS / 32];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const long long wbase = base + (long long)warp * 1024;
    unsigned my_word = 0;
    int ovf = 0;
#pragma unroll 4
    for (int j = 0; j < 32; j++) {
        const long long i = wbase + j * 32 + lane;
        const int v = (i < n) ? __ldg(P.coef + i) : 0;
        ovf |= (v > 32767 || v < -32768);
        const unsigned m = __ballot_sync(0xffffffffu, v != 0);
        if (lane == j) my_word = m;
    }
    const long long word = (wbase >> 5) + lane;
    if (word * 32 < n) P.mask[word] = my_word;
    int tot;
    warp_offsets(warp_sum(__popc(my_word)), s_w, tot);
    if (threadIdx.x == 0) P.chunk_sums[blockIdx.x] = tot;
    if (__syncthreads_or(ovf) && threadIdx.x == 0) atomicOr(&P.pk_counts[2], 1);
}

// pass 1 (unpack): per-chunk popcounts of the mask words
__global__ void __launch_bounds__(PK_THREADS) k_unpack_count(const PackPlane* __restrict__ planes) {
    const PackPlane P = planes[blockIdx.y];
    const int n = plane_n(P);
    const long long base = (long long)blockIdx.x * PK_CHUNK;
    if (base >= n) return;
    __shared__ int s_w[PK_THREADS / 32];
    const long long word = (base >> 5) + threadIdx.x;
    const unsigned w = (word * 32 < n) ? __ldg(P.mask + word) : 0u;
    int tot;
    warp_offsets(warp_sum(__popc(w)), s_w, tot);
    if (threadIdx.x == 0) P.chunk_sums[blockIdx.x] = tot;
}

// pass 2: exclusive scan of the chunk counts of one plane (one CTA per plane); total -> pk_counts (pack only)
__global__ void __launch_bounds__(PK_THREADS) k_pack_scan(const PackPlane* __restrict__ planes, int write_counts) {
    const PackPlane P = planes[blockIdx.x];
    const int n = plane_n(P);
    const int nchunks = (int)(((long long)n + PK_CHUNK - 1) / PK_CHUNK);
    __shared__ int s_w[PK_THREADS / 32];
    const int lane = threadIdx.x & 31;
    int carry = 0;
    for (int c0 = 0; c0 < nchunks; c0 += PK_THREADS) {
        const int c = c0 + threadIdx.x;
        const int v = (c < nchunks) ? P.chunk_sums[c] : 0;
        int inc = v;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) { const int t = __shfl_up_sync(0xffffffffu, inc, o); if (lane >= o) inc += t; }
        int tot;
        const int woff = warp_offsets(__shfl_sync(0xffffffffu, inc, 31), s_w, tot);
        if (c < nchunks) P.chunk_sums[c] = carry + woff + inc - v;
        carry += tot;
        __syncthreads();
    }
    if (threadIdx.x == 0 && write_counts) {
        P.pk_counts[0] = carry; P.pk_counts[1] = n; P.pk_counts[3] = (n + 31) / 32;
    }
}

// pass 3 (pack): the non-zero values, in stream order, as int16
__global__ void __launch_bounds__(PK_THREADS) k_pack_emit(const PackPlane* __restrict__ planes) {
    const PackPlane P = planes[blockIdx.y];
    const int n = plane_n(P);
    const long long base = (long long)blockIdx.x * PK_CHUNK;
    if (base >= n) return;
    __shared__ int s_w[PK_THREADS / 32];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const long long wbase = base + (long long)warp * 1024;
    const long long word = (wbase >> 5) + lane;
    const unsigned my_word = (word * 32 < n) ? P.mask[word] : 0u;           // written by k_pack_count
    int tot;
    int off = P.chunk_sums[blockIdx.x] + warp_offsets(warp_sum(__popc(my_word)), s_w, tot);
    const unsigned lt = (1u << lane) - 1u;
#pragma unroll 4
    for (int j = 0; j < 32; j++) {
        const unsigned m = __shfl_sync(0xffffffffu, my_word, j);
        if (m == 0) continue;                                               // uniform per warp
        const long long i = wbase + j * 32 + lane;
        if ((m >> lane) & 1u) P.vals[off + __popc(m & lt)] = (int16_t)__ldg(P.coef + i);
        off += __popc(m);
    }
}

// pass 3 (unpack): expand to the int32 stream
__global__ void __launch_bounds__(PK_THREADS) k_unpack_emit(const PackPlane* __restrict__ planes) {
    const PackPlane P = planes[blockIdx.y];
    const int n = plane_n(P);
    const long long base = (long long)blockIdx.x * PK_CHUNK;
    if (base >= n) return;
    __shared__ int s_w[PK_THREADS / 32];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const long long wbase = base + (long long)warp * 1024;
    const long long word = (wbase >> 5) + lane;
    const unsigned my_word = (word * 32 < n) ? __ldg(P.mask + word) : 0u;
    int tot;
    int off = P.chunk_sums[blockIdx.x] + warp_offsets(warp_sum(__popc(my_word)), s_w, tot);
    const unsigned lt = (1u << lane) - 1u;
    int32_t* out = const_cast<int32_t*>(P.coef);
#pragma unroll 4
    for (int j = 0; j < 32; j++) {
        const unsigned m = __shfl_sync(0xffffffffu, my_word, j);
        const long long i = wbase + j * 32 + lane;
        int v = 0;
        if ((m >> lane) & 1u) v = (int)__ldg(P.vals + off + __popc(m & lt));
        if (i < n) out[i] = v;
        off += __popc(m);
    }
}

}  // namespace

size_t aeaj_pack_scratch_ints(int64_t cap_coef) { return (size_t)(cap_coef / PK_CHUNK + 2); }

int launch_pack(const PackPlane* planes_dev, int nplanes, int64_t max_cap_coef, int unpack, cudaStream_t st) {
    const unsigned chunks = (unsigned)std::max<int64_t>(1, (max_cap_coef + PK_CHUNK - 1) / PK_CHUNK);
    dim3 grd(chunks, nplanes);
    if (!unpack) {
        k_pack_count<<<grd, PK_THREADS, 0, st>>>(planes_dev);
        AEAJ_LAUNCH_CHECK();
        k_pack_scan<<<nplanes, PK_THREADS, 0, st>>>(planes_dev, 1);
        AEAJ_LAUNCH_CHECK();
        k_pack_emit<<<grd, PK_THREADS, 0, st>>>(planes_dev);
        AEAJ_LAUNCH_CHECK();
    } else {
        k_unpack_count<<<grd, PK_THREADS, 0, st>>>(planes_dev);
        AEAJ_LAUNCH_CHECK();
        k_pack_scan<<<nplanes, PK_THREADS, 0, st>>>(planes_dev, 0);
        AEAJ_LAUNCH_CHECK();
        k_unpack_emit<<<grd, PK_THREADS, 0, st>>>(planes_dev);
        AEAJ_LAUNCH_CHECK();
    }
    return 0;
}
