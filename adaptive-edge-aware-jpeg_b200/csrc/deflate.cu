// deflate.cu -- device deflate of the .ajpg coefficient streams (sm_100a): one complete zlib stream per plane, the same
// bytes as the sequential definition in deflate_core.h.
//
// k_deflate_chunks: one CTA per 64 KiB chunk.  The chunk, its previous-occurrence table (uint16 per position) and the hash
// heads live in shared memory (~208 KiB, one CTA per SM).  All threads load the chunk, hash every position and form the
// Adler-32 partial sums; warp 0 links the positions into hash chains (32 positions per step, __match_any_sync) and then
// runs the lazy parse, its 32 lanes comparing 4 candidates x 32 bytes per step; thread 0 builds the Huffman codes and
// writes the block into the chunk's output slot.
// k_deflate_finish: per plane, chunk offsets, zlib header, combined Adler-32 trailer, length.
// k_deflate_gather: chunk slots -> their place in the plane's stream.
#include "aeaj_internal.cuh"
#include "deflate_core.h"

namespace {

constexpr int DF_THREADS = 256;

struct DfSmem {
    uint8_t data[DF_CHUNK + 16];
    uint16_t prev[DF_CHUNK];
    union {
        uint16_t head[1 << DF_HASH_BITS];
        DfWork work;
    } u;
    unsigned long long red[2][DF_THREADS / 32];
    int ntok;
};

__device__ __forceinline__ int64_t plane_bytes(const DeflatePlane& P) {
    return 4 * (int64_t)min((long long)max(*P.n_coef, 0), (long long)P.cap_coef);
}

// df_best_seq, with the 32 lanes of a warp: lanes 8k .. 8k + 7 compare candidate k, 4 bytes each per step.  Every lane
// returns the same result.
__device__ int df_best_warp(const uint8_t* d, const uint16_t* prev, int p, int n, int& dist) {
    int cand[DF_CANDIDATES];
    const int nc = df_candidates(prev, p, n, cand);
    if (nc == 0) return 0;
    const int lane = threadIdx.x & 31, k = lane >> 3, sub = lane & 7;
    const int maxlen = n - p < DF_MAX_MATCH ? n - p : DF_MAX_MATCH;
    int c = -1;
#pragma unroll
    for (int j = 0; j < DF_CANDIDATES; j++) if (j == k && j < nc) c = cand[j];
    int len = maxlen;
    bool done = c < 0;
    for (int off = 0; off < maxlen; off += 32) {
        int mm = 4;
        if (!done) {
#pragma unroll
            for (int j = 0; j < 4; j++) {
                const int q = off + sub * 4 + j;
                if (mm == 4 && q < maxlen && d[c + q] != d[p + q]) mm = j;
            }
        }
        const unsigned bad = __ballot_sync(0xffffffffu, mm < 4);
        const unsigned gb = (bad >> (k * 8)) & 0xffu;
        const int f = gb ? __ffs(gb) - 1 : 0;
        const int mmf = __shfl_sync(0xffffffffu, mm, k * 8 + f);
        if (!done && gb) { len = off + f * 4 + mmf; done = true; }
        if (__all_sync(0xffffffffu, done)) break;
    }
    int best = 0;
#pragma unroll
    for (int j = 0; j < DF_CANDIDATES; j++) {
        const int l = __shfl_sync(0xffffffffu, len, j * 8);
        if (j < nc && l > best) { best = l; dist = p - cand[j]; }
    }
    return best >= DF_MIN_MATCH ? best : 0;
}

__global__ void __launch_bounds__(DF_THREADS, 1) k_deflate_chunks(const DeflatePlane* __restrict__ planes) {
    const DeflatePlane P = planes[blockIdx.y];
    const int64_t nbytes = plane_bytes(P);
    const int nch = df_chunks(nbytes), c = blockIdx.x;
    if (c >= nch) return;
    extern __shared__ __align__(16) unsigned char df_smem_raw[];
    DfSmem& S = *reinterpret_cast<DfSmem*>(df_smem_raw);
    const int64_t start = (int64_t)c * DF_CHUNK;
    const int m = (int)min((int64_t)DF_CHUNK, nbytes - start);
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;

    const uint32_t* src = reinterpret_cast<const uint32_t*>(P.in + start);
    uint32_t* dw = reinterpret_cast<uint32_t*>(S.data);
    for (int i = tid; i < m / 4; i += DF_THREADS) dw[i] = __ldg(src + i);
    for (int h = tid; h < (1 << DF_HASH_BITS); h += DF_THREADS) S.u.head[h] = 0;
    __syncthreads();
    unsigned long long s1 = 0, s2 = 0;
    for (int i = tid; i < m; i += DF_THREADS) {
        const uint32_t v = S.data[i];
        s1 += v; s2 += (unsigned long long)(m - i) * v;
        S.prev[i] = (i + 4 <= m) ? (uint16_t)df_hash(S.data, i) : 0;
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) { s1 += __shfl_xor_sync(0xffffffffu, s1, o); s2 += __shfl_xor_sync(0xffffffffu, s2, o); }
    if (lane == 0) { S.red[0][warp] = s1; S.red[1][warp] = s2; }
    __syncthreads();

    if (warp == 0) {
        // hash chains: prev[i] = i - (latest earlier position with the same hash), as df_build_prev_seq
        const unsigned below = (1u << lane) - 1u;
        for (int base = 0; base < m; base += 32) {
            const int i = base + lane;
            const bool valid = i + 4 <= m;
            const int h = valid ? (int)S.prev[i] : (1 << 16) + lane;
            const unsigned grp = __match_any_sync(0xffffffffu, h);
            int pd = 0;
            if (valid) {
                const unsigned lower = grp & below;
                if (lower) pd = lane - (31 - __clz(lower));
                else { const int hd = S.u.head[h]; pd = hd ? i - (hd - 1) : 0; }
            }
            __syncwarp();
            if (valid && (grp >> lane) == 1u) S.u.head[h] = (uint16_t)(i + 1);
            if (i < m) S.prev[i] = (uint16_t)pd;
            __syncwarp();
        }
        uint16_t* tok = P.tok + (int64_t)c * DF_CHUNK;
        const int ntok = df_parse(S.data, m, [&](int p, int& dist) { return df_best_warp(S.data, S.prev, p, m, dist); },
                                  [&](int t, uint16_t v) { if (lane == 0) tok[t] = v; });
        if (lane == 0) S.ntok = ntok;
    }
    __syncthreads();
    if (tid == 0) {
        unsigned long long a = 0, b = 0;
        for (int w = 0; w < DF_THREADS / 32; w++) { a += S.red[0][w]; b += S.red[1][w]; }
        P.chunk_adler[c] = df_adler_from_sums(a, b, m);
        P.chunk_len[c] = df_encode_chunk(S.data, m, P.tok + (int64_t)c * DF_CHUNK, S.ntok, c == nch - 1,
                                         P.slots + (int64_t)c * DF_CHUNK_BOUND, &S.u.work);
    }
}

// per plane: chunk offsets, header, trailer, length; a stream that does not fit its buffer is counted in status[0]
__global__ void k_deflate_finish(const DeflatePlane* __restrict__ planes) {
    const DeflatePlane P = planes[blockIdx.x];
    if (threadIdx.x != 0) return;
    const int64_t nbytes = plane_bytes(P);
    const int nch = df_chunks(nbytes);
    int64_t off = 0;
    uint32_t adler = 1;
    for (int c = 0; c < nch; c++) {
        P.chunk_off[c] = off;
        off += P.chunk_len[c];
        adler = df_adler_combine(adler, P.chunk_adler[c], min((int64_t)DF_CHUNK, nbytes - (int64_t)c * DF_CHUNK));
    }
    const int64_t total = 2 + off + 4;
    if (total > P.cap_out) {
        *P.length = 0;
        if (P.status) atomicAdd(P.status, 1);
        return;
    }
    P.out[0] = 0x78; P.out[1] = 0x9c;
    for (int k = 0; k < 4; k++) P.out[2 + off + k] = (uint8_t)(adler >> (24 - 8 * k));
    *P.length = (int32_t)total;
}

__global__ void __launch_bounds__(DF_THREADS) k_deflate_gather(const DeflatePlane* __restrict__ planes) {
    const DeflatePlane P = planes[blockIdx.y];
    const int c = blockIdx.x;
    if (c >= df_chunks(plane_bytes(P)) || *P.length == 0) return;
    const uint8_t* s = P.slots + (int64_t)c * DF_CHUNK_BOUND;
    uint8_t* d = P.out + 2 + P.chunk_off[c];
    const int len = P.chunk_len[c];
    for (int i = threadIdx.x; i < len; i += DF_THREADS) d[i] = s[i];
}

}  // namespace

// function attributes are per device: aeaj_create calls this with the handle's device selected
int aeaj_deflate_init() {
    AEAJ_CUDA(cudaFuncSetAttribute(k_deflate_chunks, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(DfSmem)));
    return 0;
}

int launch_deflate(const DeflatePlane* planes_dev, int nplanes, int max_chunks, cudaStream_t st) {
    k_deflate_chunks<<<dim3(max_chunks, nplanes), DF_THREADS, sizeof(DfSmem), st>>>(planes_dev);
    AEAJ_LAUNCH_CHECK();
    k_deflate_finish<<<nplanes, 32, 0, st>>>(planes_dev);
    AEAJ_LAUNCH_CHECK();
    k_deflate_gather<<<dim3(max_chunks, nplanes), DF_THREADS, 0, st>>>(planes_dev);
    AEAJ_LAUNCH_CHECK();
    return 0;
}
