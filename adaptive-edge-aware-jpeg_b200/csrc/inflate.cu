// inflate.cu -- device inflate of the .ajpg coefficient streams (sm_100a): zlib streams -> the plan's coefficient buffers,
// with the result of the sequential definition in inflate_core.h (if_inflate_seq), segment count included.
//
// k_inflate_scan: per plane, every byte position right after 00 00 FF FF becomes a candidate segment start (appended to
//   one list; a position -> list index map); the byte after the zlib header is the plane's first candidate.
// k_inflate_spec: one warp per candidate decodes its blocks up to the next non-final empty stored block (or the end of the
//   final block) without writing: end, output length, status, how far before its start it copies from.  Candidates that
//   are not on the chain cost this pass and nothing else.
// k_inflate_chain: one thread per plane: header, then the chain from the first segment (if_chain), merging segments that
//   copy from before their start into the ones they need.
// k_inflate_output: one warp per merged segment decodes again, writes at its output offset (copies spread over the lanes:
//   out[s + k] = out[s - d + (k mod d)]) and forms the Adler-32 of what it wrote.
// k_inflate_finish: one thread per plane: trailer, status, bytes, segment count (if_finish).
// The decoders' tables live in shared memory, one set per warp.  Warps take candidates from a counter (persistent grid):
// segments differ in length by orders of magnitude.
#include "aeaj_internal.cuh"
#include "inflate_core.h"

namespace {

constexpr int IF_WARPS = 4;                     // per CTA: 4 x 6 KiB of tables

__device__ __forceinline__ int64_t stream_limit(const InflatePlane& P) {
    const int64_t want = 4 * (int64_t)max(*P.n_coef, 0);
    return min(want, P.cap_bytes);
}

// the plane's stream inside the input buffer, clamped to it (and to 2^31 - 16 bytes: positions are int32)
__device__ __forceinline__ void stream_range(const InflatePlane& P, int64_t in_bytes, int64_t& off, int64_t& len) {
    off = *P.offset; len = *P.length;
    if (off < 0 || off > in_bytes || len < 0) { off = 0; len = 0; }
    len = min(len, in_bytes - off);
    len = min(len, (int64_t)0x7ffffff0);
}

__global__ void __launch_bounds__(256) k_inflate_scan(const InflatePlane* __restrict__ planes, InflateArgs a) {
    const int s = blockIdx.y;
    const InflatePlane P = planes[s];
    int64_t off, len;
    stream_range(P, a.in_bytes, off, len);
    if (blockIdx.x == 0 && threadIdx.x == 0) {
        IfStream& R = a.streams[s];
        R.off = off; R.len = len; R.limit = stream_limit(P); R.expected = 4 * (int64_t)max(*P.n_coef, 0);
        IfSeg& S = a.segs[s];
        S.stream = s; S.pos = 2; S.head = 0;
    }
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    for (int64_t p = off + 4 + (int64_t)blockIdx.x * blockDim.x + threadIdx.x; p <= off + len; p += stride) {
        const uint8_t* q = a.in + p - 4;
        if (q[0] != 0 || q[1] != 0 || q[2] != 0xff || q[3] != 0xff) continue;
        const int k = atomicAdd(&a.counters[0], 1);
        int idx = -1;
        if (k < a.cap_segs - a.nplanes) {
            idx = a.nplanes + k;
            IfSeg& S = a.segs[idx];
            S.stream = s; S.pos = (int32_t)(p - off); S.head = 0;
        }
        a.map[p >> 2] = idx;
    }
}

__device__ __forceinline__ int n_candidates(const InflateArgs& a) {
    return a.nplanes + min(*(volatile int*)&a.counters[0], a.cap_segs - a.nplanes);
}

// the next candidate for this warp (counters[k]), the same value in every lane
__device__ __forceinline__ int next_candidate(const InflateArgs& a, int k) {
    int i = 0;
    if ((threadIdx.x & 31) == 0) i = atomicAdd(&a.counters[k], 1);
    return __shfl_sync(0xffffffffu, i, 0);
}

struct WarpCount : IfCount {
    __device__ void sync() { __syncwarp(); }
    __device__ bool leader() const { return (threadIdx.x & 31) == 0; }
    __device__ int bcast(int v) const { return __shfl_sync(0xffffffffu, v, 0); }
};

__global__ void __launch_bounds__(32 * IF_WARPS, 4) k_inflate_spec(InflateArgs a) {
    __shared__ IfTables tabs[IF_WARPS];
    IfTables* T = &tabs[threadIdx.x >> 5];
    const int n = n_candidates(a);
    for (int i = next_candidate(a, 1); i < n; i = next_candidate(a, 1)) {
        IfSeg& S = a.segs[i];
        const IfStream R = a.streams[S.stream];
        const int32_t pos = S.pos;
        if (i < a.nplanes && if_header(a.in + R.off, R.len) != 0) {     // k_inflate_chain reports the header
            if ((threadIdx.x & 31) == 0) S.head = 0;
            continue;
        }
        WarpCount c;
        c.pos = 0; c.limit = R.limit; c.reach = 0;
        int64_t e = -1;
        const int st = if_decode(a.in + R.off, R.len, pos, -2, T, c, &e);
        __syncwarp();
        if ((threadIdx.x & 31) == 0) { S.status = st; S.end = (int32_t)e; S.olen = c.pos; S.reach = c.reach; S.head = 0; }
    }
}

__global__ void k_inflate_chain(InflateArgs a) {
    const int s = blockIdx.x * blockDim.x + threadIdx.x;
    if (s >= a.nplanes) return;
    IfStream& R = a.streams[s];
    R.hdr = if_header(a.in + R.off, R.len);
    if (R.hdr) return;
    const int n = n_candidates(a);
    if_chain(a.segs, s, R.limit, [&](int64_t p) {
        const int64_t g = R.off + p;
        const int idx = a.map[g >> 2];
        return (idx >= a.nplanes && idx < n && a.segs[idx].stream == s && a.segs[idx].pos == p) ? idx : -1;
    });
}

// output sink of one warp: every lane decodes, lane 0 writes literals, all lanes share copies
struct WarpWrite {
    uint8_t* out;
    int64_t pos, limit;
    int lane;
    __device__ void sync() { __syncwarp(); }
    __device__ bool leader() const { return lane == 0; }
    __device__ int bcast(int v) const { return __shfl_sync(0xffffffffu, v, 0); }
    __device__ int lit(uint8_t b) {
        if (pos >= limit) return IF_LENGTH;
        if (lane == 0) out[pos] = b;
        pos++;
        return 0;
    }
    __device__ int copy(int d, int n) {
        if (d > pos) return IF_DIST_FAR;
        const int m = n > limit - pos ? (int)(limit - pos) : n;
        __syncwarp();
        uint8_t* o = out + pos;
        const uint8_t* src = o - d;
        if (d >= m) { for (int k = lane; k < m; k += 32) o[k] = src[k]; }
        else { for (int k = lane; k < m; k += 32) o[k] = src[k % d]; }
        pos += m;
        return m < n ? IF_LENGTH : 0;
    }
    __device__ int raw(const uint8_t* s, int n) {
        const int m = n > limit - pos ? (int)(limit - pos) : n;
        for (int k = lane; k < m; k += 32) out[pos + k] = s[k];
        pos += m;
        return m < n ? IF_LENGTH : 0;
    }
};

__global__ void __launch_bounds__(32 * IF_WARPS, 4) k_inflate_output(const InflatePlane* __restrict__ planes, InflateArgs a) {
    __shared__ IfTables tabs[IF_WARPS];
    IfTables* T = &tabs[threadIdx.x >> 5];
    const int lane = threadIdx.x & 31;
    const int n = n_candidates(a);
    for (int i = next_candidate(a, 2); i < n; i = next_candidate(a, 2)) {
        IfSeg& S = a.segs[i];
        if (!S.head) continue;
        const IfStream R = a.streams[S.stream];
        const int64_t out_off = S.out_off;
        WarpWrite w{planes[S.stream].out + out_off, 0, R.limit - out_off, lane};
        int64_t e = -1;
        const int st = if_decode(a.in + R.off, R.len, S.pos, S.hend, T, w, &e);
        __syncwarp();
        unsigned long long s1 = 0, s2 = 0;
        for (int64_t k = lane; k < w.pos; k += 32) {
            const uint32_t v = w.out[k];
            s1 += v;
            s2 += (unsigned long long)((uint32_t)(w.pos - k) % DF_ADLER_MOD) * v;
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) { s1 += __shfl_xor_sync(0xffffffffu, s1, o); s2 += __shfl_xor_sync(0xffffffffu, s2, o); }
        if (lane == 0) { S.hstatus = st; S.fend = (int32_t)e; S.hlen = w.pos; S.hadler = df_adler_from_sums(s1, s2, w.pos); }
    }
}

__global__ void k_inflate_finish(const InflatePlane* __restrict__ planes, InflateArgs a) {
    const int s = blockIdx.x * blockDim.x + threadIdx.x;
    if (s >= a.nplanes) return;
    const InflatePlane P = planes[s];
    const IfStream R = a.streams[s];
    int64_t bytes = 0;
    int nseg = 0;
    int st = R.hdr;
    if (!st) st = if_finish(a.in + R.off, R.len, R.expected, a.segs, s, &bytes, &nseg);
    *P.status = st;
    *P.out_bytes = bytes;
    *P.segments = nseg;
}

}  // namespace

int launch_inflate(const InflatePlane* planes_dev, const InflateArgs& a, int sm_count, cudaStream_t st) {
    AEAJ_CUDA(cudaMemsetAsync(a.counters, 0, 4 * sizeof(int), st));
    const int64_t tiles = (a.in_bytes + 256 * 16 - 1) / (256 * 16);
    k_inflate_scan<<<dim3((unsigned)std::max<int64_t>(1, std::min<int64_t>(tiles, 1024)), a.nplanes), 256, 0, st>>>(planes_dev, a);
    AEAJ_LAUNCH_CHECK();
    const int ctas = sm_count * 8;
    k_inflate_spec<<<ctas, 32 * IF_WARPS, 0, st>>>(a);
    AEAJ_LAUNCH_CHECK();
    k_inflate_chain<<<(a.nplanes + 63) / 64, 64, 0, st>>>(a);
    AEAJ_LAUNCH_CHECK();
    k_inflate_output<<<ctas, 32 * IF_WARPS, 0, st>>>(planes_dev, a);
    AEAJ_LAUNCH_CHECK();
    k_inflate_finish<<<(a.nplanes + 63) / 64, 64, 0, st>>>(planes_dev, a);
    AEAJ_LAUNCH_CHECK();
    return 0;
}
