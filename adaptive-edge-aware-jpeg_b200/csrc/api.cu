// api.cu -- the C ABI of libaeaj.so (include/aeaj.h): handles, plans, workspace carving, stage entry
// points and the fused encode / decode pipelines.  No kernels here.
#include <stdarg.h>
#include <stdlib.h>
#include <string.h>
#include <string>
#include <vector>
#include "aeaj_internal.cuh"
#include "deflate_core.h"
#include "inflate_core.h"

// ---------------------------------------------------------------------------------------------
// errors
// ---------------------------------------------------------------------------------------------
static thread_local char g_err[512] = "";
void aeaj_set_error(const char* fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof g_err, fmt, ap);
    va_end(ap);
}
extern "C" const char* aeaj_last_error(void) { return g_err; }
extern "C" int aeaj_version(void) { return AEAJ_VERSION; }

// ---------------------------------------------------------------------------------------------
// bump allocator over a caller-provided workspace
// ---------------------------------------------------------------------------------------------
struct Bump {
    uint8_t* base; size_t off;
    explicit Bump(void* p) : base((uint8_t*)p), off(0) {}
    template <typename T> T* take(size_t n) {
        off = (off + 255) & ~(size_t)255;
        T* r = base ? (T*)(base + off) : (T*)nullptr;
        off += n * sizeof(T);
        return r;
    }
    size_t used() const { return (off + 255) & ~(size_t)255; }
};

// device copy of a host descriptor array (one per kernel family of a plan).  push() uploads only when the bytes or the
// stream differ from the last push: steady-state calls issue no host-to-device copy at all, which also makes them
// capturable in a CUDA graph.  The stream is part of the check because the last upload is ordered on its own stream only.
template <typename T> struct DescTable {
    static_assert(std::is_trivially_copyable<T>::value, "descriptors are compared and uploaded as bytes");
    T* dev = nullptr;
    size_t cap = 0;
    std::vector<T> pushed;                 // what `dev` holds
    cudaStream_t stream = nullptr;         // the stream of that upload
    DescTable() = default;
    DescTable(const DescTable&) = delete;
    DescTable& operator=(const DescTable&) = delete;
    ~DescTable() { cudaFree(dev); }
    // `out` receives the device array that holds `host` once `st` reaches this point
    int push(const std::vector<T>& host, cudaStream_t st, T*& out) {
        if (host.size() > cap) {
            cudaFree(dev); dev = nullptr; cap = 0; pushed.clear();
            AEAJ_CUDA(cudaMalloc(&dev, sizeof(T) * host.size()));
            cap = host.size();
        }
        out = dev;
        if (stream == st && pushed.size() == host.size() && memcmp(pushed.data(), host.data(), sizeof(T) * host.size()) == 0) return 0;
        pushed.clear();                    // a failed upload leaves nothing that could be mistaken for the device contents
        AEAJ_CUDA(cudaMemcpyAsync(dev, host.data(), sizeof(T) * host.size(), cudaMemcpyHostToDevice, st));
        pushed = host; stream = st;
        return 0;
    }
    void forget() { pushed.clear(); }      // the next push uploads
};

static int64_t cap_leaves_of(int h, int w, int mn) { return (int64_t)aeaj_cdiv(h, mn) * aeaj_cdiv(w, mn); }
static int64_t cap_states_of(int h, int w, int mn, int root) {
    int64_t n = 1;
    for (int64_t s = 2 * (int64_t)mn; s <= root; s *= 2) n += 4 * aeaj_cdiv64(h, s) * aeaj_cdiv64(w, s);
    return n + 8;
}
static int64_t cap_coef_of(int h, int w, int top) { return (int64_t)aeaj_cdiv(h, top) * top * (int64_t)aeaj_cdiv(w, top) * top; }

static void plane_geom(PlaneDesc& P, int h, int w, int mn, int mx) {
    P.h = h; P.w = w; P.wpr = aeaj_cdiv(w, 32);
    P.ry0 = 0; P.ry1 = h;
    P.root = aeaj_root_size(h, w);
    if (mx > 0) {
        P.top = std::min(mx, P.root);
        P.ntx = aeaj_cdiv(w, P.top); P.nty = aeaj_cdiv(h, P.top);
        P.cap_leaves = cap_leaves_of(h, w, mn);
        P.cap_states = cap_states_of(h, w, mn, P.root);
        P.cap_coef = cap_coef_of(h, w, P.top);
    } else { P.top = 0; P.ntx = P.nty = 0; P.cap_leaves = P.cap_states = P.cap_coef = 0; }
}

// scratch that belongs to one plane (carved per plane; pointers may be null when b.base is null)
static void carve_plane_scratch(Bump& b, PlaneDesc& P, bool canny, bool qt) {
    if (canny) {
        P.strong = b.take<uint32_t>((size_t)P.h * P.wpr);
        P.weak = b.take<uint32_t>((size_t)P.h * P.wpr);
        P.clahe_hist = b.take<uint32_t>(16 * 256);
        P.clahe_lut = b.take<uint8_t>(16 * 256);
        P.hist = b.take<uint32_t>(256);
        P.thr = b.take<int>(2);
        P.thr_d = b.take<double>(2);
    }
    if (qt) {
        size_t ntb = (size_t)P.ntx * P.nty;
        P.tb_tot = b.take<int2>(ntb);
        P.tb_coef = b.take<int>(ntb);
        P.tb_base = b.take<int4>(ntb);
    }
}

struct ClassGeom {
    int64_t off[9], cap[9], total;
    // the class-offset table the quadtree / bucketing kernels read: offsets, then capacities
    void table(long long (&t)[18]) const { for (int k = 0; k < 9; k++) { t[k] = off[k]; t[9 + k] = cap[k]; } }
};
static void class_geom(const PlaneDesc* P, int nplanes, int lg_min, int lg_max, ClassGeom& g) {
    g.total = 0;
    for (int k = 0; k < 9; k++) { g.off[k] = 0; g.cap[k] = 0; }
    for (int k = lg_min; k <= lg_max; k++) {
        int s = 1 << k;
        int64_t c = 0;
        for (int i = 0; i < nplanes; i++) c += (int64_t)aeaj_cdiv(P[i].h, s) * aeaj_cdiv(P[i].w, s);
        g.off[k] = g.total; g.cap[k] = c; g.total += c;
    }
}

// ---------------------------------------------------------------------------------------------
// handle
// ---------------------------------------------------------------------------------------------
extern "C" int aeaj_create(int device, aeaj_handle** out) {
    if (!out) { aeaj_set_error("aeaj_create: out is NULL"); return AEAJ_EINVAL; }
    int ndev = 0;
    cudaError_t e = cudaGetDeviceCount(&ndev);
    if (e != cudaSuccess || ndev == 0) {
        aeaj_set_error("no CUDA device available (%s); libaeaj has no CPU fallback", cudaGetErrorString(e));
        return AEAJ_ENOCUDA;
    }
    AEAJ_REQUIRE(device >= 0 && device < ndev, "aeaj_create: bad device index");
    AEAJ_CUDA(cudaSetDevice(device));
    cudaDeviceProp prop;
    AEAJ_CUDA(cudaGetDeviceProperties(&prop, device));
    if (prop.major < 10) {
        aeaj_set_error("device %d is sm_%d%d; libaeaj is built for sm_100a only", device, prop.major, prop.minor);
        return AEAJ_ENOCUDA;
    }
    aeaj_handle* h = (aeaj_handle*)calloc(1, sizeof(aeaj_handle));
    if (!h) return AEAJ_ENOMEM;
    h->device = device;
    h->sm_count = prop.multiProcessorCount;
    int rc = aeaj_dct_init(h);
    if (rc) { free(h); return rc; }
    rc = aeaj_canny_init(h);
    if (rc) { free(h); return rc; }
    rc = aeaj_dct_tc_init(h);
    if (rc) { free(h); return rc; }
    rc = aeaj_color_init(h);
    if (rc) { free(h); return rc; }
    rc = aeaj_deflate_init();
    if (rc) { free(h); return rc; }
    rc = aeaj_idct_scaled_init();
    if (rc) { free(h); return rc; }
    AEAJ_CUDA(cudaMalloc(&h->srgb_lut_dev, 256 * sizeof(float)));
    *out = h;
    return 0;
}

extern "C" int aeaj_destroy(aeaj_handle* h) {
    if (!h) return 0;
    cudaSetDevice(h->device);
    cudaFree(h->pq_tabs_dev); cudaFree(h->srgb_lut_dev); cudaFree(h->dct_all_dev); cudaFree(h->dct_half_all_dev); cudaFree(h->zz_all_dev); cudaFree(h->izz_all_dev); cudaFree(h->dct_tc_tiles_dev); cudaFree(h->tc_izz_all_dev); cudaFree(h->tc_err_dev);
    free(h);
    return 0;
}

extern "C" int aeaj_set_color_tables(aeaj_handle* h, int space, const float* f1, const float* f2, const float* i1,
                                     const float* i2, const float* mid, const float* scale) {
    AEAJ_REQUIRE(h && space >= 0 && space < 8, "aeaj_set_color_tables: bad arguments");
    ColorConsts& C = h->colors_host[space];
    if (f1) memcpy(C.fwd1, f1, sizeof C.fwd1);
    if (f2) memcpy(C.fwd2, f2, sizeof C.fwd2);
    if (i1) memcpy(C.inv1, i1, sizeof C.inv1);
    if (i2) memcpy(C.inv2, i2, sizeof C.inv2);
    if (mid) memcpy(C.mid, mid, sizeof C.mid);
    if (scale) memcpy(C.scale, scale, sizeof C.scale);
    return 0;
}

// 1 (default): the PQ / sRGB / OKLAB transfer functions try the table-driven evaluation first and fall back to the exact float64
// path for the pixels whose float32 rounding it cannot guarantee; 0: exact path for every pixel.  Same results either way.
extern "C" int aeaj_set_fast_transfer(aeaj_handle* h, int on) {
    AEAJ_REQUIRE(h, "aeaj_set_fast_transfer: NULL handle");
    for (int sp = 0; sp < 8; sp++)
        h->colors_host[sp].fast = (on && (sp == AEAJ_OKLAB || sp == AEAJ_ICACB || sp == AEAJ_ICTCP || sp == AEAJ_JZAZBZ)) ? 1 : 0;
    return 0;
}

extern "C" int aeaj_set_srgb_lut(aeaj_handle* h, const float* lut) {
    AEAJ_REQUIRE(h, "aeaj_set_srgb_lut: NULL handle");
    if (!lut) { h->has_srgb_lut = 0; return 0; }
    AEAJ_CUDA(cudaSetDevice(h->device));
    AEAJ_CUDA(cudaMemcpy(h->srgb_lut_dev, lut, 256 * sizeof(float), cudaMemcpyHostToDevice));
    h->has_srgb_lut = 1;
    return 0;
}

// ---------------------------------------------------------------------------------------------
// simple stage entry points
// ---------------------------------------------------------------------------------------------
#define ST(stream) ((cudaStream_t)(stream))

extern "C" int aeaj_color_forward(aeaj_handle* h, int space, const float* rgb, float* out, size_t n, void* stream) {
    if (h && n == 0) return 0;
    AEAJ_REQUIRE(h && rgb && out && space >= 0 && space < 8, "aeaj_color_forward: bad arguments");
    return launch_color_pixels(h, space, 0, rgb, out, n, ST(stream));
}
extern "C" int aeaj_color_inverse(aeaj_handle* h, int space, const float* in, float* rgb, size_t n, void* stream) {
    if (h && n == 0) return 0;
    AEAJ_REQUIRE(h && rgb && in && space >= 0 && space < 8, "aeaj_color_inverse: bad arguments");
    return launch_color_pixels(h, space, 1, in, rgb, n, ST(stream));
}
extern "C" int aeaj_normalize(aeaj_handle* h, int space, int channel, int inverse, const float* in, float* out, size_t n, void* stream) {
    if (h && n == 0) return 0;
    AEAJ_REQUIRE(h && in && out && space >= 0 && space < 8 && channel >= 0 && channel < 3, "aeaj_normalize: bad arguments");
    return launch_normalize(in, out, n, h->colors_host[space].mid[channel], h->colors_host[space].scale[channel], inverse, ST(stream));
}
extern "C" int aeaj_downsample_area(aeaj_handle* h, const float* src, int H, int W, float* dst, int dh, int dw, void* stream) {
    AEAJ_REQUIRE(h && src && dst && H > 0 && W > 0 && dh > 0 && dw > 0 && dh <= H && dw <= W, "aeaj_downsample_area: bad arguments");
    if (dh == H && dw == W) { AEAJ_CUDA(cudaMemcpyAsync(dst, src, sizeof(float) * (size_t)H * W, cudaMemcpyDeviceToDevice, ST(stream))); return 0; }
    return launch_area(src, H, W, dst, dh, dw, nullptr, 1, 0, 0, ST(stream));
}
extern "C" int aeaj_resize_linear(aeaj_handle* h, const float* src, int sh, int sw, float* dst, int H, int W, void* stream) {
    AEAJ_REQUIRE(h && src && dst && H > 0 && W > 0 && sh > 0 && sw > 0, "aeaj_resize_linear: bad arguments");
    return launch_resize_linear(src, sh, sw, dst, H, W, ST(stream));
}
extern "C" int aeaj_cast_u8(aeaj_handle* h, const float* layer, uint8_t* out, size_t n, void* stream) {
    if (h && n == 0) return 0;
    AEAJ_REQUIRE(h && layer && out, "aeaj_cast_u8: bad arguments");
    return launch_cast_u8(layer, out, n, ST(stream));
}

// ---- single-plane stage workspace -------------------------------------------------------------
// The call's descriptor and class-offset table live in the workspace too, so that calls on separate workspaces are independent.
struct StageWs {
    PlaneDesc P;
    PlaneDesc* desc;                      // device copy of P
    long long* class_off;                 // device ClassGeom::table (quadtree / DCT calls)
    uint8_t* u8a; uint8_t* u8b;
    int* flags; int* ring; int* ctrl; int* status;
    ClassEntry* class_lists; int* class_counts;
    float* scratch256;
    ClassGeom cg;
    int ntiles, ring_cap;
    size_t bytes;
};
static void stage_ws(void* ws, int h, int w, int mn, int mx, StageWs& S) {
    memset(&S, 0, sizeof S);
    Bump b(ws);
    plane_geom(S.P, h, w, mn, mx);
    carve_plane_scratch(b, S.P, true, mx > 0);
    S.u8a = b.take<uint8_t>((size_t)h * w);
    S.u8b = b.take<uint8_t>((size_t)h * w);
    S.ntiles = hysteresis_tiles(&S.P, 1, &S.ring_cap);
    S.flags = b.take<int>((size_t)S.ntiles);
    S.ring = b.take<int>((size_t)S.ring_cap);
    S.ctrl = b.take<int>(hysteresis_ctrl_ints());
    S.status = b.take<int>(4);
    S.class_counts = b.take<int>(16);
    S.desc = b.take<PlaneDesc>(1);
    if (mx > 0) {
        class_geom(&S.P, 1, ilog2i(mn), ilog2i(mx), S.cg);
        S.class_lists = b.take<ClassEntry>((size_t)S.cg.total);
        S.class_off = b.take<long long>(18);
        if (mx >= 256) S.scratch256 = b.take<float>(aeaj_dct256_scratch_floats());
    }
    S.bytes = b.used();
}
extern "C" size_t aeaj_stage_workspace_bytes(int h, int w, int min_size, int max_size) {
    if (h <= 0 || w <= 0) return 0;
    StageWs S;
    stage_ws(nullptr, h, w, min_size, max_size, S);
    return S.bytes + 256;
}
// once per call, after S.P is complete
static int push_stage(const StageWs& S, cudaStream_t st) {
    AEAJ_CUDA(cudaMemcpyAsync(S.desc, &S.P, sizeof(PlaneDesc), cudaMemcpyHostToDevice, st));
    if (S.class_off) {
        long long t[18]; S.cg.table(t);
        AEAJ_CUDA(cudaMemcpyAsync(S.class_off, t, sizeof t, cudaMemcpyHostToDevice, st));
    }
    return 0;
}

static int run_clahe(StageWs& S, cudaStream_t st) {
    AEAJ_CUDA(cudaMemsetAsync(S.P.clahe_hist, 0, 16 * 256 * sizeof(uint32_t), st));
    int rc = launch_clahe_hist(S.desc, &S.P, 1, st); if (rc) return rc;
    return launch_clahe_lut(S.desc, 1, PeerSet{1, 0, {0}}, st);
}

extern "C" int aeaj_clahe(aeaj_handle* hd, const uint8_t* src, int h, int w, uint8_t* dst, void* ws, void* stream) {
    AEAJ_REQUIRE(hd && src && dst && ws && h > 0 && w > 0, "aeaj_clahe: bad arguments");
    StageWs S; stage_ws(ws, h, w, 0, 0, S);
    S.P.u8a = (uint8_t*)src; S.P.u8b = dst;
    int rc = push_stage(S, ST(stream)); if (rc) return rc;
    rc = run_clahe(S, ST(stream)); if (rc) return rc;
    return launch_prefilter(S.desc, &S.P, 1, 1, 0, ST(stream));
}
static int prefilter_only(const uint8_t* src, int h, int w, uint8_t* dst, void* ws, void* stream, int stages) {
    StageWs S; stage_ws(ws, h, w, 0, 0, S);
    S.P.u8a = (uint8_t*)src; S.P.u8b = dst;
    int rc = push_stage(S, ST(stream)); if (rc) return rc;
    return launch_prefilter(S.desc, &S.P, 1, stages, 0, ST(stream));
}
extern "C" int aeaj_gauss3(aeaj_handle* hd, const uint8_t* src, int h, int w, uint8_t* dst, void* ws, void* stream) {
    AEAJ_REQUIRE(hd && src && dst && ws && h > 0 && w > 0, "aeaj_gauss3: bad arguments");
    return prefilter_only(src, h, w, dst, ws, stream, 2);
}
extern "C" int aeaj_bilateral5(aeaj_handle* hd, const uint8_t* src, int h, int w, uint8_t* dst, void* ws, void* stream) {
    AEAJ_REQUIRE(hd && src && dst && ws && h > 0 && w > 0, "aeaj_bilateral5: bad arguments");
    return prefilter_only(src, h, w, dst, ws, stream, 4);
}
extern "C" int aeaj_percentile_thresholds(aeaj_handle* hd, const uint8_t* src, int h, int w, double* thr, void* ws, void* stream) {
    AEAJ_REQUIRE(hd && src && thr && ws && h > 0 && w > 0, "aeaj_percentile_thresholds: bad arguments");
    StageWs S; stage_ws(ws, h, w, 0, 0, S);
    S.P.thr_d = thr;
    cudaStream_t st = ST(stream);
    AEAJ_CUDA(cudaMemsetAsync(S.P.hist, 0, 256 * sizeof(uint32_t), st));
    int rc = push_stage(S, st); if (rc) return rc;
    rc = launch_hist_u8(src, (size_t)h * w, S.P.hist, st); if (rc) return rc;
    return launch_thresholds(S.desc, 1, PeerSet{1, 0, {0}}, st);
}

// the descriptor's tap_edge receives the edge map
static int run_nms_hysteresis(aeaj_handle* hd, StageWs& S, cudaStream_t st) {
    int rc = launch_canny_nms(S.desc, &S.P, 1, st); if (rc) return rc;
    rc = launch_hysteresis(hd, S.desc, &S.P, 1, S.ntiles, S.ring_cap, S.flags, S.ring, S.ctrl, S.status, st);
    if (rc) return rc;
    return launch_bitmap_to_u8(S.desc, &S.P, 1, st);
}
extern "C" int aeaj_canny_u8(aeaj_handle* hd, const uint8_t* src, int h, int w, const double* thr, uint8_t* edge, void* ws, void* stream) {
    AEAJ_REQUIRE(hd && src && thr && edge && ws && h > 0 && w > 0, "aeaj_canny_u8: bad arguments");
    StageWs S; stage_ws(ws, h, w, 0, 0, S);
    S.P.u8b = (uint8_t*)src; S.P.tap_edge = edge;
    cudaStream_t st = ST(stream);
    int rc = push_stage(S, st); if (rc) return rc;
    rc = launch_thresholds_from_double(thr, S.P.thr, st); if (rc) return rc;
    return run_nms_hysteresis(hd, S, st);
}
extern "C" int aeaj_canny(aeaj_handle* hd, const float* layer, int h, int w, uint8_t* edge, void* ws, void* stream) {
    AEAJ_REQUIRE(hd && layer && edge && ws && h > 0 && w > 0, "aeaj_canny: bad arguments");
    StageWs S; stage_ws(ws, h, w, 0, 0, S);
    S.P.u8a = S.u8a; S.P.u8b = S.u8b; S.P.tap_edge = edge;
    cudaStream_t st = ST(stream);
    int rc = push_stage(S, st); if (rc) return rc;
    rc = launch_cast_u8(layer, S.u8a, (size_t)h * w, st); if (rc) return rc;
    rc = run_clahe(S, st); if (rc) return rc;
    AEAJ_CUDA(cudaMemsetAsync(S.P.hist, 0, 256 * sizeof(uint32_t), st));
    rc = launch_prefilter(S.desc, &S.P, 1, 7, 1, st); if (rc) return rc;
    rc = launch_thresholds(S.desc, 1, PeerSet{1, 0, {0}}, st); if (rc) return rc;
    return run_nms_hysteresis(hd, S, st);
}

extern "C" int aeaj_quadtree_caps(int h, int w, int mn, int mx, int64_t* cl, int64_t* cs, int64_t* cc, int* root) {
    if (h <= 0 || w <= 0 || mn < 2 || mx < mn || (mn & (mn - 1)) || (mx & (mx - 1))) { aeaj_set_error("aeaj_quadtree_caps: bad arguments"); return AEAJ_EINVAL; }
    PlaneDesc P; plane_geom(P, h, w, mn, mx);
    if (cl) *cl = P.cap_leaves; if (cs) *cs = P.cap_states; if (cc) *cc = P.cap_coef; if (root) *root = P.root;
    return 0;
}
static int check_blocks(int h, int w, int mn, int mx) {
    AEAJ_REQUIRE(mn >= 2 && mx >= mn && !(mn & (mn - 1)) && !(mx & (mx - 1)), "block sizes must be powers of two with 2 <= min <= max");
    AEAJ_REQUIRE(mx <= 256, "block sizes above 256 are not supported");
    AEAJ_REQUIRE(aeaj_root_size(h, w) >= mn, "image smaller than the minimum block size");
    AEAJ_REQUIRE(std::min(mx, aeaj_root_size(h, w)) / mn <= 128, "max/min block ratio above 128 is not supported");
    return 0;
}
extern "C" int aeaj_quadtree(aeaj_handle* hd, const uint8_t* edge, int h, int w, int mn, int mx, int32_t* leaves, uint8_t* states,
                             int32_t* counts, void* ws, void* stream) {
    AEAJ_REQUIRE(hd && edge && leaves && states && counts && ws && h > 0 && w > 0, "aeaj_quadtree: bad arguments");
    int rc = check_blocks(h, w, mn, mx); if (rc) return rc;
    StageWs S; stage_ws(ws, h, w, mn, mx, S);
    S.P.leaves = leaves; S.P.states = states; S.P.counts = counts;
    cudaStream_t st = ST(stream);
    rc = push_stage(S, st); if (rc) return rc;
    AEAJ_CUDA(cudaMemsetAsync(S.class_counts, 0, 16 * sizeof(int), st));
    rc = launch_u8_to_bitmap(edge, h, w, S.P.strong, st); if (rc) return rc;
    return launch_quadtree(S.desc, &S.P, 1, mn, mx, S.class_lists, S.class_counts, S.class_off, st, nullptr);
}

static int stage_blocks(aeaj_handle* hd, bool inverse, float* layer, int h, int w, float mid, float scale, const int32_t* leaves,
                        const int32_t* counts, int mn, int mx, const int32_t* const* qtab, int32_t* coef, void* ws, cudaStream_t st) {
    int rc = check_blocks(h, w, mn, mx); if (rc) return rc;
    StageWs S; stage_ws(ws, h, w, mn, mx, S);
    S.P.layer_f32 = layer; S.P.mid = mid; S.P.scale = scale;
    S.P.leaves = (int32_t*)leaves; S.P.counts = (int32_t*)counts; S.P.coef = coef;
    for (int k = 0; k < 9; k++) S.P.qtab[k] = qtab[k];
    S.P.cap_leaves = INT32_MAX;                        // the stage API trusts counts[0] (the caller sized the leaf list)
    rc = push_stage(S, st); if (rc) return rc;
    AEAJ_CUDA(cudaMemsetAsync(S.class_counts, 0, 16 * sizeof(int), st));
    rc = launch_bucket_leaves(S.desc, &S.P, 1, S.class_lists, S.class_counts, S.class_off, ilog2i(mn), ilog2i(mx), st); if (rc) return rc;
    if (inverse) return launch_dequant_idct(hd, S.desc, S.class_lists, S.class_counts, S.cg.off, S.cg.cap, ilog2i(mn), ilog2i(mx), st, nullptr, nullptr, nullptr, 0, S.scratch256);
    return launch_dct_quant(hd, S.desc, S.class_lists, S.class_counts, S.cg.off, S.cg.cap, ilog2i(mn), ilog2i(mx), st, nullptr, nullptr, nullptr, 0, S.scratch256);
}
extern "C" int aeaj_dct_quant(aeaj_handle* hd, const float* layer, int h, int w, float mid, float scale, const int32_t* leaves,
                              const int32_t* counts, int mn, int mx, const int32_t* const* qtab, int32_t* coef, void* ws, void* stream) {
    AEAJ_REQUIRE(hd && layer && leaves && counts && qtab && coef && ws && h > 0 && w > 0, "aeaj_dct_quant: bad arguments");
    return stage_blocks(hd, false, (float*)layer, h, w, mid, scale, leaves, counts, mn, mx, qtab, coef, ws, ST(stream));
}
extern "C" int aeaj_dequant_idct(aeaj_handle* hd, const int32_t* coef, const int32_t* leaves, const int32_t* counts, int mn, int mx,
                                 const int32_t* const* qtab, int h, int w, float mid, float scale, float* layer, void* ws, void* stream) {
    AEAJ_REQUIRE(hd && layer && leaves && counts && qtab && coef && ws && h > 0 && w > 0, "aeaj_dequant_idct: bad arguments");
    return stage_blocks(hd, true, layer, h, w, mid, scale, leaves, counts, mn, mx, qtab, (int32_t*)coef, ws, ST(stream));
}

// ---------------------------------------------------------------------------------------------
// plan: geometry of a batch of same-shape images + q tables
// ---------------------------------------------------------------------------------------------
struct aeaj_plan {
    aeaj_handle* h;
    aeaj_plan_info info;
    int nplanes, lg_min, lg_max;
    std::vector<PlaneDesc> planes;       // host copy, index b*3 + l
    DescTable<PlaneDesc> planes_tab;
    int ntiles, ring_cap;
    long long* class_off_dev;
    ClassGeom cg;
    int32_t* qtab_dev; size_t qtab_entries;
    float* qtabf_dev;                    // the same entries as float
    const int32_t* qtab_ptr[2][9];       // device pointers per table (0 luma, 1 chroma) and log2 size
    const float* qtabf_ptr[2][9];
    std::vector<PackPlane> pack_planes;  // host copy of the packing descriptors
    DescTable<PackPlane> pack_tab, unpack_tab;   // separate tables (they differ in n_coef): alternating calls upload nothing
    std::vector<DeflatePlane> df_planes;
    DescTable<DeflatePlane> deflate_tab;
    std::vector<InflatePlane> if_planes;
    DescTable<InflatePlane> inflate_tab;
    std::vector<PlaneDesc> scaled_planes;  // aeaj_decode_scaled: the planes with layer_f32 on the 1/m planes of the caller's scratch
    DescTable<PlaneDesc> scaled_tab[4];    // one per log2(scale): decodes alternating between scales upload nothing either
    // one image over several GPUs (peer.cu): the other ranks' workspaces / barrier flags, opened through CUDA IPC by the caller
    PeerSet peers = {1, 0, {0}};
    void* peer_ws[AEAJ_MAX_PEERS] = {nullptr};
    int* peer_flags[AEAJ_MAX_PEERS] = {nullptr};
    int peer_epoch = 0;
    PeerSeg* peer_segs_dev = nullptr;
    int last_launches;
    bool need_full_chroma;
    int zigzag = 0;
    int tensor_dct = 0xa;         // size classes on the tcgen05 kernels: bit k = class 16 << k (aeaj_plan_set_tensor_dct)
    // optional per-stage CUDA-event timing (bench.py roofline leg)
    bool timing_on = false;
    std::vector<cudaEvent_t> ev;
    std::vector<std::string> ev_name;
    int ev_n = 0;
    cudaStream_t ev_stream = 0;
    void mark(const char* name) {
        if (!timing_on) return;
        if ((int)ev.size() <= ev_n) { cudaEvent_t e; cudaEventCreate(&e); ev.push_back(e); ev_name.push_back(""); }
        cudaEventRecord(ev[ev_n], ev_stream);
        ev_name[ev_n] = name;
        ev_n++;
    }
};
static void plan_mark_cb(void* ctx, const char* name) { ((aeaj_plan*)ctx)->mark(name); }

static int sub_ratio(int space, int& rh, int& rw) {
    switch (space) {
        case AEAJ_ICACB: case AEAJ_ICTCP: rh = 1; rw = 4; return 0;
        case AEAJ_JZAZBZ: case AEAJ_OKLAB: case AEAJ_YCBCR: case AEAJ_YCOCG: case AEAJ_YCOCG_R: rh = 2; rw = 2; return 0;
    }
    aeaj_set_error("colour space %d has no compression settings (jpeg.py:62-147)", space);
    return AEAJ_EINVAL;
}

struct PlanAux { float* full_c1; float* full_c2; int* flags; int* ring; int* ctrl; int* class_counts; ClassEntry* class_lists; float* scratch256;
                 int* pack_sums[3]; };
// carve the plan workspace: the plane pointers of p->planes and the call's buffers A; with ws == nullptr only the size
static size_t plan_carve(aeaj_plan* p, void* ws, PlanAux& A) {
    Bump b(ws);
    const int B = p->info.batch;
    for (int l = 0; l < 3; l++) {
        const size_t n = (size_t)p->info.layer_h[l] * p->info.layer_w[l];
        float* lay = b.take<float>(n * B);
        uint8_t* a = b.take<uint8_t>(n * B);
        uint8_t* c = b.take<uint8_t>(n * B);
        for (int i = 0; i < B; i++) {
            PlaneDesc& P = p->planes[i * 3 + l];
            P.layer_f32 = lay ? lay + n * i : nullptr; P.u8a = a ? a + n * i : nullptr; P.u8b = c ? c + n * i : nullptr;
        }
    }
    // accumulators of all planes are contiguous so that one memset clears them
    const int NP = p->nplanes;
    uint32_t* ch = b.take<uint32_t>((size_t)NP * 16 * 256);
    uint32_t* hi = b.take<uint32_t>((size_t)NP * 256);
    uint8_t* lut = b.take<uint8_t>((size_t)NP * 16 * 256);
    int* thr = b.take<int>((size_t)NP * 2);
    double* thrd = b.take<double>((size_t)NP * 2);
    for (int i = 0; i < NP; i++) {
        PlaneDesc& P = p->planes[i];
        P.clahe_hist = ch ? ch + (size_t)i * 16 * 256 : nullptr; P.hist = hi ? hi + (size_t)i * 256 : nullptr;
        P.clahe_lut = lut ? lut + (size_t)i * 16 * 256 : nullptr; P.thr = thr ? thr + 2 * i : nullptr; P.thr_d = thrd ? thrd + 2 * i : nullptr;
        P.strong = b.take<uint32_t>((size_t)P.h * P.wpr);
        P.weak = b.take<uint32_t>((size_t)P.h * P.wpr);
        size_t ntb = (size_t)P.ntx * P.nty;
        P.tb_tot = b.take<int2>(ntb); P.tb_coef = b.take<int>(ntb); P.tb_base = b.take<int4>(ntb);
    }
    const size_t HW = (size_t)p->info.height * p->info.width;
    if (p->need_full_chroma) { A.full_c1 = b.take<float>(HW * p->info.batch); A.full_c2 = b.take<float>(HW * p->info.batch); }
    else { A.full_c1 = A.full_c2 = nullptr; }
    A.flags = b.take<int>((size_t)p->ntiles);
    A.ring = b.take<int>((size_t)p->ring_cap);
    A.ctrl = b.take<int>(hysteresis_ctrl_ints());
    A.class_counts = b.take<int>(16);
    A.class_lists = b.take<ClassEntry>((size_t)p->cg.total);
    // the 256 x 256 kernel's intermediate tiles belong to the call (plans run concurrently on several streams)
    A.scratch256 = (p->lg_max >= 8) ? b.take<float>(aeaj_dct256_scratch_floats()) : nullptr;
    for (int l = 0; l < 3; l++) A.pack_sums[l] = b.take<int>(aeaj_pack_scratch_ints(p->info.cap_coef[l]) * p->info.batch);
    return b.used();
}

extern "C" int aeaj_plan_create(aeaj_handle* h, int batch, int height, int width, int space, int bmin, int bmax, aeaj_plan** out) {
    AEAJ_REQUIRE(h && out && batch > 0 && height > 0 && width > 0, "aeaj_plan_create: bad arguments");
    int rh, rw;
    int rc = sub_ratio(space, rh, rw); if (rc) return rc;
    AEAJ_REQUIRE(height / rh > 0 && width / rw > 0, "image too small for the chroma subsampling of this colour space");
    AEAJ_CUDA(cudaSetDevice(h->device));
    aeaj_plan* p = new aeaj_plan();
    p->h = h;
    memset(&p->info, 0, sizeof p->info);
    p->info.batch = batch; p->info.height = height; p->info.width = width; p->info.space = space;
    p->info.block_min = bmin; p->info.block_max = bmax;
    p->nplanes = batch * 3;
    p->planes.resize(p->nplanes);
    for (int l = 0; l < 3; l++) {
        int lh = l ? height / rh : height, lw = l ? width / rw : width;     // jpeg.py:676-686
        rc = check_blocks(lh, lw, bmin, bmax);
        if (rc) { delete p; return rc; }
        p->info.layer_h[l] = lh; p->info.layer_w[l] = lw;
        for (int i = 0; i < batch; i++) {
            PlaneDesc& P = p->planes[i * 3 + l];
            memset(&P, 0, sizeof P);
            plane_geom(P, lh, lw, bmin, bmax);
            P.layer = l;
            P.mid = h->colors_host[space].mid[l]; P.scale = h->colors_host[space].scale[l];
        }
        const PlaneDesc& P0 = p->planes[l];
        p->info.root[l] = P0.root; p->info.cap_leaves[l] = P0.cap_leaves; p->info.cap_states[l] = P0.cap_states; p->info.cap_coef[l] = P0.cap_coef;
        AEAJ_REQUIRE(P0.cap_coef < (int64_t)1 << 31, "layer too large for int32 coefficient offsets");
    }
    p->lg_min = ilog2i(bmin); p->lg_max = ilog2i(bmax);
    const int ch = p->info.layer_h[1], cw = p->info.layer_w[1];
    p->need_full_chroma = !((ch * 2 == height && cw * 2 == width && (width % 4) == 0) || (ch == height && cw * 4 == width));
    class_geom(p->planes.data(), p->nplanes, p->lg_min, p->lg_max, p->cg);
    p->ntiles = hysteresis_tiles(p->planes.data(), p->nplanes, &p->ring_cap);
    PlanAux A;
    p->info.workspace_bytes = (int64_t)plan_carve(p, nullptr, A) + 256;
    AEAJ_CUDA(cudaMalloc(&p->class_off_dev, sizeof(long long) * 18));
    p->pack_planes.resize(p->nplanes);
    long long off[18]; p->cg.table(off);
    AEAJ_CUDA(cudaMemcpy(p->class_off_dev, off, sizeof off, cudaMemcpyHostToDevice));
    p->qtab_dev = nullptr; p->qtabf_dev = nullptr; p->qtab_entries = 0;
    memset(p->qtab_ptr, 0, sizeof p->qtab_ptr);
    memset(p->qtabf_ptr, 0, sizeof p->qtabf_ptr);
    p->last_launches = 0;
    *out = p;
    return 0;
}

extern "C" int aeaj_plan_destroy(aeaj_plan* p) {
    if (!p) return 0;
    cudaSetDevice(p->h->device);
    cudaFree(p->class_off_dev); cudaFree(p->qtab_dev); cudaFree(p->qtabf_dev); cudaFree(p->peer_segs_dev);
    delete p;                            // the descriptor tables free their device arrays
    return 0;
}
extern "C" int aeaj_plan_get_info(const aeaj_plan* p, aeaj_plan_info* info) {
    AEAJ_REQUIRE(p && info, "aeaj_plan_get_info: bad arguments");
    *info = p->info;
    return 0;
}
extern "C" int aeaj_plan_last_launches(const aeaj_plan* p) { return p ? p->last_launches : 0; }
extern "C" int aeaj_plan_set_tensor_dct(aeaj_plan* p, int enable) {
    AEAJ_REQUIRE(p, "aeaj_plan_set_tensor_dct: NULL plan");
    p->tensor_dct = enable & 0xf;
    return 0;
}
extern "C" int aeaj_tensor_dct_status(aeaj_handle* h, int* timed_out) {
    AEAJ_REQUIRE(h && timed_out, "aeaj_tensor_dct_status: bad arguments");
    AEAJ_CUDA(cudaMemcpy(timed_out, h->tc_err_dev, 32 * sizeof(int), cudaMemcpyDeviceToHost));   /* [0] flag, [1..] phase cycles of one leaf */
    return 0;
}
extern "C" int aeaj_plan_set_stream_layout(aeaj_plan* p, int zigzag) {
    AEAJ_REQUIRE(p, "aeaj_plan_set_stream_layout: NULL plan");
    p->zigzag = zigzag != 0;
    return 0;
}

extern "C" int aeaj_plan_enable_timing(aeaj_plan* p, int enable) {
    AEAJ_REQUIRE(p, "aeaj_plan_enable_timing: NULL plan");
    p->timing_on = enable != 0;
    p->ev_n = 0;
    return 0;
}
// durations (ms) of the stages of the LAST encode or decode call on this plan; synchronises its stream.
// names_buf receives '\n'-separated stage names.
extern "C" int aeaj_plan_read_timing(aeaj_plan* p, char* names_buf, size_t names_cap, float* ms, int cap, int* n) {
    AEAJ_REQUIRE(p && names_buf && ms && n, "aeaj_plan_read_timing: bad arguments");
    *n = 0;
    names_buf[0] = 0;
    if (!p->timing_on || p->ev_n < 2) return 0;
    AEAJ_CUDA(cudaEventSynchronize(p->ev[p->ev_n - 1]));
    size_t used = 0;
    for (int i = 1; i < p->ev_n && *n < cap; i++) {
        float t = 0;
        AEAJ_CUDA(cudaEventElapsedTime(&t, p->ev[i - 1], p->ev[i]));
        const std::string& nm = p->ev_name[i];
        if (used + nm.size() + 2 > names_cap) break;
        memcpy(names_buf + used, nm.c_str(), nm.size()); used += nm.size(); names_buf[used++] = '\n'; names_buf[used] = 0;
        ms[(*n)++] = t;
    }
    return 0;
}

extern "C" int aeaj_plan_set_qtables(aeaj_plan* p, const int32_t* tables, size_t n_entries, void* stream) {
    AEAJ_REQUIRE(p && tables, "aeaj_plan_set_qtables: bad arguments");
    size_t per = 0;
    for (int k = p->lg_min; k <= p->lg_max; k++) per += (size_t)1 << (2 * k);
    AEAJ_REQUIRE(n_entries == 2 * per, "aeaj_plan_set_qtables: expected [luma sizes...][chroma sizes...] entries");
    AEAJ_CUDA(cudaSetDevice(p->h->device));
    const size_t nf = n_entries + 8 * 2 * 9;                                     // float copy: every table padded to a 32-byte boundary
    if (!p->qtab_dev) {
        AEAJ_CUDA(cudaMalloc(&p->qtab_dev, sizeof(int32_t) * n_entries));
        AEAJ_CUDA(cudaMalloc(&p->qtabf_dev, sizeof(float) * nf));
    }
    p->qtab_entries = n_entries;
    // float copy for the tensor-core epilogue, per table in the layout [s/8 column groups][s rows][8]: a warp whose lanes own
    // consecutive rows reads the 8 steps of one column group with one contiguous 256-bit load per lane (entries <= 6050: exact)
    std::vector<float> asf(nf, 0.0f);
    size_t foff[2][9] = {{0}};
    {
        size_t o = 0, of = 0;
        for (int t = 0; t < 2; t++)
            for (int k = p->lg_min; k <= p->lg_max; k++) {
                const int s = 1 << k;
                of = (of + 7) & ~(size_t)7;
                foff[t][k] = of;
                for (int r = 0; r < s; r++)
                    for (int c = 0; c < s; c++) {
                        const size_t dst = (s >= 8) ? ((size_t)(c >> 3) * s + r) * 8 + (c & 7) : (size_t)r * s + c;
                        asf[of + dst] = (float)tables[o + (size_t)r * s + c];
                    }
                o += (size_t)s * s; of += (size_t)s * s;
            }
    }
    AEAJ_CUDA(cudaMemcpyAsync(p->qtab_dev, tables, sizeof(int32_t) * n_entries, cudaMemcpyHostToDevice, ST(stream)));
    AEAJ_CUDA(cudaMemcpyAsync(p->qtabf_dev, asf.data(), sizeof(float) * nf, cudaMemcpyHostToDevice, ST(stream)));
    AEAJ_CUDA(cudaStreamSynchronize(ST(stream)));                                // `asf` is a temporary
    size_t o = 0;
    for (int t = 0; t < 2; t++)
        for (int k = p->lg_min; k <= p->lg_max; k++) { p->qtab_ptr[t][k] = p->qtab_dev + o; p->qtabf_ptr[t][k] = p->qtabf_dev + foff[t][k]; o += (size_t)1 << (2 * k); }
    for (int i = 0; i < p->nplanes; i++)
        for (int k = 0; k < 9; k++) {
            p->planes[i].qtab[k] = p->qtab_ptr[p->planes[i].layer ? 1 : 0][k];
            p->planes[i].qtabf[k] = p->qtabf_ptr[p->planes[i].layer ? 1 : 0][k];
        }
    return 0;
}

static int plan_push_planes(aeaj_plan* p, cudaStream_t st, PlaneDesc*& planes_dev) {
    for (auto& P : p->planes) {
        P.zigzag = p->zigzag;
        for (int k = 0; k < 9; k++) P.zz[k] = p->h->zz_dev[k];
    }
    return p->planes_tab.push(p->planes, st, planes_dev);
}

// full-res luma rows [band0, band1) -> rows of every layer (chroma rows scale with the subsampling ratio)
static int set_band(aeaj_plan* p, int band0, int band1) {
    const int H = p->info.height;
    if (band1 < 0) band1 = H;
    AEAJ_REQUIRE(band0 >= 0 && band0 < band1 && band1 <= H, "bad band");
    const bool full = (band0 == 0 && band1 == H);
    for (int i = 0; i < p->nplanes; i++) {
        PlaneDesc& P = p->planes[i];
        const int rh = H / P.h;                                    // 1 or 2 (jpeg.py:62-147)
        if (!full) {
            AEAJ_REQUIRE(p->info.batch == 1, "halo-split bands need batch 1");
            const int align = rh * std::max(128, p->info.block_max);  // no leaf, filter tile or chroma cell may straddle a band
            AEAJ_REQUIRE(H % P.h == 0 && band0 % align == 0 && (band1 % align == 0 || band1 == H),
                         "band boundaries must be multiples of max(128, block_max) rows in every layer");
        }
        P.ry0 = band0 / rh; P.ry1 = (band1 == H) ? P.h : band1 / rh;
        // rows above / below the band: the neighbour rank's workspace if this plan is one rank of a multi-GPU halo-split
        P.peer_up = P.peer_dn = 0;
        if (p->peers.world > 1 && !full) {
            if (band0 > 0 && p->peers.rank > 0) P.peer_up = p->peers.delta[p->peers.rank - 1];
            if (band1 < H && p->peers.rank + 1 < p->peers.world) P.peer_dn = p->peers.delta[p->peers.rank + 1];
        }
    }
    return 0;
}

// The phases of an encode / decode, in the order one call runs them.  `phases` of encode_impl / decode_impl is a bit set of them;
// [band0, band1) restricts every phase but hysteresis to a band of full-resolution rows (the halo-split schedule below).
enum { AEAJ_PHASE_COLOR = 0,      /* clears accumulators; colour + subsample + u8 cast of the band                             */
       AEAJ_PHASE_CLAHE_HIST = 1, /* CLAHE tile histograms of the band                                                         */
       AEAJ_PHASE_PREFILTER = 2,  /* LUTs (sum of every band's partial histograms) + CLAHE / Gauss / bilateral of the band      */
       AEAJ_PHASE_NMS = 3,        /* thresholds (sum of every band's partial histograms) + Sobel / NMS of the band              */
       AEAJ_PHASE_HYST = 4,       /* hysteresis, whole image (needs every band's strong / weak rows)                           */
       AEAJ_PHASE_QT_COUNT = 5,   /* quadtree: node counts of the band's top blocks                                            */
       AEAJ_PHASE_QT_EMIT = 6,    /* needs every band's counts; scan + states / leaves / work lists of the band                */
       AEAJ_PHASE_DCT = 7 };      /* DCT + quantise of the band's leaves (coefficients at global offsets)                      */
enum { AEAJ_DPHASE_IDCT = 0,      /* dequantise + IDCT + merge of the band's leaves                                            */
       AEAJ_DPHASE_COLOR = 1 };   /* needs the neighbouring chroma rows; upsample + inverse colour of the band                  */

static int encode_impl(aeaj_plan* p, const aeaj_encode_io* io, void* workspace, cudaStream_t st, unsigned phases, int band0, int band1) {
    AEAJ_REQUIRE(p && io && workspace && (io->rgb || io->rgb_u8) && io->counts, "aeaj_encode: bad arguments (rgb or rgb_u8 required)");
    AEAJ_REQUIRE(p->qtab_dev, "aeaj_encode: quantisation tables not set (aeaj_plan_set_qtables)");
    aeaj_handle* h = p->h;
    const int B = p->info.batch, NP = p->nplanes;
    int launches = 0;
    PlanAux A;
    plan_carve(p, workspace, A);
    bool any_tap_edge = false;
    for (int l = 0; l < 3; l++) {
        AEAJ_REQUIRE(io->coef[l] && io->leaves[l] && io->states[l], "aeaj_encode: NULL output buffer");
        for (int i = 0; i < B; i++) {
            PlaneDesc& P = p->planes[i * 3 + l];
            P.coef = io->coef[l] + (size_t)i * p->info.cap_coef[l];
            P.leaves = io->leaves[l] + (size_t)i * p->info.cap_leaves[l] * 4;
            P.states = io->states[l] + (size_t)i * p->info.cap_states[l];
            P.counts = io->counts + ((size_t)i * 3 + l) * 4;
            P.packed_states = io->packed_states[l] ? io->packed_states[l] + (size_t)i * ((p->info.cap_states[l] + 3) / 4) : nullptr;
            P.tap_edge = io->tap_edges[l] ? io->tap_edges[l] + (size_t)i * P.h * P.w : nullptr;
        }
        any_tap_edge |= io->tap_edges[l] != nullptr;
    }
    int rc = set_band(p, band0, band1); if (rc) return rc;
    PlaneDesc* Pd;
    rc = plan_push_planes(p, st, Pd); if (rc) return rc;
    p->ev_n = 0; p->ev_stream = st; p->mark("start");
    // a whole-image call on a plan that is one rank of a halo-split is a plain single-GPU call: no partial histograms to sum
    const bool whole = band0 == 0 && (band1 < 0 || band1 == p->info.height);
    const PeerSet solo = {1, 0, {0}};
    const PeerSet& peers = whole ? solo : p->peers;
    if (phases & (1u << AEAJ_PHASE_COLOR)) {
        AEAJ_CUDA(cudaMemsetAsync(p->planes[0].clahe_hist, 0, (size_t)NP * 16 * 256 * sizeof(uint32_t), st));
        AEAJ_CUDA(cudaMemsetAsync(p->planes[0].hist, 0, (size_t)NP * 256 * sizeof(uint32_t), st));
        AEAJ_CUDA(cudaMemsetAsync(A.class_counts, 0, 16 * sizeof(int), st));
        if (peers.world > 1)                               // sharded quadtree: this rank fills only its band's leaf slots; the others read as absent
            for (int l = 0; l < 3; l++) AEAJ_CUDA(cudaMemsetAsync(io->leaves[l], 0, sizeof(int32_t) * 4 * (size_t)p->info.cap_leaves[l], st));
        // colour + chroma subsampling + u8 cast
        rc = launch_color_forward_planar(h, p->info.space, io->rgb, io->rgb ? nullptr : io->rgb_u8, B, p->info.height, p->info.width, Pd, p->planes.data(),
                                         A.full_c1, A.full_c2, st, &launches, band0, band1);
        if (rc) return rc;
        p->mark("color_forward_planar");
    }
    // Canny pipeline on all planes of the batch at once
    if (phases & (1u << AEAJ_PHASE_CLAHE_HIST)) {
        rc = launch_clahe_hist(Pd, p->planes.data(), NP, st); if (rc) return rc;
        launches++;
        p->mark("clahe_hist");
    }
    if (phases & (1u << AEAJ_PHASE_PREFILTER)) {
        rc = launch_clahe_lut(Pd, NP, peers, st); if (rc) return rc;
        p->mark("clahe_lut");
        rc = launch_prefilter(Pd, p->planes.data(), NP, 7, 1, st); if (rc) return rc;
        p->mark("prefilter");
        launches += 2;
    }
    if (phases & (1u << AEAJ_PHASE_NMS)) {
        rc = launch_thresholds(Pd, NP, peers, st); if (rc) return rc;
        p->mark("thresholds");
        rc = launch_canny_nms(Pd, p->planes.data(), NP, st); if (rc) return rc;
        p->mark("canny_nms");
        launches += 2;
    }
    if (phases & (1u << AEAJ_PHASE_HYST)) {
        rc = launch_hysteresis(h, Pd, p->planes.data(), NP, p->ntiles, p->ring_cap, A.flags, A.ring, A.ctrl, io->status, st); if (rc) return rc;
        p->mark("hysteresis");
        launches += 1;
        if (any_tap_edge) {
            rc = launch_bitmap_to_u8(Pd, p->planes.data(), NP, st); if (rc) return rc;
            launches++;
        }
        for (int l = 0; l < 3; l++)
            if (io->tap_layers[l])
                AEAJ_CUDA(cudaMemcpyAsync(io->tap_layers[l], p->planes[l].layer_f32, sizeof(float) * (size_t)B * p->info.layer_h[l] * p->info.layer_w[l],
                                          cudaMemcpyDeviceToDevice, st));
    }
    // quadtree: per-top-block counts (band), scan over all top blocks (needs every band's counts), emit (band)
    const int qt_parts = ((phases & (1u << AEAJ_PHASE_QT_COUNT)) ? 1 : 0) | ((phases & (1u << AEAJ_PHASE_QT_EMIT)) ? 6 : 0);
    if (qt_parts) {
        rc = launch_quadtree(Pd, p->planes.data(), NP, p->info.block_min, p->info.block_max, A.class_lists, A.class_counts,
                             p->class_off_dev, st, &launches, qt_parts);
        if (rc) return rc;
        if ((qt_parts & 4) && (io->packed_states[0] || io->packed_states[1] || io->packed_states[2])) {
            rc = launch_pack_states(Pd, p->planes.data(), NP, st); if (rc) return rc;
            launches++;
        }
        p->mark("quadtree");
    }
    if (phases & (1u << AEAJ_PHASE_DCT)) {
        rc = launch_dct_quant(h, Pd, A.class_lists, A.class_counts, p->cg.off, p->cg.cap, p->lg_min, p->lg_max, st, &launches,
                              plan_mark_cb, p, p->tensor_dct, A.scratch256);
        if (rc) return rc;
        if (io->status) AEAJ_CUDA(cudaMemcpyAsync(io->status + 2, h->tc_err_dev, sizeof(int), cudaMemcpyDeviceToDevice, st));
    }
    p->last_launches = launches;
    return 0;
}

extern "C" int aeaj_encode(aeaj_plan* p, const aeaj_encode_io* io, void* workspace, void* stream) {
    return encode_impl(p, io, workspace, ST(stream), (1u << (AEAJ_PHASE_DCT + 1)) - 1, 0, -1);      // every phase, whole image
}

static int decode_impl(aeaj_plan* p, const aeaj_decode_io* io, void* workspace, cudaStream_t st, unsigned phases, int band0, int band1) {
    AEAJ_REQUIRE(p && io && workspace && (io->rgb || io->rgb_u8) && io->counts, "aeaj_decode: bad arguments (rgb or rgb_u8 required)");
    AEAJ_REQUIRE(p->qtab_dev, "aeaj_decode: quantisation tables not set (aeaj_plan_set_qtables)");
    aeaj_handle* h = p->h;
    const int B = p->info.batch, NP = p->nplanes;
    int launches = 0;
    PlanAux A;
    plan_carve(p, workspace, A);
    for (int l = 0; l < 3; l++) {
        AEAJ_REQUIRE(io->coef[l] && io->leaves[l], "aeaj_decode: NULL input buffer");
        for (int i = 0; i < B; i++) {
            PlaneDesc& P = p->planes[i * 3 + l];
            P.coef = (int32_t*)io->coef[l] + (size_t)i * p->info.cap_coef[l];
            P.leaves = (int32_t*)io->leaves[l] + (size_t)i * p->info.cap_leaves[l] * 4;
            P.counts = (int32_t*)io->counts + ((size_t)i * 3 + l) * 4;
            P.packed_states = nullptr;
            P.tap_edge = nullptr;
        }
    }
    int rc = set_band(p, band0, band1); if (rc) return rc;
    PlaneDesc* Pd;
    rc = plan_push_planes(p, st, Pd); if (rc) return rc;
    p->ev_n = 0; p->ev_stream = st; p->mark("start");
    if (phases & (1u << AEAJ_DPHASE_IDCT)) {
        AEAJ_CUDA(cudaMemsetAsync(A.class_counts, 0, 16 * sizeof(int), st));
        rc = launch_bucket_leaves(Pd, p->planes.data(), NP, A.class_lists, A.class_counts, p->class_off_dev, p->lg_min, p->lg_max, st);
        if (rc) return rc;
        launches++;
        p->mark("bucket_leaves");
        rc = launch_dequant_idct(h, Pd, A.class_lists, A.class_counts, p->cg.off, p->cg.cap, p->lg_min, p->lg_max, st, &launches,
                                 plan_mark_cb, p, p->tensor_dct, A.scratch256);
        if (rc) return rc;
        if (io->status) {
            AEAJ_CUDA(cudaMemcpyAsync(io->status + 2, h->tc_err_dev, sizeof(int), cudaMemcpyDeviceToDevice, st));
            AEAJ_CUDA(cudaMemcpyAsync(io->status + 3, A.class_counts + 15, sizeof(int), cudaMemcpyDeviceToDevice, st));
        }
        for (int l = 0; l < 3; l++)
            if (io->tap_layers[l])
                AEAJ_CUDA(cudaMemcpyAsync(io->tap_layers[l], p->planes[l].layer_f32, sizeof(float) * (size_t)B * p->info.layer_h[l] * p->info.layer_w[l],
                                          cudaMemcpyDeviceToDevice, st));
    }
    if (phases & (1u << AEAJ_DPHASE_COLOR)) {
        rc = launch_upsample_color_inverse(h, p->info.space, p->planes.data(), B, p->info.height, p->info.width, io->rgb, io->rgb_u8, st, band0, band1);
        if (rc) return rc;
        launches++;
        p->mark("upsample_color_inverse");
    }
    p->last_launches = launches;
    return 0;
}
extern "C" int aeaj_decode(aeaj_plan* p, const aeaj_decode_io* io, void* workspace, void* stream) {
    return decode_impl(p, io, workspace, ST(stream), 0x3u, 0, -1);
}

// ---------------------------------------------------------------------------------------------
// scaled decode (idct_scaled.cu): 1/scale of every layer from the top-left coefficients of each leaf
// ---------------------------------------------------------------------------------------------
struct ScaledGeom {
    int k, m;                        // scale; the IDCT's own factor min(scale, block_min)
    int out_h, out_w;
    int hm[3], wm[3];                // the 1/m layers
    int hk[3], wk[3];                // the 1/scale layers (== the 1/m layers when scale <= block_min)
};
static int scaled_geom(const aeaj_plan* p, int scale, ScaledGeom& g) {
    AEAJ_REQUIRE(scale == 1 || scale == 2 || scale == 4 || scale == 8, "aeaj_decode_scaled: scale must be 1, 2, 4 or 8");
    g.k = scale; g.m = std::min(scale, p->info.block_min);
    g.out_h = aeaj_cdiv(p->info.height, scale); g.out_w = aeaj_cdiv(p->info.width, scale);
    for (int l = 0; l < 3; l++) {
        g.hm[l] = aeaj_cdiv(p->info.layer_h[l], g.m); g.wm[l] = aeaj_cdiv(p->info.layer_w[l], g.m);
        g.hk[l] = aeaj_cdiv(p->info.layer_h[l], scale); g.wk[l] = aeaj_cdiv(p->info.layer_w[l], scale);
    }
    return 0;
}
// the caller's scratch: per layer the batch's 1/m planes, then (scale > block_min) the 1/scale planes; nullptr: size only
static size_t scaled_carve(const aeaj_plan* p, const ScaledGeom& g, void* scratch, float* mp[3], float* kp[3]) {
    if (g.k == 1) { for (int l = 0; l < 3; l++) mp[l] = kp[l] = nullptr; return 0; }
    Bump b(scratch ? (void*)(((uintptr_t)scratch + 255) & ~(uintptr_t)255) : nullptr);
    const int B = p->info.batch;
    for (int l = 0; l < 3; l++) {
        mp[l] = b.take<float>((size_t)B * g.hm[l] * g.wm[l]);
        kp[l] = (g.k > g.m) ? b.take<float>((size_t)B * g.hk[l] * g.wk[l]) : mp[l];
    }
    return b.used() + 256;
}

extern "C" int aeaj_decode_scaled_geometry(const aeaj_plan* p, int scale, int* out_h, int* out_w, int layer_h[3], int layer_w[3],
                                           int64_t* scratch_bytes) {
    AEAJ_REQUIRE(p && out_h && out_w && layer_h && layer_w && scratch_bytes, "aeaj_decode_scaled_geometry: bad arguments");
    ScaledGeom g;
    int rc = scaled_geom(p, scale, g); if (rc) return rc;
    *out_h = g.out_h; *out_w = g.out_w;
    for (int l = 0; l < 3; l++) { layer_h[l] = g.hk[l]; layer_w[l] = g.wk[l]; }
    float* mp[3]; float* kp[3];
    *scratch_bytes = (int64_t)scaled_carve(p, g, nullptr, mp, kp);
    return 0;
}

extern "C" int aeaj_decode_scaled(aeaj_plan* p, const aeaj_decode_io* io, int scale, void* workspace, void* scratch, void* stream) {
    AEAJ_REQUIRE(p && io && workspace && (io->rgb || io->rgb_u8) && io->counts, "aeaj_decode_scaled: bad arguments (rgb or rgb_u8 required)");
    AEAJ_REQUIRE(p->peers.world == 1, "aeaj_decode_scaled: a plan with peers (multi-GPU halo-split) is not supported");
    ScaledGeom g;
    int rc = scaled_geom(p, scale, g); if (rc) return rc;
    const cudaStream_t st = ST(stream);
    if (scale == 1) return decode_impl(p, io, workspace, st, 0x3u, 0, -1);
    AEAJ_REQUIRE(scratch, "aeaj_decode_scaled: NULL scratch");
    AEAJ_REQUIRE(p->qtab_dev, "aeaj_decode_scaled: quantisation tables not set (aeaj_plan_set_qtables)");
    aeaj_handle* h = p->h;
    const int B = p->info.batch, NP = p->nplanes;
    PlanAux A;
    plan_carve(p, workspace, A);
    float* mp[3]; float* kp[3];
    scaled_carve(p, g, scratch, mp, kp);
    p->scaled_planes = p->planes;
    for (int l = 0; l < 3; l++) {
        AEAJ_REQUIRE(io->coef[l] && io->leaves[l], "aeaj_decode_scaled: NULL input buffer");
        for (int i = 0; i < B; i++) {
            PlaneDesc& P = p->scaled_planes[i * 3 + l];
            P.coef = (int32_t*)io->coef[l] + (size_t)i * p->info.cap_coef[l];
            P.leaves = (int32_t*)io->leaves[l] + (size_t)i * p->info.cap_leaves[l] * 4;
            P.counts = (int32_t*)io->counts + ((size_t)i * 3 + l) * 4;
            P.packed_states = nullptr;
            P.tap_edge = nullptr;
            P.ry0 = 0; P.ry1 = P.h; P.peer_up = P.peer_dn = 0;
            P.zigzag = p->zigzag;
            for (int k = 0; k < 9; k++) P.zz[k] = h->zz_dev[k];
            P.layer_f32 = mp[l] + (size_t)i * g.hm[l] * g.wm[l];
        }
    }
    PlaneDesc* Pd;
    rc = p->scaled_tab[ilog2i(scale)].push(p->scaled_planes, st, Pd); if (rc) return rc;
    int launches = 0;
    p->ev_n = 0; p->ev_stream = st; p->mark("start");
    AEAJ_CUDA(cudaMemsetAsync(A.class_counts, 0, 16 * sizeof(int), st));
    rc = launch_bucket_leaves(Pd, p->scaled_planes.data(), NP, A.class_lists, A.class_counts, p->class_off_dev, p->lg_min, p->lg_max, st);
    if (rc) return rc;
    launches++;
    p->mark("bucket_leaves");
    rc = launch_idct_scaled(h, Pd, A.class_lists, A.class_counts, p->cg.off, p->cg.cap, p->lg_min, p->lg_max, g.m, st, &launches);
    if (rc) return rc;
    p->mark("idct_scaled");
    if (g.k > g.m) {
        for (int l = 0; l < 3; l++) {
            rc = launch_box_reduce(mp[l], g.hm[l], g.wm[l], kp[l], g.hk[l], g.wk[l], g.k / g.m, B, st); if (rc) return rc;
            launches++;
        }
        p->mark("box_reduce");
    }
    if (io->status) {
        AEAJ_CUDA(cudaMemcpyAsync(io->status + 2, h->tc_err_dev, sizeof(int), cudaMemcpyDeviceToDevice, st));
        AEAJ_CUDA(cudaMemcpyAsync(io->status + 3, A.class_counts + 15, sizeof(int), cudaMemcpyDeviceToDevice, st));
    }
    for (int l = 0; l < 3; l++)
        if (io->tap_layers[l])
            AEAJ_CUDA(cudaMemcpyAsync(io->tap_layers[l], kp[l], sizeof(float) * (size_t)B * g.hk[l] * g.wk[l], cudaMemcpyDeviceToDevice, st));
    // the colour tail reads the 1/scale layers through host descriptors of their final geometry
    PlaneDesc tail[3];
    for (int l = 0; l < 3; l++) {
        memset(&tail[l], 0, sizeof tail[l]);
        tail[l].h = g.hk[l]; tail[l].w = g.wk[l]; tail[l].ry0 = 0; tail[l].ry1 = g.hk[l]; tail[l].layer = l;
        tail[l].layer_f32 = kp[l];
    }
    rc = launch_upsample_color_inverse(h, p->info.space, tail, B, g.out_h, g.out_w, io->rgb, io->rgb_u8, st);
    if (rc) return rc;
    launches++;
    p->mark("upsample_color_inverse");
    p->last_launches = launches;
    return 0;
}

// ---------------------------------------------------------------------------------------------
// packed coefficient streams (pack.cu)
// ---------------------------------------------------------------------------------------------
static int pack_impl(aeaj_plan* p, const int32_t* const* coef3, const int32_t* counts, const aeaj_packed_io* pk, void* workspace, cudaStream_t st, int unpack) {
    AEAJ_REQUIRE(p && coef3 && pk && pk->counts && workspace && (unpack || counts), "aeaj_(un)pack_coefficients: bad arguments");
    const int B = p->info.batch;
    PlanAux A;
    plan_carve(p, workspace, A);
    int64_t max_cap = 1;
    for (int l = 0; l < 3; l++) {
        AEAJ_REQUIRE(coef3[l] && pk->mask[l] && pk->vals[l], "aeaj_(un)pack_coefficients: NULL buffer");
        const int64_t cap = p->info.cap_coef[l];
        max_cap = std::max(max_cap, cap);
        const size_t per = aeaj_pack_scratch_ints(cap);
        for (int i = 0; i < B; i++) {
            PackPlane& P = p->pack_planes[i * 3 + l];
            P.coef = coef3[l] + (size_t)i * cap;
            P.mask = pk->mask[l] + (size_t)i * (cap / 32 + 1);
            P.vals = pk->vals[l] + (size_t)i * cap;
            P.pk_counts = pk->counts + ((size_t)i * 3 + l) * 4;
            P.n_coef = unpack ? P.pk_counts + 1 : counts + ((size_t)i * 3 + l) * 4 + 2;
            P.chunk_sums = A.pack_sums[l] + per * i;
            P.cap_coef = cap;
        }
    }
    if (!unpack) AEAJ_CUDA(cudaMemsetAsync(pk->counts, 0, sizeof(int32_t) * 12 * (size_t)B, st));
    PackPlane* table;
    int rc = (unpack ? p->unpack_tab : p->pack_tab).push(p->pack_planes, st, table); if (rc) return rc;
    return launch_pack(table, p->nplanes, max_cap, unpack, st);
}
extern "C" int aeaj_pack_coefficients(aeaj_plan* p, const int32_t* const* coef3, const int32_t* counts, const aeaj_packed_io* out,
                                      void* workspace, void* stream) {
    return pack_impl(p, coef3, counts, out, workspace, ST(stream), 0);
}
extern "C" int aeaj_unpack_coefficients(aeaj_plan* p, const aeaj_packed_io* in, int32_t* const* coef3, void* workspace, void* stream) {
    return pack_impl(p, coef3, nullptr, in, workspace, ST(stream), 1);
}
// ---------------------------------------------------------------------------------------------
// device deflate of the coefficient streams (deflate.cu)
// ---------------------------------------------------------------------------------------------
static int64_t deflate_chunks_cap(const aeaj_plan* p, int l) { return df_chunks(4 * p->info.cap_coef[l]); }
static int64_t deflate_cap_out(const aeaj_plan* p, int l) { return (df_stream_bound(4 * p->info.cap_coef[l]) + 15) & ~(int64_t)15; }

// the deflate scratch, per layer, per image: output slots | tokens | chunk offsets | lengths | Adler-32 sums.  Sets the scratch
// pointers of planes[nplanes] (nullptr: size only) and returns the bytes the caller provides.
static size_t deflate_carve(const aeaj_plan* p, void* scratch, DeflatePlane* planes) {
    Bump b(scratch ? (void*)(((uintptr_t)scratch + 255) & ~(uintptr_t)255) : nullptr);
    for (int l = 0; l < 3; l++) {
        const int64_t nch = deflate_chunks_cap(p, l);
        for (int i = 0; i < p->info.batch; i++) {
            DeflatePlane size_only;
            DeflatePlane& P = planes ? planes[i * 3 + l] : size_only;
            P.slots = b.take<uint8_t>(nch * DF_CHUNK_BOUND);
            P.tok = b.take<uint16_t>(nch * DF_CHUNK);
            P.chunk_off = b.take<int64_t>(nch);
            P.chunk_len = b.take<int32_t>(nch);
            P.chunk_adler = b.take<uint32_t>(nch);
        }
    }
    return b.used() + 256;
}

extern "C" int aeaj_deflate_caps(const aeaj_plan* p, int64_t* cap_out3, int64_t* scratch_bytes) {
    AEAJ_REQUIRE(p && cap_out3 && scratch_bytes, "aeaj_deflate_caps: bad arguments");
    for (int l = 0; l < 3; l++) cap_out3[l] = deflate_cap_out(p, l);
    *scratch_bytes = (int64_t)deflate_carve(p, nullptr, nullptr);
    return 0;
}

extern "C" int aeaj_deflate_coefficients(aeaj_plan* p, const int32_t* const* coef3, const int32_t* counts, const aeaj_deflate_io* io,
                                         void* scratch, void* stream) {
    AEAJ_REQUIRE(p && coef3 && counts && io && io->lengths && scratch, "aeaj_deflate_coefficients: bad arguments");
    const cudaStream_t st = ST(stream);
    const int B = p->info.batch;
    p->df_planes.resize(p->nplanes);
    deflate_carve(p, scratch, p->df_planes.data());
    int max_chunks = 1;
    for (int l = 0; l < 3; l++) {
        AEAJ_REQUIRE(coef3[l] && io->out[l], "aeaj_deflate_coefficients: NULL buffer");
        const int64_t cap = p->info.cap_coef[l], nch = deflate_chunks_cap(p, l), cap_out = deflate_cap_out(p, l);
        max_chunks = std::max<int>(max_chunks, (int)nch);
        for (int i = 0; i < B; i++) {
            DeflatePlane& P = p->df_planes[i * 3 + l];
            P.in = (const uint8_t*)(coef3[l] + (size_t)i * cap);
            P.n_coef = counts + ((size_t)i * 3 + l) * 4 + 2;
            P.cap_coef = cap;
            P.out = io->out[l] + (size_t)i * cap_out;
            P.cap_out = cap_out;
            P.length = io->lengths + (size_t)i * 3 + l;
            P.status = io->status;
        }
    }
    if (io->status) AEAJ_CUDA(cudaMemsetAsync(io->status, 0, 4 * sizeof(int32_t), st));
    DeflatePlane* table;
    int rc = p->deflate_tab.push(p->df_planes, st, table); if (rc) return rc;
    return launch_deflate(table, p->nplanes, max_chunks, st);
}

// ---------------------------------------------------------------------------------------------
// device inflate of the coefficient streams (inflate.cu)
// ---------------------------------------------------------------------------------------------
// scratch: counters | per-plane streams | candidate segments | position map; the list holds every sync point of real
// streams (one per 64 KiB chunk of output at most a few bytes apart only for hostile input); beyond it, a plane decodes
// the rest of its stream in one piece
struct InflateLayout { int64_t cap_segs, streams, segs, map, total; };
static InflateLayout inflate_layout(int nplanes, int64_t in_bytes) {
    InflateLayout L;
    L.cap_segs = std::min<int64_t>(nplanes + in_bytes / 16 + 64, 1 << 30);
    L.streams = 256;
    L.segs = L.streams + ((nplanes * (int64_t)sizeof(IfStream) + 255) & ~(int64_t)255);
    L.map = L.segs + ((L.cap_segs * (int64_t)sizeof(IfSeg) + 255) & ~(int64_t)255);
    L.total = L.map + (in_bytes / 4 + 1) * 4 + 256;
    return L;
}

extern "C" int aeaj_inflate_scratch_bytes(const aeaj_plan* p, int64_t in_bytes, int64_t* scratch_bytes) {
    AEAJ_REQUIRE(p && scratch_bytes && in_bytes >= 0, "aeaj_inflate_scratch_bytes: bad arguments");
    *scratch_bytes = inflate_layout(p->nplanes, in_bytes).total;
    return 0;
}

extern "C" int aeaj_inflate_coefficients(aeaj_plan* p, const aeaj_inflate_io* io, const int32_t* counts, int64_t in_bytes,
                                         void* scratch, void* stream) {
    AEAJ_REQUIRE(p && io && counts && scratch && in_bytes >= 0 && io->offsets && io->lengths && io->status && io->out_bytes &&
                 io->segments && (io->in || in_bytes == 0), "aeaj_inflate_coefficients: bad arguments");
    const cudaStream_t st = ST(stream);
    const int B = p->info.batch;
    p->if_planes.resize(p->nplanes);
    for (int l = 0; l < 3; l++) {
        AEAJ_REQUIRE(io->coef[l], "aeaj_inflate_coefficients: NULL buffer");
        const int64_t cap = p->info.cap_coef[l];
        for (int i = 0; i < B; i++) {
            const size_t k = (size_t)i * 3 + l;
            InflatePlane& P = p->if_planes[k];
            P.offset = io->offsets + k;
            P.length = io->lengths + k;
            P.n_coef = counts + k * 4 + 2;
            P.out = (uint8_t*)(io->coef[l] + (size_t)i * cap);
            P.cap_bytes = 4 * cap;
            P.status = io->status + k;
            P.out_bytes = io->out_bytes + k;
            P.segments = io->segments + k;
        }
    }
    const InflateLayout L = inflate_layout(p->nplanes, in_bytes);
    uint8_t* base = (uint8_t*)(((uintptr_t)scratch + 255) & ~(uintptr_t)255);
    InflateArgs a;
    a.in = io->in; a.in_bytes = in_bytes; a.nplanes = p->nplanes; a.cap_segs = (int)L.cap_segs;
    a.counters = (int*)base;
    a.streams = (IfStream*)(base + L.streams);
    a.segs = (IfSeg*)(base + L.segs);
    a.map = (int32_t*)(base + L.map);
    InflatePlane* table;
    int rc = p->inflate_tab.push(p->if_planes, st, table); if (rc) return rc;
    return launch_inflate(table, a, p->h->sm_count, st);
}

extern "C" int aeaj_pack_coefficients_host(const int32_t* coef, int64_t n, uint32_t* mask, int16_t* vals, int64_t* nnz, int* overflow) {
    AEAJ_REQUIRE(coef && mask && vals && nnz && n >= 0, "aeaj_pack_coefficients_host: bad arguments");
    int64_t k = 0;
    int ovf = 0;
    for (int64_t w = 0; w * 32 < n; w++) {
        uint32_t m = 0;
        const int64_t e = std::min<int64_t>(n - w * 32, 32);
        for (int64_t i = 0; i < e; i++) {
            const int32_t v = coef[w * 32 + i];
            if (v != 0) { m |= 1u << i; vals[k++] = (int16_t)v; ovf |= (v > 32767 || v < -32768); }
        }
        mask[w] = m;
    }
    *nnz = k;
    if (overflow) *overflow = ovf;
    return 0;
}
extern "C" int aeaj_unpack_coefficients_host(const uint32_t* mask, const int16_t* vals, int64_t n, int64_t nnz, int32_t* coef) {
    AEAJ_REQUIRE(coef && mask && (vals || nnz == 0) && n >= 0 && nnz >= 0, "aeaj_unpack_coefficients_host: bad arguments");
    int64_t k = 0;
    for (int64_t w = 0; w * 32 < n; w++) {
        const uint32_t m = mask[w];
        const int64_t e = std::min<int64_t>(n - w * 32, 32);
        if (m == 0) { for (int64_t i = 0; i < e; i++) coef[w * 32 + i] = 0; continue; }
        for (int64_t i = 0; i < e; i++) {
            int32_t v = 0;
            if ((m >> i) & 1u) { AEAJ_REQUIRE(k < nnz, "packed stream: more mask bits than values"); v = vals[k++]; }
            coef[w * 32 + i] = v;
        }
    }
    AEAJ_REQUIRE(k == nnz, "packed stream: value count does not match the mask");
    return 0;
}

// gather / scatter of one frame's variable-length streams into / out of one contiguous arena (include/aeaj.h)
extern "C" int aeaj_copy_segments(const aeaj_segment* segs_host, int n, void* table_dev, void* stream) {
    AEAJ_REQUIRE(n >= 0 && (n == 0 || segs_host), "aeaj_copy_segments: bad arguments");
    static_assert(sizeof(aeaj_segment) == sizeof(PeerSeg), "segment layout");
    long long maxb = 0;
    int m = 0;
    std::vector<PeerSeg> segs((size_t)n);
    for (int i = 0; i < n; i++) {
        const aeaj_segment& s = segs_host[i];
        AEAJ_REQUIRE(s.bytes >= 0, "aeaj_copy_segments: negative size");
        if (s.bytes == 0) continue;
        AEAJ_REQUIRE(s.src && s.dst, "aeaj_copy_segments: NULL range");
        segs[m].src = s.src; segs[m].dst = s.dst; segs[m].bytes = s.bytes; m++;
        maxb = std::max<long long>(maxb, s.bytes);
    }
    if (m == 0) return 0;
    if (m <= AEAJ_SEGS_BY_PARAM) return launch_copy_segments_param(segs.data(), m, maxb, ST(stream));   // table in the kernel parameters: no upload
    AEAJ_REQUIRE(table_dev, "aeaj_copy_segments: more than 64 ranges need the device scratch table");
    AEAJ_CUDA(cudaMemcpyAsync(table_dev, segs.data(), sizeof(PeerSeg) * m, cudaMemcpyHostToDevice, ST(stream)));   // pageable: staged before return
    return launch_peer_gather((const PeerSeg*)table_dev, m, maxb, ST(stream));
}

// ---------------------------------------------------------------------------------------------
// one image over several GPUs: peers (peer.cu)
// ---------------------------------------------------------------------------------------------
extern "C" int aeaj_plan_set_peers(aeaj_plan* p, int rank, int world, void* const* peer_workspaces_host, void* const* peer_flags_host) {
    AEAJ_REQUIRE(p && world >= 1 && world <= AEAJ_MAX_PEERS && rank >= 0 && rank < world, "aeaj_plan_set_peers: bad arguments");
    AEAJ_REQUIRE(p->info.batch == 1, "a multi-GPU halo-split plan holds one image");
    AEAJ_REQUIRE(world == 1 || (peer_workspaces_host && peer_flags_host), "aeaj_plan_set_peers: NULL peer tables");
    p->peers.world = world; p->peers.rank = rank;
    for (int r = 0; r < AEAJ_MAX_PEERS; r++) {
        p->peer_ws[r] = r < world && peer_workspaces_host ? peer_workspaces_host[r] : nullptr;
        p->peer_flags[r] = r < world && peer_flags_host ? (int*)peer_flags_host[r] : nullptr;
        p->peers.delta[r] = 0;
    }
    for (int r = 0; r < world && world > 1; r++) {
        AEAJ_REQUIRE(p->peer_ws[r] && p->peer_flags[r], "aeaj_plan_set_peers: NULL peer pointer");
        p->peers.delta[r] = (long long)((const char*)p->peer_ws[r] - (const char*)p->peer_ws[rank]);
    }
    p->planes_tab.forget();
    if (world > 1 && !p->peer_segs_dev) {
        AEAJ_CUDA(cudaSetDevice(p->h->device));
        AEAJ_CUDA(cudaMalloc(&p->peer_segs_dev, sizeof(PeerSeg) * 64 * 2));
    }
    return 0;
}

// band b of n: full-resolution rows [b*H/n, (b+1)*H/n) (H is a multiple of n, run_halo checks it)
static int band_row(const aeaj_plan* p, int b, int n) { return p->info.height / n * b; }

// all ranks meet: everything the ranks enqueued before the barrier is complete and visible before anything enqueued after it runs
static int peer_barrier(aeaj_plan* p, cudaStream_t st) {
    if (p->peers.world <= 1) return 0;
    p->peer_epoch++;
    return launch_peer_barrier(p->peer_flags, p->peers.rank, p->peers.world, p->peer_epoch, p->h->tc_err_dev, st);
}

// copy the other ranks' rows into this rank's buffers.  what = 0: the strong / weak candidate bitmaps (before the replicated
// hysteresis); what = 1: the per-top-block quadtree totals (before the scan).  Rank r owns band r of world.
static int peer_gather(aeaj_plan* p, int what, void* workspace, cudaStream_t st) {
    const int world = p->peers.world, rank = p->peers.rank;
    if (world <= 1) return 0;
    PlanAux A;
    plan_carve(p, workspace, A);
    const int H = p->info.height;
    std::vector<PeerSeg> segs;
    long long maxb = 0;
    auto add = [&](const void* mine, long long off, long long bytes, int r) {
        if (bytes <= 0) return;
        PeerSeg s;
        s.dst = (char*)mine + off; s.src = (const char*)mine + p->peers.delta[r] + off; s.bytes = bytes;
        segs.push_back(s); maxb = std::max(maxb, bytes);
    };
    for (int r = 0; r < world; r++) {
        if (r == rank) continue;
        const int b0 = band_row(p, r, world), b1 = band_row(p, r + 1, world);
        for (int l = 0; l < 3; l++) {
            const PlaneDesc& P = p->planes[l];
            const int rh = H / P.h;
            const int y0 = b0 / rh, y1 = (b1 == H) ? P.h : b1 / rh;
            if (what == 0) {
                add(P.strong, (long long)y0 * P.wpr * 4, (long long)(y1 - y0) * P.wpr * 4, r);
                add(P.weak, (long long)y0 * P.wpr * 4, (long long)(y1 - y0) * P.wpr * 4, r);
            } else {
                const int t0 = y0 / P.top, t1 = aeaj_cdiv(y1, P.top);      // top-block rows of that band
                add(P.tb_tot, (long long)t0 * P.ntx * sizeof(int2), (long long)(t1 - t0) * P.ntx * sizeof(int2), r);
                add(P.tb_coef, (long long)t0 * P.ntx * sizeof(int), (long long)(t1 - t0) * P.ntx * sizeof(int), r);
            }
        }
    }
    AEAJ_REQUIRE(segs.size() <= 64, "too many gather segments");
    PeerSeg* dev = p->peer_segs_dev + (what ? 64 : 0);
    AEAJ_CUDA(cudaMemcpyAsync(dev, segs.data(), sizeof(PeerSeg) * segs.size(), cudaMemcpyHostToDevice, st));
    return launch_peer_gather(dev, (int)segs.size(), maxb, st);
}

// The halo-split schedule, written once.  A step is a barrier of all ranks, a gather, or one phase.  A phase step runs once for
// every band the call covers, in band order: phase-major, because COLOR clears the histogram accumulators that every band's
// CLAHE_HIST adds to.  Hysteresis covers the whole image and runs once.
enum HaloStepKind { STEP_BARRIER, STEP_GATHER, STEP_PHASE, STEP_PHASE_ONCE };
struct HaloStep { HaloStepKind kind; int arg; };
static const HaloStep ENCODE_HALO[] = {
    {STEP_BARRIER, 0},                                    // the previous call's neighbours are done reading this rank's planes
    {STEP_PHASE, AEAJ_PHASE_COLOR}, {STEP_PHASE, AEAJ_PHASE_CLAHE_HIST}, {STEP_BARRIER, 0},
    {STEP_PHASE, AEAJ_PHASE_PREFILTER}, {STEP_BARRIER, 0},
    {STEP_PHASE, AEAJ_PHASE_NMS}, {STEP_BARRIER, 0},
    {STEP_GATHER, 0}, {STEP_PHASE_ONCE, AEAJ_PHASE_HYST}, {STEP_PHASE, AEAJ_PHASE_QT_COUNT}, {STEP_BARRIER, 0},
    {STEP_GATHER, 1}, {STEP_PHASE, AEAJ_PHASE_QT_EMIT}, {STEP_PHASE, AEAJ_PHASE_DCT}};
static const HaloStep DECODE_HALO[] = {{STEP_PHASE, AEAJ_DPHASE_IDCT}, {STEP_BARRIER, 0}, {STEP_PHASE, AEAJ_DPHASE_COLOR}};

// Walks `steps` for the bands this call covers: on a plan with peers this rank's band (bands == world), without peers every band
// in turn on this GPU (barriers and gathers do nothing there).  run(phases, band0, band1) is encode_impl / decode_impl.
template <size_t N, class Run>
static int run_halo(aeaj_plan* p, const HaloStep (&steps)[N], int bands, void* workspace, cudaStream_t st, Run run) {
    AEAJ_REQUIRE(p && bands >= 1 && p->info.height % bands == 0, "halo-split: the image height must be a multiple of bands >= 1");
    int first = 0, last = bands;
    if (p->peers.world > 1) {
        AEAJ_REQUIRE(bands == p->peers.world, "halo-split: a plan with peers runs one band per rank (bands == world)");
        AEAJ_REQUIRE(workspace == p->peer_ws[p->peers.rank], "halo-split: the workspace must be the shared allocation registered with aeaj_plan_set_peers");
        first = p->peers.rank; last = first + 1;
    }
    for (const HaloStep& s : steps) {
        int rc = 0;
        if (s.kind == STEP_BARRIER) rc = peer_barrier(p, st);
        else if (s.kind == STEP_GATHER) rc = peer_gather(p, s.arg, workspace, st);
        else
            for (int b = first; b < (s.kind == STEP_PHASE_ONCE ? first + 1 : last) && !rc; b++)
                rc = run(1u << s.arg, band_row(p, b, bands), band_row(p, b + 1, bands));
        if (rc) return rc;
    }
    return 0;
}
extern "C" int aeaj_encode_halo(aeaj_plan* p, const aeaj_encode_io* io, void* workspace, void* stream, int bands) {
    const cudaStream_t st = ST(stream);
    return run_halo(p, ENCODE_HALO, bands, workspace, st,
                    [&](unsigned ph, int b0, int b1) { return encode_impl(p, io, workspace, st, ph, b0, b1); });
}
extern "C" int aeaj_decode_halo(aeaj_plan* p, const aeaj_decode_io* io, void* workspace, void* stream, int bands) {
    const cudaStream_t st = ST(stream);
    return run_halo(p, DECODE_HALO, bands, workspace, st,
                    [&](unsigned ph, int b0, int b1) { return decode_impl(p, io, workspace, st, ph, b0, b1); });
}

// ---------------------------------------------------------------------------------------------
// host-side helpers (entropy-coding side; CPU only)
// ---------------------------------------------------------------------------------------------
// The state stream comes from a file: nothing in it is trusted.  Rejected (AEAJ_EINVAL, the shim raises ValueError where the
// reference dies with a KeyError on zigzag_cache[size], jpeg.py:665): a root that is not the layer's root, a split below
// size 2, a leaf outside [block_min, block_max] (0 = unchecked) or outside the layer.  State 3 splits like the reference's
// `else` branch (jpeg.py:793); a truncated stream yields the leaves seen so far, as jpeg.py:784 does.
extern "C" int aeaj_states_to_leaves_host(const uint8_t* states, int n_states, int root, int h, int w, int block_min, int block_max,
                                          int32_t* leaves, int* n_leaves, int64_t* n_coef) {
    AEAJ_REQUIRE(states && leaves && n_leaves && n_states >= 0 && root > 0 && h > 0 && w > 0, "aeaj_states_to_leaves_host: bad arguments");
    AEAJ_REQUIRE(root == aeaj_root_size(h, w), "state stream: root size does not match the layer shape");
    struct Node { int x, y, s; };
    std::vector<Node> st;
    st.push_back({0, 0, root});
    int nl = 0, si = 0;
    int64_t off = 0;
    while (!st.empty() && si < n_states) {
        Node nd = st.back(); st.pop_back();
        int s = states[si++];
        if (s == 0) {
            AEAJ_REQUIRE(nd.x < w && nd.y < h, "state stream: leaf outside the layer");
            AEAJ_REQUIRE(nd.s >= 2 && (block_max <= 0 || (nd.s >= block_min && nd.s <= block_max)), "state stream: leaf size outside the block range");
            AEAJ_REQUIRE(off + (int64_t)nd.s * nd.s < ((int64_t)1 << 31), "state stream: coefficient offsets overflow");
            leaves[4 * nl] = nd.x; leaves[4 * nl + 1] = nd.y; leaves[4 * nl + 2] = nd.s; leaves[4 * nl + 3] = (int32_t)off;
            off += (int64_t)nd.s * nd.s; nl++;
        } else if (s != 2) {
            AEAJ_REQUIRE(nd.s >= 4 && (block_min <= 0 || nd.s > block_min), "state stream: split below the minimum block size");
            int hs = nd.s / 2;
            st.push_back({nd.x + hs, nd.y + hs, hs});
            st.push_back({nd.x, nd.y + hs, hs});
            st.push_back({nd.x + hs, nd.y, hs});
            st.push_back({nd.x, nd.y, hs});
        }
    }
    *n_leaves = nl;
    if (n_coef) *n_coef = off;
    return 0;
}
extern "C" int aeaj_pack_states_host(const uint8_t* states, int n, uint8_t* packed) {
    AEAJ_REQUIRE(states && packed && n >= 0, "aeaj_pack_states_host: bad arguments");
    for (int i = 0; i < (n + 3) / 4; i++) {
        unsigned v = 0;
        for (int k = 0; k < 4; k++) { int idx = 4 * i + k; v = (v << 2) | (idx < n ? (states[idx] & 3u) : 0u); }
        packed[i] = (uint8_t)v;
    }
    return 0;
}
