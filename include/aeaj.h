/*
 * aeaj.h -- C ABI of libaeaj.so: the B200 (sm_100a) implementation of the adaptive edge-aware
 * JPEG hot path.  This is the drop-in boundary: plain pointers and sizes, no C++/torch types.
 *
 * The reference (fevzibabaoglu/adaptive-edge-aware-jpeg) is pure Python and has no FFI of its own;
 * each entry point below replaces the reference call site cited beside it (paths under
 * /root/reference/src).  The Python host shim that binds these with ctypes lives in
 * adaptive-edge-aware-jpeg_b200/aeaj/native.py; INTEGRATION.md shows the binding a maintainer of
 * the reference would add.
 *
 * Conventions
 *   - every export returns int: 0 = ok, <0 = AEAJ_E*, >0 = cudaError_t; aeaj_last_error() gives text.
 *   - all data pointers are DEVICE pointers unless the name ends in _host.
 *   - every call is asynchronous on the cudaStream_t passed as `void* stream` (NULL = default stream)
 *     unless documented otherwise; the caller owns every buffer; the library owns only handles/plans.
 *   - a handle/plan is not re-entrant; distinct handles are independent.
 *   - images are float32 HWC in [0,1] (image.py:80); layers are planar float32 (jpeg.py:263-264);
 *     edge maps are uint8 {0,1}; quantised coefficients are int32 (jpeg.py:501).
 */
#ifndef AEAJ_H
#define AEAJ_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define AEAJ_VERSION 3

#if defined(__GNUC__)
#define AEAJ_API __attribute__((visibility("default")))
#else
#define AEAJ_API
#endif

enum {
    AEAJ_OK = 0,
    AEAJ_EINVAL = -1,      /* bad argument (the Python shim raises ValueError/TypeError before this) */
    AEAJ_ENOMEM = -2,
    AEAJ_ENOCUDA = -3,     /* no usable sm_100 device: there is NO CPU fallback */
    AEAJ_ECAPACITY = -4,   /* a caller-provided output buffer was too small */
    AEAJ_ENOTCONVERGED = -5
};

/* colour spaces: keys of COLOR_SPACE_SETTINGS (jpeg.py:62-147) + XYZ (conversion.py:65-70) */
enum {
    AEAJ_YCBCR = 0, AEAJ_YCOCG = 1, AEAJ_YCOCG_R = 2, AEAJ_OKLAB = 3,
    AEAJ_ICACB = 4, AEAJ_ICTCP = 5, AEAJ_JZAZBZ = 6, AEAJ_XYZ = 7
};

typedef struct aeaj_handle aeaj_handle;
typedef struct aeaj_plan aeaj_plan;

AEAJ_API const char* aeaj_last_error(void);
AEAJ_API int aeaj_version(void);

/* one handle per (device, stream user). Uploads DCT matrices and colour constants. */
AEAJ_API int aeaj_create(int device, aeaj_handle** out);
AEAJ_API int aeaj_destroy(aeaj_handle* h);

/* Colour constants that the reference derives with numpy at import time (np.linalg.inv of float32
 * matrices: oklab.py:35,47; icacb.py:149,159; ictcp.py:149,159; jzazbz.py:196,206) and the
 * 256-entry sRGB->linear table evaluated with the host libm exactly as common.py:34-60 does.
 * fwd1/fwd2/inv1/inv2: 3x3 row-major float32 for `space`; srgb_lut: 256 float32 or NULL. */
AEAJ_API int aeaj_set_color_tables(aeaj_handle* h, int space, const float* fwd1_host, const float* fwd2_host,
                          const float* inv1_host, const float* inv2_host, const float* mid_host,
                          const float* scale_host);
/* The transfer functions of the non-linear spaces (PQ: common.py:94-159, sRGB: common.py:62-92, OKLAB: oklab.py:73,94) raise to
 * fixed powers in float64.  on = 1 (default): table + polynomial evaluation with a carried error bound, and the exact float64
 * path for every pixel whose float32 rounding the bound cannot guarantee -- bit-identical results, several times faster.
 * on = 0: the exact path for every pixel (what the tests compare the fast path with). */
AEAJ_API int aeaj_set_fast_transfer(aeaj_handle* h, int on);
AEAJ_API int aeaj_set_srgb_lut(aeaj_handle* h, const float* lut256_host);

/* ---------------------------------------------------------------------------------------------
 * stage entry points (stage-isolated parity; each is the kernel the fused path uses)
 * ------------------------------------------------------------------------------------------- */

/* convert("sRGB", space, x) / convert(space, "sRGB", x)  (conversion.py:95-124); x is (n,3) */
AEAJ_API int aeaj_color_forward(aeaj_handle* h, int space, const float* rgb, float* out, size_t n, void* stream);
AEAJ_API int aeaj_color_inverse(aeaj_handle* h, int space, const float* in, float* rgb, size_t n, void* stream);
/* apply_normalization(space, x, inverse) on one channel (conversion.py:126-157; jpeg.py:387-390,452-455) */
AEAJ_API int aeaj_normalize(aeaj_handle* h, int space, int channel, int inverse, const float* in, float* out,
                   size_t n, void* stream);
/* cv.resize(INTER_AREA) (jpeg.py:336) and cv.resize(INTER_LINEAR) (jpeg.py:352) on one plane */
AEAJ_API int aeaj_downsample_area(aeaj_handle* h, const float* src, int H, int W, float* dst, int dh, int dw, void* stream);
AEAJ_API int aeaj_resize_linear(aeaj_handle* h, const float* src, int sh, int sw, float* dst, int H, int W, void* stream);

/* Device scratch for ANY single-plane stage call below on an (h,w) plane with the given block range
 * (upper bound over all stages; pass min_size = max_size = 0 if no quadtree/DCT call is made).
 * The workspace also holds the call's descriptors: two stage calls in flight at once need two workspaces, not two handles. */
AEAJ_API size_t aeaj_stage_workspace_bytes(int h, int w, int min_size, int max_size);

/* EdgeDetection.canny stages (edge_detection.py:70-86), one (h,w) plane each. */
AEAJ_API int aeaj_cast_u8(aeaj_handle* hd, const float* layer, uint8_t* out, size_t n, void* stream);               /* :70 */
AEAJ_API int aeaj_clahe(aeaj_handle* hd, const uint8_t* src, int h, int w, uint8_t* dst, void* ws, void* stream);   /* :73-74 */
AEAJ_API int aeaj_gauss3(aeaj_handle* hd, const uint8_t* src, int h, int w, uint8_t* dst, void* ws, void* stream);  /* :77 */
AEAJ_API int aeaj_bilateral5(aeaj_handle* hd, const uint8_t* src, int h, int w, uint8_t* dst, void* ws, void* stream); /* :78 */
/* np.percentile(img,10), np.percentile(img,30) (:81-82) -> thr[0], thr[1] as float64 on the device */
AEAJ_API int aeaj_percentile_thresholds(aeaj_handle* hd, const uint8_t* src, int h, int w, double* thr, void* ws, void* stream);
/* cv.Canny(img, lo, hi, apertureSize=3, L2gradient=True) (:85); thr = 2 float64 on the device; edge uint8 {0,1} */
AEAJ_API int aeaj_canny_u8(aeaj_handle* hd, const uint8_t* src, int h, int w, const double* thr, uint8_t* edge,
                  void* ws, void* stream);
/* the whole of EdgeDetection.canny(layer) -> uint8 {0,1} */
AEAJ_API int aeaj_canny(aeaj_handle* hd, const float* layer, int h, int w, uint8_t* edge, void* ws, void* stream);

/* QuadTree(edge, max, min).get_leaves_and_states() (quadtree.py:71-165).
 * edge: uint8 {0,1} (h,w).  leaves: int32 [cap_leaves][4] = x, y, size, coefficient offset (DFS order).
 * states: uint8 [cap_states] in {0 leaf, 1 split, 2 absent} (DFS pre-order).
 * counts: int32[4] on the device = n_leaves, n_states, n_coef, root size. */
AEAJ_API int aeaj_quadtree_caps(int h, int w, int min_size, int max_size, int64_t* cap_leaves, int64_t* cap_states,
                       int64_t* cap_coef, int* root);
AEAJ_API int aeaj_quadtree(aeaj_handle* hd, const uint8_t* edge, int h, int w, int min_size, int max_size,
                  int32_t* leaves, uint8_t* states, int32_t* counts, void* ws, void* stream);

/* normalise + leaf extraction with reflect padding + cv.dct + quantise (jpeg.py:387-404,471,497-504)
 * for the leaves of one layer.  qtab_dev_ptrs_host: HOST array of 9 DEVICE pointers, entry log2(s) is the
 * s*s int32 table quantization_matrix_cache[layer][s] (jpeg.py:228-238), NULL for unused sizes.
 * counts: the device int32[4] written by aeaj_quadtree (no host sync needed in between). */
AEAJ_API int aeaj_dct_quant(aeaj_handle* hd, const float* layer, int h, int w, float mid, float scale,
                   const int32_t* leaves, const int32_t* counts, int min_size, int max_size,
                   const int32_t* const* qtab_dev_ptrs_host, int32_t* coef, void* ws, void* stream);
/* dequantise + cv.idct + merge + crop + denormalise (jpeg.py:508-529,483,410-459) */
AEAJ_API int aeaj_dequant_idct(aeaj_handle* hd, const int32_t* coef, const int32_t* leaves, const int32_t* counts,
                      int min_size, int max_size, const int32_t* const* qtab_dev_ptrs_host, int h, int w,
                      float mid, float scale, float* layer, void* ws, void* stream);

/* ---------------------------------------------------------------------------------------------
 * fused batch path: Jpeg.compress minus _entropy_encode (jpeg.py:262-270) and
 * Jpeg.decompress minus _entropy_decode (jpeg.py:285-297) for `batch` images of one shape.
 * ------------------------------------------------------------------------------------------- */
typedef struct {
    int batch, height, width, space, block_min, block_max;
    int layer_h[3], layer_w[3], root[3];
    int64_t cap_leaves[3];   /* per image, per layer */
    int64_t cap_states[3];
    int64_t cap_coef[3];
    int64_t workspace_bytes; /* device scratch the caller must provide to encode/decode */
} aeaj_plan_info;

AEAJ_API int aeaj_plan_create(aeaj_handle* h, int batch, int height, int width, int space, int block_min,
                     int block_max, aeaj_plan** out);
AEAJ_API int aeaj_plan_destroy(aeaj_plan* p);
AEAJ_API int aeaj_plan_get_info(const aeaj_plan* p, aeaj_plan_info* info);
/* quantisation tables computed on the host exactly as jpeg.py:688-724 does (Python math.log, int()):
 * for table t in {0 luma, 1 chroma} and each size class s = block_min..block_max the s*s int32
 * entries, concatenated in ascending size order: [luma sizes...][chroma sizes...]. */
AEAJ_API int aeaj_plan_set_qtables(aeaj_plan* p, const int32_t* tables_host, size_t n_entries, void* stream);

typedef struct {
    const float* rgb;        /* [batch][H][W][3] in [0,1]; may be NULL when rgb_u8 is given */
    int32_t* coef[3];        /* [batch][cap_coef[l]]  leaf order, row-major blocks */
    int32_t* leaves[3];      /* [batch][cap_leaves[l]][4] x,y,size,coef offset */
    uint8_t* states[3];      /* [batch][cap_states[l]] */
    int32_t* counts;         /* [batch][3][4] n_leaves, n_states, n_coef, root */
    float* tap_layers[3];    /* optional [batch][h_l][w_l]: downsampled un-normalised layers */
    uint8_t* tap_edges[3];   /* optional [batch][h_l][w_l]: edge maps {0,1} */
    int32_t* status;         /* device int32[64]: [0] hysteresis tile re-visits, [1] hysteresis converged (1 = ok),
                                [2] a tensor-core DCT kernel gave up on a barrier wait (0 = ok), rest diagnostics */
    uint8_t* packed_states[3]; /* optional [batch][(cap_states[l]+3)/4]: the state stream packed 2 bits per state,
                                  MSB first, zero padded -- the bytes _entropy_encode writes (jpeg.py:563-571) */
    const uint8_t* rgb_u8;   /* alternative input (used when rgb == NULL): 8-bit pixels [batch][H][W][3], converted on the
                                device as Image.load does, imread(path).astype(float32) / 255.0 (image.py:84) -- a quarter
                                of the bytes over PCIe / HBM for the same result */
} aeaj_encode_io;

typedef struct {
    const int32_t* coef[3];
    const int32_t* leaves[3];
    const int32_t* counts;   /* [batch][3][4] (only n_leaves is read) */
    float* rgb;              /* [batch][H][W][3]; may be NULL when only rgb_u8 is wanted */
    float* tap_layers[3];    /* optional [batch][h_l][w_l]: merged + denormalised layers */
    uint8_t* rgb_u8;         /* optional [batch][H][W][3]: Image.get_uint8() / Image.save(), (data * 255).astype(uint8)
                                (image.py:112,127), written by the same kernel */
    int32_t* status;         /* optional device int32[64]: [2] tensor-core IDCT barrier timeout (0 = ok), [3] number of leaves
                                that were skipped because they do not fit the plan (bad size / position / offset; 0 = ok) */
} aeaj_decode_io;

AEAJ_API int aeaj_encode(aeaj_plan* p, const aeaj_encode_io* io, void* workspace, void* stream);
AEAJ_API int aeaj_decode(aeaj_plan* p, const aeaj_decode_io* io, void* workspace, void* stream);

/* Scaled decode: the image at 1/scale of its size, scale in {1, 2, 4, 8} -- previews and thumbnails without decoding, moving
 * and shrinking every pixel (libjpeg's scale_num / scale_denom, PIL's draft()).  The output is ceil(H/scale) x ceil(W/scale).
 * With m = min(scale, block_min), each leaf (x, y, s) decodes to (s/m) x (s/m) samples of a 1/m layer from the top-left
 * t x t (t = s/m) of its dequantised coefficients Y: (1/m) C_t^T Y C_t / scale_l + mid_l, C_t the orthonormal t-point DCT (the
 * 1/m keeps each leaf's mean); where scale > block_min, each sample of the 1/scale layer is the mean of the in-bounds samples
 * of its leaf-aligned (scale/m) x (scale/m) group.  The layers then go through aeaj_decode's upsample + inverse colour kernel.
 * There is no reference counterpart: the reference always decodes at full size (jpeg.py:274-297).
 * aeaj_decode_scaled_geometry: the output size, the final layer sizes and the bytes of the caller-owned device scratch the call
 * needs (separate from the plan workspace; 0 for scale 1).  aeaj_decode_scaled: io->rgb / io->rgb_u8 [batch][out_h][out_w][3];
 * io->tap_layers[l] (optional): the final scaled layers [batch][layer_h[l]][layer_w[l]]; io->status as in aeaj_decode.
 * scale 1 runs aeaj_decode's schedule (scratch may be NULL).  AEAJ_EINVAL for another scale, a plan with peers, or NULL buffers.
 * Asynchronous on `stream`, no host sync; after the first call on a plan, steady-state calls issue no host-to-device copy and
 * can be captured in a CUDA graph. */
AEAJ_API int aeaj_decode_scaled_geometry(const aeaj_plan* p, int scale, int* out_h, int* out_w, int layer_h[3], int layer_w[3],
                                         int64_t* scratch_bytes);
AEAJ_API int aeaj_decode_scaled(aeaj_plan* p, const aeaj_decode_io* io, int scale, void* workspace, void* scratch, void* stream);

/* ---------------------------------------------------------------------------------------------
 * halo-split of ONE large image over several GPUs of one node (SURVEY 8e, config C4) into `bands` row bands: band b is the
 * full-resolution rows [b*H/bands, (b+1)*H/bands).  H must be a multiple of `bands`; with more than one band the plan holds
 * one image and every band boundary is a multiple of max(128, block_max) rows in every layer, so that no leaf, filter tile
 * or chroma cell straddles two bands.
 * One process per GPU; the ranks share their plan workspaces through CUDA IPC and the kernels read the few rows they need
 * from the neighbour GPU directly over NVLink -- no collective library on the data path.
 *   aeaj_peer_alloc / aeaj_peer_export: allocate the workspace (and a 64-byte-per-rank flag array) as exportable device
 *   memory and produce its 64-byte IPC handle; aeaj_peer_open / aeaj_peer_close: map / unmap another rank's allocation.
 *   aeaj_plan_set_peers: rank, world (<= 8) and, per rank, the address of its workspace and of its flag array as mapped in
 *   THIS process (own entries: the local allocations).
 *   aeaj_encode_halo / aeaj_decode_halo: one rank's whole schedule in one call, on `stream`.  With peers (world > 1) `bands`
 *   must equal world, `workspace` must be the shared allocation, and the call runs band `rank`: the CLAHE / percentile kernels
 *   sum the per-rank partial histograms, the stencil kernels read the halo rows outside the band from the neighbours'
 *   workspaces, device-side barriers order each rank's writes before the others' reads, and two gathers copy the other bands'
 *   rows of the strong / weak bitmaps (hysteresis runs on the whole image on every rank) and of the quadtree block totals.
 *   Every rank ends with its band's leaves / states / coefficients at their global positions of the streams.  Without peers
 *   the call runs every band in turn on this GPU, through the same schedule, and ends with the whole image's result.
 * Every rank of a split must make the same sequence of calls (each one issues the same barriers).
 * ------------------------------------------------------------------------------------------- */
AEAJ_API int aeaj_peer_alloc(size_t bytes, void** ptr);
AEAJ_API int aeaj_peer_free(void* ptr);
AEAJ_API int aeaj_peer_export(void* ptr, void* handle64_host);
AEAJ_API int aeaj_peer_open(const void* handle64_host, void** ptr);
AEAJ_API int aeaj_peer_close(void* ptr);
AEAJ_API int aeaj_plan_set_peers(aeaj_plan* p, int rank, int world, void* const* peer_workspaces_host, void* const* peer_flags_host);
AEAJ_API int aeaj_encode_halo(aeaj_plan* p, const aeaj_encode_io* io, void* workspace, void* stream, int bands);
AEAJ_API int aeaj_decode_halo(aeaj_plan* p, const aeaj_decode_io* io, void* workspace, void* stream, int bands);

/* ---------------------------------------------------------------------------------------------
 * host-side helpers for the entropy-coding side (plain CPU code, no device work):
 * the 2-bit state stream (jpeg.py:563-571) and its inverse (jpeg.py:768-800 + 428-448).
 * ------------------------------------------------------------------------------------------- */
/* states (0 leaf, 1 split, 2 absent; DFS pre-order) -> leaves_host[n][4] = x, y, size, coef offset.
 * The stream is untrusted input: AEAJ_EINVAL if `root` is not the root size of an (h, w) layer, if a leaf lies outside
 * the layer or outside [block_min, block_max] (pass 0, 0 to skip the range check), or if a node is split below size 2. */
AEAJ_API int aeaj_states_to_leaves_host(const uint8_t* states_host, int n_states, int root, int h, int w,
                               int block_min, int block_max, int32_t* leaves_host, int* n_leaves, int64_t* n_coef);
/* 2 bits per state, MSB first, zero padded; packed_host holds ceil(n_states/4) bytes */
AEAJ_API int aeaj_pack_states_host(const uint8_t* states_host, int n_states, uint8_t* packed_host);

/* ---------------------------------------------------------------------------------------------
 * Packed coefficient streams for the trip to the host-side entropy coder and back (jpeg.py:573-590, 655-672): once the
 * hot path is on the GPU, two thirds of the PCIe bytes of an encode + decode are int32 coefficients, most of them zero.
 * Lossless packed form of one plane's stream of n coefficients (either block layout):
 *     mask: uint32[ceil(n/32)], bit i of word j set <=> coefficient 32 j + i is non-zero;  vals: int16[nnz], the
 *     non-zero coefficients in stream order (|c| <= 127 * block size <= 32512 for normalised samples).
 * counts: int32 [batch][3][4] on the device = nnz, n_coef, overflow flag (a value did not fit int16: move that plane as
 * int32 instead), number of mask words.  aeaj_pack_coefficients reads the n_coef of aeaj_encode's `counts`;
 * aeaj_unpack_coefficients reads them from in->counts.  Both are asynchronous on `stream` and use the plan workspace.
 * The *_host functions are the CPU counterparts for the container writer / reader (no device work).
 * ------------------------------------------------------------------------------------------- */
typedef struct {
    uint32_t* mask[3];       /* [batch][cap_coef[l] / 32 + 1] */
    int16_t* vals[3];        /* [batch][cap_coef[l]] */
    int32_t* counts;         /* [batch][3][4] */
} aeaj_packed_io;
AEAJ_API int aeaj_pack_coefficients(aeaj_plan* p, const int32_t* const* coef3, const int32_t* counts, const aeaj_packed_io* out,
                                    void* workspace, void* stream);
AEAJ_API int aeaj_unpack_coefficients(aeaj_plan* p, const aeaj_packed_io* in, int32_t* const* coef3, void* workspace, void* stream);
AEAJ_API int aeaj_pack_coefficients_host(const int32_t* coef_host, int64_t n_coef, uint32_t* mask_host, int16_t* vals_host,
                                         int64_t* nnz, int* overflow);
AEAJ_API int aeaj_unpack_coefficients_host(const uint32_t* mask_host, const int16_t* vals_host, int64_t n_coef, int64_t nnz,
                                           int32_t* coef_host);

/* One frame's worth of variable-length streams (packed coefficients, leaves, states of the three layers) in ONE transfer:
 * copies n byte ranges device -> device in a single launch, so that the caller can gather everything the host-side entropy
 * coder needs (jpeg.py:531-597) into one contiguous arena, move it with one cudaMemcpy, and scatter what comes back
 * (jpeg.py:599-674) the same way -- instead of ~27 small copies per frame, each paying its own DMA set-up.
 * Any alignment and size; ranges whose two ends are 16-byte (4-byte) aligned are moved with 128-bit (32-bit) accesses.
 * Up to 64 ranges travel in the kernel's parameters (no upload of any kind); beyond that the table is staged through
 * `table_dev`, caller-owned device scratch of at least n * sizeof(aeaj_segment) bytes (may be NULL for n <= 64). */
typedef struct { const void* src; void* dst; int64_t bytes; } aeaj_segment;
AEAJ_API int aeaj_copy_segments(const aeaj_segment* segs_host, int n, void* table_dev, void* stream);

/* ---------------------------------------------------------------------------------------------
 * Device entropy coder: deflate of the coefficient streams on the GPU, an alternative to the host's zlib level 9
 * (jpeg.py:590) that moves only the compressed bytes over PCIe.  Each plane's stream of n_coef int32 (little-endian, as
 * stored; with aeaj_plan_set_stream_layout(1) the bytes _entropy_encode hands to zlib) becomes ONE complete zlib stream
 * (RFC 1950) that any inflate reads.  The bytes are not zlib's: the stream is coded in independent 64 KiB chunks, each one
 * deflate block (dynamic, fixed or stored, whichever is smallest) ending byte-aligned.  They depend only on the input bytes
 * -- not on the batch, the position in it, the stream or the GPU.  n_coef is read from counts[b][l][2] on the device (no
 * host sync).  aeaj_deflate_caps: per-layer capacity of one plane's output (every input fits) and the bytes of the
 * caller-owned device scratch the call needs (separate from the plan workspace).  Asynchronous on `stream`; after the first
 * call on a plan, steady-state calls issue no host-to-device copy and can be captured in a CUDA graph.
 * ------------------------------------------------------------------------------------------- */
typedef struct {
    uint8_t* out[3];         /* [batch][cap_out[l]]: one zlib stream per plane */
    int32_t* lengths;        /* [batch][3] bytes written, on the device (0 if a stream did not fit) */
    int32_t* status;         /* optional device int32[4]: [0] planes whose stream did not fit (0 = ok) */
} aeaj_deflate_io;
AEAJ_API int aeaj_deflate_caps(const aeaj_plan* p, int64_t* cap_out3, int64_t* scratch_bytes);
AEAJ_API int aeaj_deflate_coefficients(aeaj_plan* p, const int32_t* const* coef3, const int32_t* counts,
                                       const aeaj_deflate_io* io, void* scratch, void* stream);

/* ---------------------------------------------------------------------------------------------
 * Device entropy decoder: inflate of the coefficient streams on the GPU, the counterpart of aeaj_deflate_coefficients and
 * an alternative to the host's zlib.decompress (jpeg.py:659): only the compressed bytes cross PCIe, and the coefficients
 * land in the buffers aeaj_decode reads.  Plane (b, l)'s zlib stream is in[offsets[b][l], + lengths[b][l]) (device arrays;
 * ranges outside [0, in_bytes) are clamped to it; streams must not overlap); it must inflate to exactly
 * 4 * counts[b][l][2] bytes (counts as aeaj_decode takes them, read on the device), written to coef[l] + b * cap_coef[l].
 * Any zlib stream is read (RFC 1950 / 1951, as zlib's inflate accepts it: the reference's level-9 files included); it is
 * decoded in parallel at its sync points (the non-final empty stored blocks of Z_SYNC_FLUSH / Z_FULL_FLUSH, which the
 * device coder writes after every 64 KiB chunk) and one warp per plane where it has none.  Per plane on the device:
 *   status: 0 ok, 1 header (FCHECK, method, window), 2 preset dictionary, 3 block type, 4 stored length, 5 code lengths,
 *           6 invalid symbol, 7 distance too far back, 8 truncated, 9 Adler-32 mismatch, 10 length (the stream does not
 *           inflate to exactly the expected bytes; decoding stops at the expected length);
 *   out_bytes: bytes written (never beyond the expected length or the buffer);  segments: parts decoded independently.
 * Nothing outside a stream's bytes is read and nothing outside [0, expected) of its plane is written, whatever the input.
 * aeaj_inflate_scratch_bytes: the caller-owned device scratch for inputs of up to in_bytes (separate from the workspace).
 * Asynchronous on `stream`, no host sync; after the first call on a plan, steady-state calls issue no host-to-device copy
 * and can be captured in a CUDA graph.
 * ------------------------------------------------------------------------------------------- */
typedef struct {
    const uint8_t* in;       /* the zlib streams */
    const int64_t* offsets;  /* [batch][3] */
    const int64_t* lengths;  /* [batch][3] */
    int32_t* coef[3];        /* [batch][cap_coef[l]] */
    int32_t* status;         /* [batch][3] */
    int64_t* out_bytes;      /* [batch][3] */
    int32_t* segments;       /* [batch][3] */
} aeaj_inflate_io;
AEAJ_API int aeaj_inflate_scratch_bytes(const aeaj_plan* p, int64_t in_bytes, int64_t* scratch_bytes);
AEAJ_API int aeaj_inflate_coefficients(aeaj_plan* p, const aeaj_inflate_io* io, const int32_t* counts, int64_t in_bytes,
                                       void* scratch, void* stream);

/* Stream layout (SURVEY 8f rank 1).  zigzag = 0 (default): each block of the coefficient stream is row-major,
 * i.e. the reference's img_quantized blocks.  zigzag = 1: each block is stored in the zigzag order of
 * Jpeg._zigzag_ordering (jpeg.py:726-766), i.e. the stream is byte-for-byte what _entropy_encode hands to zlib
 * (jpeg.py:579-590); aeaj_decode then expects that layout. */
AEAJ_API int aeaj_plan_set_stream_layout(aeaj_plan* p, int zigzag);

/* Tensor-core path for the DCT (cv.dct, jpeg.py:471) and IDCT (cv.idct, jpeg.py:483) of the size classes 16 .. 128: tcgen05
 * kind::tf32, error-compensated 3xTF32, FP32 accumulation in tensor memory; (128/S)^2 leaves of size S form one 128 x 128 tile
 * that is transformed with block-diagonal DCT matrices.  `mask` bit k selects the tensor-core kernel for class 16 << k (default
 * 0xa: 32 and 128, the classes where it is faster; 0 = the FP32-FMA kernels everywhere -- same parity class, the quantiser is exact in both, DESIGN.md 4).
 * aeaj_tensor_dct_status: timed_out must point to int[32]; [0] is set if a tensor-core kernel ever gave up on a barrier
 * wait (also reported in the status words of aeaj_encode / aeaj_decode).  Synchronises the device. */
AEAJ_API int aeaj_plan_set_tensor_dct(aeaj_plan* p, int mask);
AEAJ_API int aeaj_tensor_dct_status(aeaj_handle* h, int* timed_out);

/* number of kernel launches issued by the last aeaj_encode / aeaj_decode on this plan */
AEAJ_API int aeaj_plan_last_launches(const aeaj_plan* p);

/* optional per-stage timing with CUDA events on the launching stream (measurement only).
 * aeaj_plan_read_timing returns the stage durations (ms) of the LAST encode or decode call;
 * names_buf receives newline-separated stage names.  It synchronises that call's last event. */
AEAJ_API int aeaj_plan_enable_timing(aeaj_plan* p, int enable);
AEAJ_API int aeaj_plan_read_timing(aeaj_plan* p, char* names_buf, size_t names_cap, float* ms, int cap, int* n);

#ifdef __cplusplus
}
#endif
#endif /* AEAJ_H */
