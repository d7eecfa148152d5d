// deflate_core.h -- the chunked deflate coder of the .ajpg coefficient streams, shared by the device kernels (deflate.cu)
// and the host build that defines it (tests/native/deflate_check.cpp).  Everything here is __host__ __device__ and
// sequential; the device runs the prev-table build and the match search warp-parallel (deflate.cu), with the same result.
//
// A plane's byte stream (the int32 coefficients, little-endian) is cut into independent chunks of DF_CHUNK bytes.  No
// match reaches before its chunk's start, so chunks are coded in parallel.  Every chunk is ONE deflate block (dynamic
// Huffman, or fixed codes, or stored -- whichever is smallest), followed, unless it is the plane's last chunk, by an empty
// stored block as Z_SYNC_FLUSH writes it: each chunk's output is then a whole number of bytes and the chunks concatenate.
// The zlib stream (RFC 1950) is the 2-byte header, the chunks, and the Adler-32 of the input, combined from per-chunk
// partial sums.
//
// Match candidates are positional, so the parse does not depend on how the search is parallelised: at position p they are
// the DF_CANDIDATES most recent earlier positions q of the chunk whose 4 bytes at q hash like the 4 bytes at p, and with
// p - q <= 32768.  The longest match wins; of equal lengths, the most recent.  The parse is one-step lazy: a match shorter
// than DF_LAZY_BELOW is emitted only if the match at p + 1 is not longer.
#pragma once
#include <stdint.h>

#ifdef __CUDACC__
#define DF_HD __host__ __device__ __forceinline__
#else
#define DF_HD inline
#endif

constexpr int DF_CHUNK = 65536;            // input bytes per chunk (the last chunk of a plane may be shorter)
constexpr int DF_CHUNK_BOUND = DF_CHUNK + 16;   // output bytes of one chunk at most: stored blocks (2 x 5 header bytes) + flush (5)
constexpr int DF_HASH_BITS = 13;
constexpr int DF_CANDIDATES = 4;
constexpr int DF_LAZY_BELOW = 64;
constexpr int DF_WINDOW = 32768;
constexpr int DF_MAX_MATCH = 258;
constexpr int DF_MIN_MATCH = 4;            // candidates share a 4-byte hash; shorter matches are not searched for

// ------------------------------------------------------------------------------------------------------------------------
// tokens: uint16 per literal (the byte value), two uint16 per match: 0x8000 | (length - 3), then distance - 1
// ------------------------------------------------------------------------------------------------------------------------
DF_HD int df_ilog2(uint32_t v) {
#ifdef __CUDA_ARCH__
    return 31 - __clz(v);
#else
    return 31 - __builtin_clz(v);
#endif
}
// length - 3 (0..255) -> lit/len symbol index - 257 (0..28), extra bits
DF_HD int df_len_sym(int L, int& ebits) {
    if (L < 8) { ebits = 0; return L; }
    if (L == 255) { ebits = 0; return 28; }
    ebits = df_ilog2((uint32_t)L) - 2;
    return 4 * ebits + ((L >> ebits) & 3) + 4;
}
// distance - 1 (0..32767) -> distance symbol (0..29), extra bits
DF_HD int df_dist_sym(int D, int& ebits) {
    if (D < 4) { ebits = 0; return D; }
    ebits = df_ilog2((uint32_t)D) - 1;
    return 2 * ebits + ((D >> ebits) & 1) + 2;
}

DF_HD uint32_t df_hash(const uint8_t* d, int i) {
    const uint32_t v = (uint32_t)d[i] | ((uint32_t)d[i + 1] << 8) | ((uint32_t)d[i + 2] << 16) | ((uint32_t)d[i + 3] << 24);
    return (v * 2654435761u) >> (32 - DF_HASH_BITS);
}

// prev[i] = i - (latest earlier position with the same hash), 0 if none; defined for i <= n - 4, 0 beyond.
// head: 1 << DF_HASH_BITS entries of scratch.  (The device builds the same table warp-serially, deflate.cu.)
inline void df_build_prev_seq(const uint8_t* d, int n, uint16_t* prev, uint16_t* head) {
    for (int h = 0; h < (1 << DF_HASH_BITS); h++) head[h] = 0;
    for (int i = 0; i < n; i++) {
        if (i + 4 > n) { prev[i] = 0; continue; }
        const uint32_t h = df_hash(d, i);
        prev[i] = head[h] ? (uint16_t)(i - (head[h] - 1)) : 0;
        head[h] = (uint16_t)(i + 1);
    }
}

DF_HD int df_match_len(const uint8_t* d, int a, int b, int maxlen) {
    int k = 0;
    while (k < maxlen && d[a + k] == d[b + k]) k++;
    return k;
}

// the candidate positions of p in chain order (most recent first); returns how many
DF_HD int df_candidates(const uint16_t* prev, int p, int n, int* cand) {
    int k = 0;
    if (p + DF_MIN_MATCH > n) return 0;
    int c = p;
    for (; k < DF_CANDIDATES; k++) {
        const int pd = prev[c];
        if (pd == 0 || (p - (c - pd)) > DF_WINDOW) break;
        c -= pd;
        cand[k] = c;
    }
    return k;
}

// best match at p: length (0 if below DF_MIN_MATCH), distance in `dist`
inline int df_best_seq(const uint8_t* d, const uint16_t* prev, int p, int n, int& dist) {
    int cand[DF_CANDIDATES];
    const int nc = df_candidates(prev, p, n, cand);
    const int maxlen = n - p < DF_MAX_MATCH ? n - p : DF_MAX_MATCH;
    int best = 0;
    for (int k = 0; k < nc; k++) {
        const int l = df_match_len(d, cand[k], p, maxlen);
        if (l > best) { best = l; dist = p - cand[k]; if (l == maxlen) break; }
    }
    return best >= DF_MIN_MATCH ? best : 0;
}

// one-step lazy parse of d[0, n) into tokens; `best(p, dist)` returns the best match at p.  Returns the token count.
template <class Best, class Put>
DF_HD int df_parse(const uint8_t* d, int n, Best best, Put put) {
    int p = 0, ntok = 0, L = 0, D = 0;
    bool have = false;
    while (p < n) {
        if (!have) L = best(p, D);
        have = false;
        if (L == 0) { put(ntok++, (uint16_t)d[p]); p++; continue; }
        if (L < DF_LAZY_BELOW && p + 1 < n) {
            int D2 = 0;
            const int L2 = best(p + 1, D2);
            if (L2 > L) { put(ntok++, (uint16_t)d[p]); p++; L = L2; D = D2; have = true; continue; }
        }
        put(ntok++, (uint16_t)(0x8000 | (L - 3)));
        put(ntok++, (uint16_t)(D - 1));
        p += L;
    }
    return ntok;
}

// ------------------------------------------------------------------------------------------------------------------------
// Huffman code lengths, limited to `maxbits`
// ------------------------------------------------------------------------------------------------------------------------
constexpr int DF_NLIT = 286, DF_NDIST = 30, DF_NCL = 19;

// code lengths of an optimal prefix code for weights a[0..n-1] sorted ascending, in place (Moffat & Katajainen 1995):
// a[i] becomes the length of the i-th lightest symbol.  n >= 2.
DF_HD void df_min_redundancy(uint32_t* a, int n) {
    int root = 0, leaf = 2, next;
    a[0] += a[1];
    for (next = 1; next < n - 1; next++) {
        if (leaf >= n || a[root] < a[leaf]) { a[next] = a[root]; a[root++] = (uint32_t)next; }
        else a[next] = a[leaf++];
        if (leaf >= n || (root < next && a[root] < a[leaf])) { a[next] += a[root]; a[root++] = (uint32_t)next; }
        else a[next] += a[leaf++];
    }
    a[n - 2] = 0;
    for (next = n - 3; next >= 0; next--) a[next] = a[a[next]] + 1;
    int avbl = 1, used = 0, dpth = 0;
    root = n - 2; next = n - 1;
    while (avbl > 0) {
        while (root >= 0 && (int)a[root] == dpth) { used++; root--; }
        while (avbl > used) { a[next--] = (uint32_t)dpth; avbl--; }
        avbl = 2 * used; dpth++; used = 0;
    }
}

// lens[s] for freq[s] (0 for unused symbols).  One used symbol gets length 1; two or more get a complete code whose
// lengths do not exceed maxbits.  key / w: scratch of nsym entries.  Returns the number of used symbols.
DF_HD int df_huff_lengths(const uint32_t* freq, int nsym, int maxbits, uint8_t* lens, uint32_t* key, uint32_t* w) {
    int m = 0;
    for (int s = 0; s < nsym; s++) {
        lens[s] = 0;
        if (freq[s]) key[m++] = (freq[s] << 9) | (uint32_t)s;          // freq <= 65537: unique keys, ordered by (freq, symbol)
    }
    if (m == 0) return 0;
    if (m == 1) { lens[key[0] & 511] = 1; return 1; }
    for (int gap = m / 2; gap > 0; gap /= 2)                            // Shell sort; the keys are unique, so the order is too
        for (int i = gap; i < m; i++) {
            const uint32_t v = key[i];
            int j = i;
            for (; j >= gap && key[j - gap] > v; j -= gap) key[j] = key[j - gap];
            key[j] = v;
        }
    for (int i = 0; i < m; i++) w[i] = key[i] >> 9;
    df_min_redundancy(w, m);
    int count[33];
    for (int l = 0; l < 33; l++) count[l] = 0;
    for (int i = 0; i < m; i++) count[w[i] < 32 ? w[i] : 32]++;
    // length limiting: fold the lengths above maxbits into maxbits, then lengthen the deepest shorter codes until the
    // Kraft sum is exactly 1 again (the lightest symbols keep the longest codes)
    for (int l = maxbits + 1; l < 33; l++) { count[maxbits] += count[l]; count[l] = 0; }
    uint32_t total = 0;
    for (int l = maxbits; l > 0; l--) total += (uint32_t)count[l] << (maxbits - l);
    while (total != (1u << maxbits)) {
        count[maxbits]--;
        for (int l = maxbits - 1; l > 0; l--)
            if (count[l]) { count[l]--; count[l + 1] += 2; break; }
        total--;
    }
    int i = 0;                                                          // lightest symbols first: longest codes
    for (int l = maxbits; l > 0; l--)
        for (int k = 0; k < count[l]; k++) lens[key[i++] & 511] = (uint8_t)l;
    return m;
}

// canonical codes (RFC 1951 3.2.2), bit-reversed for the LSB-first bit writer
DF_HD void df_codes(const uint8_t* lens, int nsym, uint16_t* codes) {
    int bl_count[16], next_code[16];
    for (int l = 0; l < 16; l++) bl_count[l] = 0;
    for (int s = 0; s < nsym; s++) bl_count[lens[s]]++;
    bl_count[0] = 0;
    int code = 0;
    for (int l = 1; l < 16; l++) { code = (code + bl_count[l - 1]) << 1; next_code[l] = code; }
    for (int s = 0; s < nsym; s++) {
        const int l = lens[s];
        if (!l) { codes[s] = 0; continue; }
        uint32_t c = (uint32_t)next_code[l]++, r = 0;
        for (int k = 0; k < l; k++) { r = (r << 1) | (c & 1); c >>= 1; }
        codes[s] = (uint16_t)r;
    }
}

// ------------------------------------------------------------------------------------------------------------------------
// block coder
// ------------------------------------------------------------------------------------------------------------------------
struct DfBits {
    uint8_t* out;
    int pos;
    uint64_t acc;
    int nb;
    DF_HD void put(uint32_t v, int n) {
        acc |= (uint64_t)v << nb; nb += n;
        while (nb >= 8) { out[pos++] = (uint8_t)acc; acc >>= 8; nb -= 8; }
    }
    DF_HD void align() { if (nb) put(0, 8 - nb); }
};

// scratch of one block coder (device: shared memory of the chunk's CTA)
struct DfWork {
    uint32_t freq_l[DF_NLIT], freq_d[DF_NDIST], freq_c[DF_NCL];
    uint32_t key[DF_NLIT], w[DF_NLIT];
    uint8_t len_l[288], len_d[DF_NDIST], len_c[DF_NCL];       // 288: the fixed code counts symbols 286 and 287 too
    uint16_t code_l[288], code_d[DF_NDIST], code_c[DF_NCL];
    uint16_t rle[DF_NLIT + DF_NDIST];              // code-length symbol | repeat value << 5
    int nrle;
};

DF_HD int df_fixed_len(int s) { return s < 144 ? 8 : (s < 256 ? 9 : (s < 280 ? 7 : 8)); }

// symbols 16 / 17 / 18 for runs of one code length (RFC 1951 3.2.7)
DF_HD void df_rle(const uint8_t* lens, int n, DfWork* w) {
    int i = 0;
    while (i < n) {
        const int v = lens[i];
        int r = 1;
        while (i + r < n && lens[i + r] == v) r++;
        i += r;
        if (v == 0) {
            while (r >= 11) { const int k = r < 138 ? r : 138; w->rle[w->nrle++] = (uint16_t)(18 | ((k - 11) << 5)); r -= k; }
            if (r >= 3) { w->rle[w->nrle++] = (uint16_t)(17 | ((r - 3) << 5)); r = 0; }
        } else {
            w->rle[w->nrle++] = (uint16_t)v; r--;
            while (r >= 3) { const int k = r < 6 ? r : 6; w->rle[w->nrle++] = (uint16_t)(16 | ((k - 3) << 5)); r -= k; }
        }
        while (r-- > 0) w->rle[w->nrle++] = (uint16_t)v;
    }
}

DF_HD void df_count(const uint16_t* tok, int ntok, DfWork* w) {
    for (int s = 0; s < DF_NLIT; s++) w->freq_l[s] = 0;
    for (int s = 0; s < DF_NDIST; s++) w->freq_d[s] = 0;
    for (int t = 0; t < ntok; t++) {
        const uint16_t v = tok[t];
        if (v & 0x8000) {
            int e;
            w->freq_l[257 + df_len_sym(v & 0xff, e)]++;
            w->freq_d[df_dist_sym(tok[++t], e)]++;
        } else w->freq_l[v]++;
    }
    w->freq_l[256] = 1;
}

DF_HD void df_put_tokens(DfBits& bw, const uint16_t* tok, int ntok, const uint16_t* cl, const uint8_t* ll,
                         const uint16_t* cd, const uint8_t* ld) {
    for (int t = 0; t < ntok; t++) {
        const uint16_t v = tok[t];
        if (v & 0x8000) {
            int e;
            const int L = v & 0xff, ls = df_len_sym(L, e);
            bw.put(cl[257 + ls], ll[257 + ls]);
            if (e) bw.put((uint32_t)L & ((1u << e) - 1), e);
            const int D = tok[++t], ds = df_dist_sym(D, e);
            bw.put(cd[ds], ld[ds]);
            if (e) bw.put((uint32_t)D & ((1u << e) - 1), e);
        } else bw.put(cl[v], ll[v]);
    }
    bw.put(cl[256], ll[256]);
}

// codes d[0, n) (tokens `tok`) as one block into `out`; last: the plane's final chunk.  Returns the bytes written
// (at most n + 15, DF_CHUNK_BOUND).
DF_HD int df_encode_chunk(const uint8_t* d, int n, const uint16_t* tok, int ntok, bool last, uint8_t* out, DfWork* w) {
    df_count(tok, ntok, w);
    df_huff_lengths(w->freq_l, DF_NLIT, 15, w->len_l, w->key, w->w);
    if (df_huff_lengths(w->freq_d, DF_NDIST, 15, w->len_d, w->key, w->w) == 0) w->len_d[0] = 1;   // one declared distance code
    int hlit = DF_NLIT, hdist = DF_NDIST;
    while (hlit > 257 && !w->len_l[hlit - 1]) hlit--;
    while (hdist > 1 && !w->len_d[hdist - 1]) hdist--;
    w->nrle = 0;
    df_rle(w->len_l, hlit, w);
    df_rle(w->len_d, hdist, w);
    for (int s = 0; s < DF_NCL; s++) w->freq_c[s] = 0;
    for (int i = 0; i < w->nrle; i++) w->freq_c[w->rle[i] & 31]++;
    if (df_huff_lengths(w->freq_c, DF_NCL, 7, w->len_c, w->key, w->w) == 1)   // inflate wants a complete code-length code
        w->len_c[w->len_c[0] ? 1 : 0] = 1;
    const uint8_t ORDER[DF_NCL] = {16, 17, 18, 0, 8, 7, 9, 6, 10, 5, 11, 4, 12, 3, 13, 2, 14, 1, 15};
    int hclen = DF_NCL;
    while (hclen > 4 && !w->len_c[ORDER[hclen - 1]]) hclen--;

    // sizes in bits of the three block types
    uint64_t extra = 0, dyn = 3 + 5 + 5 + 4 + 3 * (uint64_t)hclen, fix = 3;
    for (int s = 0; s < DF_NLIT; s++) {
        const uint64_t f = w->freq_l[s];
        if (!f) continue;
        dyn += f * w->len_l[s]; fix += f * (uint64_t)df_fixed_len(s);
        if (s >= 265 && s < 285) extra += f * (uint64_t)((s - 261) / 4);
    }
    for (int s = 0; s < DF_NDIST; s++) {
        const uint64_t f = w->freq_d[s];
        if (!f) continue;
        dyn += f * w->len_d[s]; fix += f * 5;
        if (s >= 4) extra += f * (uint64_t)((s - 2) / 2);
    }
    for (int i = 0; i < w->nrle; i++) {
        const int s = w->rle[i] & 31;
        dyn += w->len_c[s] + (s == 16 ? 2 : (s == 17 ? 3 : (s == 18 ? 7 : 0)));
    }
    dyn += extra; fix += extra;
    const int nstored = n ? (n + 65534) / 65535 : 1;
    const uint64_t stored = 8 * ((uint64_t)n + 5 * (uint64_t)nstored);

    DfBits bw{out, 0, 0, 0};
    const uint32_t fin = last ? 1u : 0u;
    if (stored < dyn && stored < fix) {
        for (int b = 0; b < nstored; b++) {
            const int o = b * 65535, len = (n - o) < 65535 ? (n - o) : 65535;
            bw.put((b == nstored - 1) ? fin : 0u, 3);
            bw.align();
            bw.put((uint32_t)len, 16); bw.put((uint32_t)len ^ 0xffffu, 16);
            for (int i = 0; i < len; i++) bw.out[bw.pos++] = d[o + i];
        }
    } else if (fix <= dyn) {
        for (int s = 0; s < 288; s++) w->len_l[s] = (uint8_t)df_fixed_len(s);
        for (int s = 0; s < DF_NDIST; s++) w->len_d[s] = 5;
        df_codes(w->len_l, 288, w->code_l);
        df_codes(w->len_d, DF_NDIST, w->code_d);
        bw.put(fin | (1u << 1), 3);
        df_put_tokens(bw, tok, ntok, w->code_l, w->len_l, w->code_d, w->len_d);
    } else {
        df_codes(w->len_l, DF_NLIT, w->code_l);
        df_codes(w->len_d, DF_NDIST, w->code_d);
        df_codes(w->len_c, DF_NCL, w->code_c);
        bw.put(fin | (2u << 1), 3);
        bw.put((uint32_t)(hlit - 257), 5); bw.put((uint32_t)(hdist - 1), 5); bw.put((uint32_t)(hclen - 4), 4);
        for (int i = 0; i < hclen; i++) bw.put(w->len_c[ORDER[i]], 3);
        for (int i = 0; i < w->nrle; i++) {
            const int s = w->rle[i] & 31, r = w->rle[i] >> 5;
            bw.put(w->code_c[s], w->len_c[s]);
            if (s == 16) bw.put((uint32_t)r, 2); else if (s == 17) bw.put((uint32_t)r, 3); else if (s == 18) bw.put((uint32_t)r, 7);
        }
        df_put_tokens(bw, tok, ntok, w->code_l, w->len_l, w->code_d, w->len_d);
    }
    if (!last) { bw.put(0, 3); bw.align(); bw.put(0, 16); bw.put(0xffff, 16); }   // Z_SYNC_FLUSH: empty stored block
    bw.align();
    return bw.pos;
}

// ------------------------------------------------------------------------------------------------------------------------
// Adler-32 from per-chunk partial sums
// ------------------------------------------------------------------------------------------------------------------------
constexpr uint32_t DF_ADLER_MOD = 65521;
// Adler-32 of d[0, n) from s1 = sum d[i] and s2 = sum (n - i) d[i]
DF_HD uint32_t df_adler_from_sums(uint64_t s1, uint64_t s2, int64_t n) {
    const uint32_t a = (uint32_t)((1 + s1) % DF_ADLER_MOD), b = (uint32_t)(((uint64_t)n + s2) % DF_ADLER_MOD);
    return (b << 16) | a;
}
// Adler-32 of x followed by y, len2 = length of y
DF_HD uint32_t df_adler_combine(uint32_t x, uint32_t y, int64_t len2) {
    const uint64_t a1 = x & 0xffff, b1 = x >> 16, a2 = y & 0xffff, b2 = y >> 16, r = (uint64_t)len2 % DF_ADLER_MOD;
    const uint64_t a = (a1 + a2 + DF_ADLER_MOD - 1) % DF_ADLER_MOD;
    const uint64_t b = (b1 + b2 + r * ((a1 + DF_ADLER_MOD - 1) % DF_ADLER_MOD)) % DF_ADLER_MOD;
    return (uint32_t)((b << 16) | a);
}

DF_HD int df_chunks(int64_t nbytes) { return nbytes <= 0 ? 1 : (int)((nbytes + DF_CHUNK - 1) / DF_CHUNK); }
// bytes of a plane's zlib stream at most: header, chunks, trailer
DF_HD int64_t df_stream_bound(int64_t nbytes) { return 2 + (int64_t)df_chunks(nbytes) * DF_CHUNK_BOUND + 4; }

#ifndef __CUDACC__
// the whole zlib stream of d[0, n), sequentially: the definition the device output is checked against
inline int64_t df_deflate_seq(const uint8_t* d, int64_t n, uint8_t* out, uint16_t* prev, uint16_t* head, uint16_t* tok, DfWork* w) {
    out[0] = 0x78; out[1] = 0x9c;
    int64_t pos = 2;
    uint32_t adler = 1;
    const int nch = df_chunks(n);
    for (int c = 0; c < nch; c++) {
        const uint8_t* x = d + (int64_t)c * DF_CHUNK;
        const int m = (int)((n - (int64_t)c * DF_CHUNK) < DF_CHUNK ? (n - (int64_t)c * DF_CHUNK) : DF_CHUNK);
        df_build_prev_seq(x, m, prev, head);
        const int ntok = df_parse(x, m, [&](int p, int& dist) { return df_best_seq(x, prev, p, m, dist); },
                                  [&](int i, uint16_t v) { tok[i] = v; });
        pos += df_encode_chunk(x, m, tok, ntok, c == nch - 1, out + pos, w);
        uint64_t s1 = 0, s2 = 0;
        for (int i = 0; i < m; i++) { s1 += x[i]; s2 += (uint64_t)(m - i) * x[i]; }
        adler = df_adler_combine(adler, df_adler_from_sums(s1, s2, m), m);
    }
    for (int k = 3; k >= 0; k--) out[pos++] = (uint8_t)(adler >> (8 * k));
    return pos;
}
#endif
