// inflate_core.h -- the zlib (RFC 1950 / 1951) decoder of the .ajpg coefficient streams, shared by the device kernels
// (inflate.cu) and the host build that defines it (tests/native/inflate_check.cpp).  Everything here is sequential; the
// device runs it one warp per segment, every lane decoding the same bits and the lanes sharing the output writes.
//
// A stream is accepted if and only if zlib's inflate (as Python's zlib.decompress runs it) accepts it, and then gives the
// same bytes: the header checks, the table rules of zlib's inflate_table (over-subscribed and incomplete code sets, with
// the one-code exception), the order in which inflate.c asks for bits and rejects, distances up to the output produced so
// far (zlib without INFLATE_STRICT), and bytes after the Adler-32 trailer ignored.  The decoder reads nothing outside
// its stream's bytes (bits past the end are truncation), writes nothing outside [0, limit) of its output, and every loop
// is bounded by the input bits and the output length.
//
// Segments: a non-final empty stored block (Z_SYNC_FLUSH / Z_FULL_FLUSH; the device coder ends every 64 KiB chunk with
// one) leaves the stream byte-aligned right after the bytes 00 00 FF FF.  Every such position is a candidate segment start.
// The speculative pass decodes each candidate's blocks up to the next such block without writing (if_decode with an
// IfCount sink), recording where it ends, how much it produces and how far back before its own start it copies from.
// if_chain walks the true chain from the stream's first block and merges a segment that copies from before its start into
// the segments it needs; the output pass decodes each merged segment at its output offset; if_finish combines the
// Adler-32 and sets the status.  if_inflate_seq runs the same steps one after another: the definition the device matches.
#pragma once
#include <stdint.h>
#include "deflate_core.h"

// statuses of one stream (aeaj_inflate_coefficients, include/aeaj.h)
enum {
    IF_OK = 0,
    IF_HEADER = 1,          // CMF / FLG: bad FCHECK, method != 8 or CINFO > 7
    IF_NEED_DICT = 2,       // FDICT set
    IF_BLOCK_TYPE = 3,      // BTYPE 11
    IF_STORED_LEN = 4,      // LEN != ~NLEN
    IF_CODE_LENGTHS = 5,    // too many codes, bad code-length code, bad repeat, over-subscribed / incomplete, no end-of-block
    IF_BAD_SYMBOL = 6,      // a code that is not in the set, lit/len 286 / 287, distance 30 / 31
    IF_DIST_FAR = 7,        // a distance beyond the output produced so far
    IF_TRUNCATED = 8,       // the stream ends before its trailer
    IF_CHECK = 9,           // Adler-32 mismatch
    IF_LENGTH = 10,         // the stream does not inflate to exactly the expected number of bytes
    // segment ends (internal)
    IF_SYNC = 16,           // after a non-final empty stored block
    IF_FINAL = 17,          // after the final block
};

constexpr int IF_ENOUGH_L = 852, IF_ENOUGH_D = 592;   // zlib's ENOUGH_LENS / ENOUGH_DISTS for root bits 9 / 6
constexpr int IF_ROOT_L = 9, IF_ROOT_D = 6, IF_ROOT_C = 7;

// table entry: bits [0, 8) code length (in the sub-table: beyond the root bits), [8, 12) kind, [12, 16) extra bits or
// sub-table bits, [16, 32) value: literal, length / distance base, or sub-table offset
enum { IF_K_LIT = 0, IF_K_LEN = 1, IF_K_EOB = 2, IF_K_BAD = 3, IF_K_LINK = 4, IF_K_DIST = 5 };
DF_HD uint32_t if_entry(int bits, int kind, int extra, int val) {
    return (uint32_t)bits | ((uint32_t)kind << 8) | ((uint32_t)extra << 12) | ((uint32_t)val << 16);
}
#define IF_BITS(e) ((int)((e) & 0xff))
#define IF_KIND(e) ((int)(((e) >> 8) & 0xf))
#define IF_EXTRA(e) ((int)(((e) >> 12) & 0xf))
#define IF_VAL(e) ((int)((e) >> 16))

// what symbol s of a table of `type` decodes to (type: 0 code lengths, 1 literal/length, 2 distance)
DF_HD uint32_t if_sym_entry(int type, int s, int bits) {
    if (type == 0) return if_entry(bits, IF_K_LIT, 0, s);
    if (type == 1) {
        if (s < 256) return if_entry(bits, IF_K_LIT, 0, s);
        if (s == 256) return if_entry(bits, IF_K_EOB, 0, 0);
        const int i = s - 257;
        if (i >= 29) return if_entry(bits, IF_K_BAD, 0, 0);               // 286, 287 (fixed code only)
        if (i < 8) return if_entry(bits, IF_K_LEN, 0, 3 + i);
        if (i == 28) return if_entry(bits, IF_K_LEN, 0, 258);
        const int e = (i - 4) >> 2;
        return if_entry(bits, IF_K_LEN, e, ((4 + (i & 3)) << e) + 3);
    }
    if (s >= 30) return if_entry(bits, IF_K_BAD, 0, 0);                   // 30, 31 (fixed code only)
    if (s < 4) return if_entry(bits, IF_K_DIST, 0, 1 + s);
    const int e = (s - 2) >> 1;
    return if_entry(bits, IF_K_DIST, e, ((2 + (s & 1)) << e) + 1);
}

// zlib's inflate_table: root table of `root` bits (lowered to the longest code, raised to the shortest), sub-tables for
// longer codes.  Returns 0, or -1 for an over-subscribed or incomplete set (one 1-bit code is allowed except for the
// code-length code).  No codes at all: a 1-bit table that decodes to an invalid code (the code-length code: to length 0,
// as zlib's CODELENS loop reads that entry).
DF_HD int if_build(const uint8_t* lens, int n, int type, uint32_t* table, int cap, int root_req, int* root_out, int16_t* work) {
    int16_t* count = work;                                           // [16], then rem [16]
    for (int l = 0; l < 16; l++) count[l] = 0;
    for (int s = 0; s < n; s++) count[lens[s]]++;
    int max = 15;
    while (max >= 1 && count[max] == 0) max--;
    if (max == 0) {
        table[0] = table[1] = type == 0 ? if_entry(1, IF_K_LIT, 0, 0) : if_entry(1, IF_K_BAD, 0, 0);
        *root_out = 1;
        return 0;
    }
    int min = 1;
    while (min < max && count[min] == 0) min++;
    int root = root_req > max ? max : root_req;
    if (root < min) root = min;
    int left = 1;
    for (int l = 1; l <= 15; l++) {
        left <<= 1;
        left -= count[l];
        if (left < 0) return -1;
    }
    if (left > 0 && (type == 0 || max != 1)) return -1;
    const int size = 1 << root;
    if (size > cap) return -1;
    for (int i = 0; i < size; i++) table[i] = if_entry(1, IF_K_BAD, 0, 0);   // only the 1-bit incomplete code keeps one
    int16_t* rem = work + 16;
    for (int l = 0; l < 16; l++) rem[l] = count[l];
    int code = 0, next = size, cur_prefix = -1, cur_sub = 0, cur_bits = 0;
    for (int len = 1; len <= max; len++) {
        for (int s = 0; s < n; s++) {
            if (lens[s] != len) continue;
            uint32_t r = 0;                                          // canonical code, bit-reversed
            for (int k = 0, c = code; k < len; k++, c >>= 1) r = (r << 1) | (uint32_t)(c & 1);
            code++;
            rem[len]--;
            if (len <= root) {
                const uint32_t e = if_sym_entry(type, s, len);
                for (int i = (int)r; i < size; i += 1 << len) table[i] = e;
                continue;
            }
            const int prefix = (int)(r & (uint32_t)(size - 1));
            if (prefix != cur_prefix) {                               // new sub-table: as many bits as its codes need
                int curr = len - root, lf = 1 << curr;
                while (curr + root < max) {
                    lf -= rem[curr + root] + (curr + root == len ? 1 : 0);
                    if (lf <= 0) break;
                    curr++;
                    lf <<= 1;
                }
                if (next + (1 << curr) > cap) return -1;
                cur_prefix = prefix; cur_sub = next; cur_bits = curr;
                table[prefix] = if_entry(root, IF_K_LINK, curr, next);
                next += 1 << curr;
            }
            const uint32_t e = if_sym_entry(type, s, len - root);
            for (int i = (int)(r >> root); i < (1 << cur_bits); i += 1 << (len - root)) table[cur_sub + i] = e;
        }
        code <<= 1;
    }
    *root_out = root;
    return 0;
}

// LSB-first bit reader over in[0, end): hold holds nb bits; refill() leaves nb >= 57 unless the input is exhausted, so
// "fewer than n bits after refill()" is "the stream ends inside these n bits"
struct IfBits {
    const uint8_t* in;
    int64_t pos, end;
    uint64_t hold;
    int nb;
    DF_HD void refill() { while (nb <= 56 && pos < end) { hold |= (uint64_t)in[pos++] << nb; nb += 8; } }
    DF_HD bool need(int n) { refill(); return nb >= n; }
    DF_HD uint32_t peek(int n) const { return (uint32_t)(hold & ((1ull << n) - 1)); }
    DF_HD void drop(int n) { hold >>= n; nb -= n; }
    DF_HD int64_t byte_pos() const { return pos - (nb >> 3); }      // with nb a multiple of 8
};

// one symbol: 0, or IF_TRUNCATED when the code does not end inside the stream
DF_HD int if_decode_sym(IfBits& br, const uint32_t* tab, int root, uint32_t& e) {
    br.refill();
    e = tab[br.peek(root)];
    int b = IF_BITS(e);
    if (IF_KIND(e) == IF_K_LINK) {
        const uint32_t s = tab[IF_VAL(e) + (int)(br.peek(root + IF_EXTRA(e)) >> root)];
        b = root + IF_BITS(s);
        e = s;
    }
    if (b > br.nb) return IF_TRUNCATED;
    br.drop(b);
    return 0;
}

// the order of the code-length code lengths (RFC 1951 3.2.7), 5 bits per entry (no array: it would live in local memory)
DF_HD int if_order(int i) {
    return i < 12 ? (int)((0x22caa324e804a30ull >> (5 * i)) & 31) : (int)((0x3c2e1346cull >> (5 * (i - 12))) & 31);
}

// per-decoder tables (device: shared memory of the decoding warp)
struct IfTables {
    uint32_t lit[IF_ENOUGH_L];        // also the code-length code while a dynamic header is read
    uint32_t dist[IF_ENOUGH_D];
    uint8_t lens[320];
    int16_t work[32];                 // if_build's counts
};

// a table build: on the device one lane builds, the warp waits and takes its result
template <class Sink>
DF_HD int if_build_by(Sink& sk, const uint8_t* lens, int n, int type, uint32_t* table, int cap, int root_req, int* root, IfTables* T) {
    int rc = 0, r = 0;
    if (sk.leader()) rc = if_build(lens, n, type, table, cap, root_req, &r, T->work);
    sk.sync();
    *root = sk.bcast(r);
    return sk.bcast(rc);
}

// Decodes blocks of in[0, len) from byte position `start` into `sink`.  stop_at: -2 stops at the first non-final empty
// stored block, -1 never stops there, >= 0 stops there when it ends at byte stop_at.  Returns IF_SYNC / IF_FINAL with
// *end the byte position after that block (byte-aligned), or an error status.  Sink: pos (bytes produced), lit(b),
// copy(dist, n), raw(src, n) returning 0 or a status, sync() after the tables are written.
template <class Sink>
DF_HD int if_decode(const uint8_t* in, int64_t len, int64_t start, int64_t stop_at, IfTables* T, Sink& sk, int64_t* end) {
    IfBits br{in, start, len, 0, 0};
    int lroot = 0, droot = 0;
    for (;;) {
        if (!br.need(3)) return IF_TRUNCATED;
        const int last = (int)br.peek(1), type = (int)(br.peek(3) >> 1);
        br.drop(3);
        if (type == 0) {                                                // stored
            br.drop(br.nb & 7);
            if (!br.need(32)) return IF_TRUNCATED;
            const uint32_t n = br.peek(16), nn = (uint32_t)(br.hold >> 16) & 0xffff;
            if (n != (nn ^ 0xffffu)) return IF_STORED_LEN;
            br.drop(32);
            const int64_t p = br.byte_pos();
            br.pos = p; br.hold = 0; br.nb = 0;
            if (n == 0 && !last && (stop_at == -2 || stop_at == p)) { *end = p; return IF_SYNC; }
            if ((int64_t)n > len - p) {
                const int rc = sk.raw(in + p, (int)(len - p));
                return rc ? rc : IF_TRUNCATED;
            }
            const int rc = sk.raw(in + p, (int)n);
            if (rc) return rc;
            br.pos = p + n;
        } else if (type == 3) {
            return IF_BLOCK_TYPE;
        } else {
            if (type == 1) {                                            // fixed codes
                if (sk.leader()) for (int s = 0; s < 288; s++) T->lens[s] = (uint8_t)df_fixed_len(s);
                if_build_by(sk, T->lens, 288, 1, T->lit, IF_ENOUGH_L, IF_ROOT_L, &lroot, T);
                sk.sync();
                if (sk.leader()) for (int s = 0; s < 32; s++) T->lens[s] = 5;
                if_build_by(sk, T->lens, 32, 2, T->dist, IF_ENOUGH_D, IF_ROOT_D, &droot, T);
            } else {                                                    // dynamic: inflate.c TABLE / LENLENS / CODELENS
                if (!br.need(14)) return IF_TRUNCATED;
                const int nlen = (int)br.peek(5) + 257, ndist = (int)(br.peek(10) >> 5) + 1, ncode = (int)(br.peek(14) >> 10) + 4;
                br.drop(14);
                if (nlen > 286 || ndist > 30) return IF_CODE_LENGTHS;
                for (int i = 0; i < 19; i++) T->lens[i] = 0;
                for (int i = 0; i < ncode; i++) {
                    if (!br.need(3)) return IF_TRUNCATED;
                    T->lens[if_order(i)] = (uint8_t)br.peek(3);
                    br.drop(3);
                }
                int croot = 0;
                if (if_build_by(sk, T->lens, 19, 0, T->lit, IF_ENOUGH_L, IF_ROOT_C, &croot, T)) return IF_CODE_LENGTHS;
                sk.sync();
                const int total = nlen + ndist;
                int have = 0;
                while (have < total) {
                    uint32_t e;
                    if (if_decode_sym(br, T->lit, croot, e)) return IF_TRUNCATED;
                    const int v = IF_VAL(e);
                    if (v < 16) { T->lens[have++] = (uint8_t)v; continue; }
                    int rep, val = 0;
                    if (v == 16) {
                        if (!br.need(2)) return IF_TRUNCATED;
                        if (have == 0) return IF_CODE_LENGTHS;
                        val = T->lens[have - 1];
                        rep = 3 + (int)br.peek(2); br.drop(2);
                    } else if (v == 17) {
                        if (!br.need(3)) return IF_TRUNCATED;
                        rep = 3 + (int)br.peek(3); br.drop(3);
                    } else {
                        if (!br.need(7)) return IF_TRUNCATED;
                        rep = 11 + (int)br.peek(7); br.drop(7);
                    }
                    if (have + rep > total) return IF_CODE_LENGTHS;
                    while (rep--) T->lens[have++] = (uint8_t)val;
                }
                if (T->lens[256] == 0) return IF_CODE_LENGTHS;
                sk.sync();
                if (if_build_by(sk, T->lens, nlen, 1, T->lit, IF_ENOUGH_L, IF_ROOT_L, &lroot, T)) return IF_CODE_LENGTHS;
                if (if_build_by(sk, T->lens + nlen, ndist, 2, T->dist, IF_ENOUGH_D, IF_ROOT_D, &droot, T)) return IF_CODE_LENGTHS;
            }
            sk.sync();
            for (;;) {                                                  // inflate.c LEN / LENEXT / DIST / DISTEXT
                uint32_t e;
                if (if_decode_sym(br, T->lit, lroot, e)) return IF_TRUNCATED;
                const int k = IF_KIND(e);
                if (k == IF_K_LIT) { const int rc = sk.lit((uint8_t)IF_VAL(e)); if (rc) return rc; continue; }
                if (k == IF_K_EOB) break;
                if (k != IF_K_LEN) return IF_BAD_SYMBOL;
                int n = IF_VAL(e);
                if (IF_EXTRA(e)) {
                    if (!br.need(IF_EXTRA(e))) return IF_TRUNCATED;
                    n += (int)br.peek(IF_EXTRA(e)); br.drop(IF_EXTRA(e));
                }
                if (if_decode_sym(br, T->dist, droot, e)) return IF_TRUNCATED;
                if (IF_KIND(e) != IF_K_DIST) return IF_BAD_SYMBOL;
                int d = IF_VAL(e);
                if (IF_EXTRA(e)) {
                    if (!br.need(IF_EXTRA(e))) return IF_TRUNCATED;
                    d += (int)br.peek(IF_EXTRA(e)); br.drop(IF_EXTRA(e));
                }
                const int rc = sk.copy(d, n);
                if (rc) return rc;
            }
        }
        sk.sync();
        if (last) {
            br.drop(br.nb & 7);
            *end = br.byte_pos();
            return IF_FINAL;
        }
    }
}

// speculative sink: counts the output, records how far before the segment's start a copy reaches
struct IfCount {
    int64_t pos, limit;
    int32_t reach;
    DF_HD void sync() {}
    DF_HD bool leader() const { return true; }
    DF_HD int bcast(int v) const { return v; }
    DF_HD int lit(uint8_t) { if (pos >= limit) return IF_LENGTH; pos++; return 0; }
    DF_HD int copy(int d, int n) {
        if (d > pos && d - pos > reach) reach = (int32_t)(d - pos);
        if (n > limit - pos) { pos = limit; return IF_LENGTH; }
        pos += n;
        return 0;
    }
    DF_HD int raw(const uint8_t*, int n) {
        if (n > limit - pos) { pos = limit; return IF_LENGTH; }
        pos += n;
        return 0;
    }
};

// sequential output sink: out[0, limit)
struct IfWrite {
    uint8_t* out;
    int64_t pos, limit;
    void sync() {}
    bool leader() const { return true; }
    int bcast(int v) const { return v; }
    int lit(uint8_t b) { if (pos >= limit) return IF_LENGTH; out[pos++] = b; return 0; }
    int copy(int d, int n) {
        if (d > pos) return IF_DIST_FAR;
        const int m = n > limit - pos ? (int)(limit - pos) : n;
        for (int k = 0; k < m; k++) out[pos + k] = out[pos + k - d];
        pos += m;
        return m < n ? IF_LENGTH : 0;
    }
    int raw(const uint8_t* s, int n) {
        const int m = n > limit - pos ? (int)(limit - pos) : n;
        for (int k = 0; k < m; k++) out[pos + k] = s[k];
        pos += m;
        return m < n ? IF_LENGTH : 0;
    }
};

// zlib header (inflate.c HEAD / DICTID): 0, or the stream's status
DF_HD int if_header(const uint8_t* in, int64_t len) {
    if (len < 2) return IF_TRUNCATED;
    const int cmf = in[0], flg = in[1];
    if (((cmf << 8) | flg) % 31) return IF_HEADER;
    if ((cmf & 15) != 8) return IF_HEADER;
    if ((cmf >> 4) + 8 > 15) return IF_HEADER;
    if (flg & 0x20) return len < 6 ? IF_TRUNCATED : IF_NEED_DICT;
    return 0;
}

// one candidate segment and, for the segments that start a merged segment, what the chain and the output pass add
struct IfSeg {
    int32_t stream, pos;      // the candidate: stream index, byte position in the stream
    int32_t end, status;      // speculative pass: byte position after the segment; IF_SYNC, IF_FINAL or an error
    int64_t olen;             //   bytes it produces
    int32_t reach, head;      //   bytes before its start it copies from; chain: 1 if a merged segment starts here
    int32_t next, prev;       // chain: the next / previous merged segment (index), -1 if none
    int32_t hend, fend;       // chain: byte position where the merged segment ends, -1 = at the stream's end; output: where it did
    int64_t out_off;          // chain: output offset
    int64_t hlen;             // output pass: bytes written
    int32_t hstatus;          //   IF_SYNC, IF_FINAL or an error
    uint32_t hadler;          //   Adler-32 of those bytes
};

// one stream of a batch (device pipeline): its bytes in the input buffer, output limit, header status
struct IfStream {
    int64_t off, len, limit, expected;
    int32_t hdr, pad;
};

DF_HD void if_spec(const uint8_t* in, int64_t len, int64_t limit, IfTables* T, IfSeg& S) {
    IfCount c{0, limit, 0};
    int64_t e = -1;
    S.status = if_decode(in, len, S.pos, -2, T, c, &e);
    S.end = (int32_t)e;
    S.olen = c.pos;
    S.reach = c.reach;
    S.head = 0;
}

// the chain of one stream from its first segment segs[first]; lookup(p) is the index of the candidate at byte p or -1.
// Marks the merged segments (head, out_off, hend, next); a segment that copies from before its start joins the merged
// segment before it, and that one the one before while they together hold fewer bytes than it reaches back.
template <class Lookup>
DF_HD void if_chain(IfSeg* segs, int first, int64_t limit, Lookup lookup) {
    int h = first, s = first;
    segs[h].head = 1; segs[h].prev = -1; segs[h].out_off = 0;
    int64_t cum = 0;
    for (;;) {
        const IfSeg& S = segs[s];
        const int64_t cum_end = cum + S.olen;
        const int nx = (S.status == IF_SYNC && cum_end <= limit) ? lookup(S.end) : -1;
        if (nx < 0) break;                                   // final, error, over length, or no speculative result:
        cum = cum_end;                                       // the last merged segment decodes to the stream's end
        if (segs[nx].reach > 0) {
            while (segs[nx].reach > cum - segs[h].out_off && segs[h].prev >= 0) {
                segs[h].head = 0;
                h = segs[h].prev;
            }
        } else {
            segs[h].hend = S.end; segs[h].next = nx;
            segs[nx].head = 1; segs[nx].prev = h; segs[nx].out_off = cum;
            h = nx;
        }
        s = nx;
    }
    segs[h].hend = -1; segs[h].next = -1;
}

// status, bytes and merged segments of one stream from its output pass
DF_HD int if_finish(const uint8_t* in, int64_t len, int64_t expected, const IfSeg* segs, int first, int64_t* out_bytes, int* nseg) {
    uint32_t adler = 1;
    int64_t total = 0;
    int n = 0;
    for (int h = first; h >= 0; h = segs[h].next) {
        const IfSeg& S = segs[h];
        n++;
        total = S.out_off + S.hlen;
        if (S.hstatus != IF_SYNC && S.hstatus != IF_FINAL) { *out_bytes = total; *nseg = n; return S.hstatus; }
        adler = df_adler_combine(adler, S.hadler, S.hlen);
        if (S.hstatus == IF_FINAL) {
            *out_bytes = total; *nseg = n;
            if (len - S.fend < 4) return IF_TRUNCATED;
            const uint32_t want = ((uint32_t)in[S.fend] << 24) | ((uint32_t)in[S.fend + 1] << 16) | ((uint32_t)in[S.fend + 2] << 8) | in[S.fend + 3];
            if (want != adler) return IF_CHECK;
            return total == expected ? IF_OK : IF_LENGTH;
        }
    }
    *out_bytes = total; *nseg = n;
    return IF_TRUNCATED;                                        // unreachable: the last merged segment decodes to the end
}

#ifndef __CUDACC__
#include <algorithm>
#include <vector>
// the whole pipeline of one stream, sequentially: what aeaj_inflate_coefficients gives, segment count included.
// out: at least min(expected, cap) bytes; writes only there.
inline int if_inflate_seq(const uint8_t* in, int64_t len, uint8_t* out, int64_t expected, int64_t cap, int64_t* out_bytes, int* nseg) {
    *out_bytes = 0; *nseg = 0;
    const int hs = if_header(in, len);
    if (hs) return hs;
    const int64_t limit = expected < cap ? expected : cap;
    std::vector<IfSeg> segs;
    std::vector<int64_t> at;                                    // candidate positions, ascending
    IfSeg s0{};
    s0.pos = 2;
    segs.push_back(s0); at.push_back(2);
    for (int64_t p = 4; p <= len; p++)
        if (in[p - 4] == 0 && in[p - 3] == 0 && in[p - 2] == 0xff && in[p - 1] == 0xff) {
            IfSeg s{};
            s.pos = (int32_t)p;
            segs.push_back(s); at.push_back(p);
        }
    IfTables T;
    for (auto& s : segs) if_spec(in, len, limit, &T, s);
    if_chain(segs.data(), 0, limit, [&](int64_t p) {
        const auto it = std::lower_bound(at.begin() + 1, at.end(), p);
        return it != at.end() && *it == p ? (int)(it - at.begin()) : -1;
    });
    for (auto& s : segs) {
        if (!s.head) continue;
        IfWrite w{out + s.out_off, 0, limit - s.out_off};
        int64_t e = -1;
        s.hstatus = if_decode(in, len, s.pos, s.hend, &T, w, &e);
        s.fend = (int32_t)e;
        s.hlen = w.pos;
        uint64_t s1 = 0, s2 = 0;
        for (int64_t i = 0; i < w.pos; i++) { s1 += w.out[i]; s2 += (uint64_t)((w.pos - i) % DF_ADLER_MOD) * w.out[i]; }
        s.hadler = df_adler_from_sums(s1, s2, w.pos);
    }
    return if_finish(in, len, expected, segs.data(), 0, out_bytes, nseg);
}
#endif
