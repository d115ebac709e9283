// (2d) zstd frames on the device (RFC 8878): the zstd half of the VBZ HDF5 filter, so a fast5 chunk can
// cross PCIe as its file stores it.  Every check libzstd 1.5 makes on a one-shot decode of a single frame
// is made here too, and a frame that fails one gets a non-zero status (WSTR_ZSTD_*).
//
// One warp per frame; persistent warps pull frames longest-first from the staged plan.  The warp walks
// the frame in lockstep: every lane parses the same headers and decodes the same sequences (reads of the
// same address are broadcasts), and the bulk work is split across lanes:
//   - decoding tables (Huffman <= 12 bits, as libzstd accepts; FSE LL/ML <= 9, OF <= 8) in shared memory,
//     Huffman cells filled lane-parallel;
//   - the four Huffman streams of a literal section decoded by lanes 0-3, into the tail of the frame's own
//     output range (which the block's output reaches only after the last literal is consumed);
//   - raw and RLE blocks, literal runs and matches copied lane-parallel in 32-byte steps; a match closer
//     than 32 bytes replicates its period.
// Bitstreams are read exactly as libzstd's BIT_DStream reads them (a 64-bit container refilled from the
// end of the stream towards its start), so over-read streams end as libzstd's do.
#include <limits.h>
#include <stdint.h>

#include "wstr_internal.h"

#define ZHD __host__ __device__ __forceinline__

namespace wstr_zstd {

constexpr int WARPS = 4;                 // warps (frames in flight) per CTA
constexpr int64_t BLOCK_MAX = 1 << 17;   // ZSTD_BLOCKSIZE_MAX
constexpr int HUF_LOG_MAX = 12;          // HUF_TABLELOG_MAX of libzstd (RFC 8878 allows 11)
constexpr int MIN_CBLOCK = 2;            // MIN_CBLOCK_SIZE: literal header + 1 byte

struct Frame {
    int64_t in_off, in_bytes, out_off, out_bytes;
    int64_t index;                       // the caller's frame number: where its status goes
};

struct SeqCell {                         // one FSE state of a sequence table
    uint32_t base;                       // baseline of the code's value
    uint16_t next;                       // new-state baseline
    uint8_t nbits, extra;                // state bits, the code's extra bits
};
struct WtCell {                          // one FSE state of the Huffman-weight table
    uint16_t next;
    uint8_t sym, nbits;
};

struct Smem {
    uint16_t huf[1 << HUF_LOG_MAX];      // symbol | nbBits << 8
    SeqCell ll[512], ml[512], of[256];
    WtCell wt[64];
    int16_t norm[256];
    uint16_t fse_next[256];              // next state of each symbol while a table is built
    uint8_t weights[256];
    int32_t ok4[4];                      // per Huffman stream: decoded and consumed exactly
};

struct Lanes {
    int id, n;
    ZHD void sync() const {
#ifdef __CUDA_ARCH__
        __syncwarp();
#endif
    }
};

ZHD int highbit(uint32_t v) {   // v > 0
#ifdef __CUDA_ARCH__
    return 31 - __clz(v);
#else
    return 31 - __builtin_clz(v);
#endif
}

// 8 little-endian bytes at p through the two aligned words that hold them (the frame's span is 16-byte
// aligned and padded, and p + 8 never passes a stream's end, so neither word leaves the padded span)
ZHD uint64_t ld64(const uint8_t *p) {
    const uintptr_t a = reinterpret_cast<uintptr_t>(p);
    const uint64_t *w = reinterpret_cast<const uint64_t *>(a & ~(uintptr_t)7);
    const int r = (int)(a & 7) * 8;
    const uint64_t lo = w[0];
    return r ? (lo >> r) | (w[1] << (64 - r)) : lo;
}
ZHD uint32_t ld16(const uint8_t *p) { return p[0] | (uint32_t)p[1] << 8; }
ZHD uint32_t ld24(const uint8_t *p) { return ld16(p) | (uint32_t)p[2] << 16; }
ZHD uint32_t ld32(const uint8_t *p) { return ld24(p) | (uint32_t)p[3] << 24; }

// ---- backward bitstream, libzstd's BIT_DStream_t on a 64-bit container ---------------------------------
enum { BIT_UNFINISHED = 0, BIT_END_OF_BUFFER = 1, BIT_COMPLETED = 2, BIT_OVERFLOW = 3 };
struct BitD {
    uint64_t c;
    uint32_t consumed;
    const uint8_t *ptr, *start, *limit;
};
ZHD bool bit_init(BitD &b, const uint8_t *src, int64_t n) {
    if (n < 1) return false;
    b.start = src;
    b.limit = src + 8;
    const uint32_t last = src[n - 1];
    if (last == 0) return false;             // no end mark
    if (n >= 8) {
        b.ptr = src + n - 8;
        b.c = ld64(b.ptr);
        b.consumed = 8 - highbit(last);
    } else {
        b.ptr = src;
        b.c = 0;
        for (int i = 0; i < n; ++i) b.c |= (uint64_t)src[i] << (8 * i);
        b.consumed = 8 - highbit(last) + (uint32_t)(8 - n) * 8;
    }
    return true;
}
ZHD uint64_t bit_look(const BitD &b, int n) { return (b.c << (b.consumed & 63)) >> 1 >> ((63 - n) & 63); }
ZHD uint64_t bit_read(BitD &b, int n) {
    const uint64_t v = bit_look(b, n);
    b.consumed += n;
    return v;
}
ZHD int bit_reload(BitD &b) {
    if (b.consumed > 64) return BIT_OVERFLOW;
    if (b.ptr >= b.limit) {
        b.ptr -= b.consumed >> 3;
        b.consumed &= 7;
        b.c = ld64(b.ptr);
        return BIT_UNFINISHED;
    }
    if (b.ptr == b.start) return b.consumed < 64 ? BIT_END_OF_BUFFER : BIT_COMPLETED;
    int64_t nb = b.consumed >> 3;
    int res = BIT_UNFINISHED;
    if (b.ptr - nb < b.start) {
        nb = b.ptr - b.start;
        res = BIT_END_OF_BUFFER;
    }
    b.ptr -= nb;
    b.consumed -= (uint32_t)nb * 8;
    b.c = ld64(b.ptr);
    return res;
}
ZHD bool bit_end(const BitD &b) { return b.ptr == b.start && b.consumed == 64; }

// ---- FSE --------------------------------------------------------------------------------------------------
// FSE_readNCount of libzstd, to the letter: *max_sv in = largest symbol allowed, out = last symbol read.
// Returns the header's size, or -1.  norm[] is written by the writer lane only.
ZHD int64_t read_ncount_8(int16_t *norm, bool writer, int *max_sv, int *table_log, const uint8_t *ip0,
                          const uint8_t *iend) {
    const uint8_t *ip = ip0;
    const int max_sv1 = *max_sv + 1;
    if (writer)
        for (int s = 0; s < max_sv1; ++s) norm[s] = 0;
    uint32_t bits = ld32(ip);
    int nb = (int)(bits & 0xF) + 5;
    if (nb > 15) return -1;
    bits >>= 4;
    int bit_count = 4;
    *table_log = nb;
    int remaining = (1 << nb) + 1;
    int threshold = 1 << nb;
    nb++;
    int charnum = 0;
    bool previous0 = false;
    for (;;) {
        if (previous0) {
            int repeats;
            {
                const uint32_t x = ~bits | 0x80000000u;
#ifdef __CUDA_ARCH__
                repeats = (__ffs((int)x) - 1) >> 1;
#else
                repeats = __builtin_ctz(x) >> 1;
#endif
            }
            while (repeats >= 12) {
                charnum += 3 * 12;
                if (ip <= iend - 7) {
                    ip += 3;
                } else {
                    bit_count -= (int)(8 * (iend - 7 - ip));
                    bit_count &= 31;
                    ip = iend - 4;
                }
                bits = ld32(ip) >> bit_count;
                const uint32_t x = ~bits | 0x80000000u;
#ifdef __CUDA_ARCH__
                repeats = (__ffs((int)x) - 1) >> 1;
#else
                repeats = __builtin_ctz(x) >> 1;
#endif
            }
            charnum += 3 * repeats;
            bits >>= 2 * repeats;
            bit_count += 2 * repeats;
            charnum += bits & 3;
            bit_count += 2;
            if (charnum >= max_sv1) break;
            if (ip <= iend - 7 || ip + (bit_count >> 3) <= iend - 4) {
                ip += bit_count >> 3;
                bit_count &= 7;
            } else {
                bit_count -= (int)(8 * (iend - 4 - ip));
                bit_count &= 31;
                ip = iend - 4;
            }
            bits = ld32(ip) >> bit_count;
        }
        {
            const int mx = (2 * threshold - 1) - remaining;
            int count;
            if ((int)(bits & (uint32_t)(threshold - 1)) < mx) {
                count = (int)(bits & (uint32_t)(threshold - 1));
                bit_count += nb - 1;
            } else {
                count = (int)(bits & (uint32_t)(2 * threshold - 1));
                if (count >= threshold) count -= mx;
                bit_count += nb;
            }
            count--;
            if (count >= 0) remaining -= count;
            else remaining += count;
            if (writer) norm[charnum] = (int16_t)count;
            charnum++;
            previous0 = count == 0;
            if (remaining < threshold) {
                if (remaining <= 1) break;
                nb = highbit((uint32_t)remaining) + 1;
                threshold = 1 << (nb - 1);
            }
            if (charnum >= max_sv1) break;
            if (ip <= iend - 7 || ip + (bit_count >> 3) <= iend - 4) {
                ip += bit_count >> 3;
                bit_count &= 7;
            } else {
                bit_count -= (int)(8 * (iend - 4 - ip));
                bit_count &= 31;
                ip = iend - 4;
            }
            bits = ld32(ip) >> bit_count;
        }
    }
    if (remaining != 1) return -1;
    if (charnum > max_sv1) return -1;
    if (bit_count > 32) return -1;
    *max_sv = charnum - 1;
    ip += (bit_count + 7) >> 3;
    return ip - ip0;
}

// the same on a header shorter than 8 bytes: libzstd parses a zero-padded 8-byte copy
ZHD int64_t read_ncount(int16_t *norm, bool writer, int *max_sv, int *table_log, const uint8_t *ip,
                        int64_t n) {
    if (n >= 8) return read_ncount_8(norm, writer, max_sv, table_log, ip, ip + n);
    uint8_t buf[8] = {0, 0, 0, 0, 0, 0, 0, 0};
    for (int i = 0; i < n; ++i) buf[i] = ip[i];
    const int64_t r = read_ncount_8(norm, writer, max_sv, table_log, buf, buf + 8);
    if (r < 0 || r > n) return -1;
    return r;
}

// symbol spread of FSE_buildDTable / ZSTD_buildFSETable: sym_of[u] for every cell; returns high_threshold
template <class Put>
ZHD void fse_spread(const int16_t *norm, int max_sv, int table_log, Put put) {
    const int size = 1 << table_log, mask = size - 1;
    int high = size - 1;
    for (int s = 0; s <= max_sv; ++s)
        if (norm[s] == -1) put(high--, s);
    const int step = (size >> 1) + (size >> 3) + 3;
    int pos = 0;
    for (int s = 0; s <= max_sv; ++s)
        for (int i = 0; i < norm[s]; ++i) {
            put(pos, s);
            do pos = (pos + step) & mask;
            while (pos > high);
        }
}

// code tables of RFC 8878 section 3.1.1.3.2.1, as arithmetic (no local arrays)
ZHD int ll_bits(int c) {
    return c < 16 ? 0 : c < 20 ? 1 : c < 22 ? 2 : c < 24 ? 3 : c == 24 ? 4 : c - 19;
}
ZHD uint32_t ll_base(int c) {
    if (c < 16) return (uint32_t)c;
    if (c < 20) return 16u + 2u * (uint32_t)(c - 16);
    if (c < 25) return c == 20 ? 24u : c == 21 ? 28u : c == 22 ? 32u : c == 23 ? 40u : 48u;
    return 1u << (c - 19);
}
ZHD int ml_bits(int c) {
    return c < 32 ? 0 : c < 36 ? 1 : c < 38 ? 2 : c < 40 ? 3 : c < 42 ? 4 : c == 42 ? 5 : c - 36;
}
ZHD uint32_t ml_base(int c) {
    if (c < 32) return (uint32_t)c + 3u;
    if (c < 36) return 35u + 2u * (uint32_t)(c - 32);
    if (c < 43) return c == 36 ? 43u : c == 37 ? 47u : c == 38 ? 51u : c == 39 ? 59u : c == 40 ? 67u : c == 41 ? 83u : 99u;
    return (1u << (c - 36)) + 3u;
}
// offset codes: value (1 << c) + bits, minus 3 past the repeat codes (libzstd's OF_base)
ZHD uint32_t of_base(int c) { return c < 2 ? (uint32_t)c : (1u << c) - 3u; }

enum { T_LL = 0, T_OF = 1, T_ML = 2 };
ZHD void code_of(int kind, int s, uint32_t *base, int *extra) {
    if (kind == T_LL) {
        *base = ll_base(s);
        *extra = ll_bits(s);
    } else if (kind == T_ML) {
        *base = ml_base(s);
        *extra = ml_bits(s);
    } else {
        *base = of_base(s);
        *extra = s;
    }
}

// the predefined distributions (RFC 8878 3.1.1.3.2.2), symbol by symbol
ZHD int16_t default_count(int kind, int i) {
    if (kind == T_LL) return i == 0 ? 4 : i == 1 ? 3 : i < 13 ? 2 : i < 16 ? 1 : i < 25 ? 2 : i == 25 ? 3 : i == 26 ? 2 : i < 32 ? 1 : -1;
    if (kind == T_ML) return i == 0 ? 1 : i == 1 ? 4 : i == 2 ? 3 : i < 9 ? 2 : i < 46 ? 1 : -1;
    return i < 6 ? 1 : i < 9 ? 2 : i < 24 ? 1 : -1;
}
ZHD int default_norm(int kind, int16_t *norm) {
    const int n = kind == T_LL ? 36 : kind == T_ML ? 53 : 29;
    for (int i = 0; i < n; ++i) norm[i] = default_count(kind, i);
    return n - 1;
}

// decoding table of a sequence code from its normalised counts (writer lane only)
ZHD void build_seq_table(SeqCell *tab, int kind, const int16_t *norm, int max_sv, int table_log, uint16_t *next) {
    const int size = 1 << table_log;
    fse_spread(norm, max_sv, table_log, [&](int u, int s) { tab[u].extra = (uint8_t)s; });
    for (int s = 0; s <= max_sv; ++s) next[s] = norm[s] == -1 ? 1 : (uint16_t)norm[s];
    for (int u = 0; u < size; ++u) {
        const int s = tab[u].extra;
        const uint32_t x = next[s]++;
        const int nb = table_log - highbit(x);
        uint32_t base;
        int extra;
        code_of(kind, s, &base, &extra);
        tab[u].base = base;
        tab[u].extra = (uint8_t)extra;
        tab[u].nbits = (uint8_t)nb;
        tab[u].next = (uint16_t)((x << nb) - size);
    }
}

// ---- the frame decoder ------------------------------------------------------------------------------------
struct Dec {
    const uint8_t *in;       // frame start
    int64_t in_n;
    uint8_t *out;            // frame output
    int64_t cap;             // = Frame_Content_Size
    Smem *sm;
    Lanes L;
    // entropy carried from block to block
    int huf_log;             // 0: no Huffman table yet
    int seq_log[3];          // table log of LL / OF / ML (the tables live in sm)
    bool fse_entropy;        // a block has decoded sequences (repeat mode allowed)
    uint32_t rep[3];
};

// lane-parallel forward copy that is safe for dst < src overlapping (read, sync, write per step)
ZHD void copy_fwd(const Lanes &L, uint8_t *dst, const uint8_t *src, int64_t n) {
    for (int64_t b = 0; b < n; b += L.n) {
        const int64_t j = b + L.id;
        const uint8_t v = j < n ? src[j] : 0;
        L.sync();
        if (j < n) dst[j] = v;
        L.sync();
    }
}

// match copy: out[op + j] = out[op - off + j], j < ml; off >= 1 and every source byte already written
ZHD void copy_match(const Lanes &L, uint8_t *op, uint32_t off, int64_t ml) {
    const uint8_t *src = op - off;
    if (L.n == 1) {
        for (int64_t j = 0; j < ml; ++j) op[j] = src[j];
        return;
    }
    if (off >= 32) {
        for (int64_t b = 0; b < ml; b += 32) {
            const int64_t j = b + L.id;
            if (j < ml) op[j] = src[j];
            L.sync();
        }
    } else {
        for (int64_t b = 0; b < ml; b += 32) {
            const int64_t j = b + L.id;
            if (j < ml) op[j] = src[j % off];
        }
        L.sync();
    }
}

// Huffman table of a literal section (HUF_readStats + HUF_readDTableX1).  Returns its size or -1.
ZHD int64_t read_huffman(Dec &d, const uint8_t *ip, int64_t n) {
    Smem &sm = *d.sm;
    const bool w0 = d.L.id == 0;
    if (n < 1) return -1;
    int64_t isize = ip[0];
    int osize;
    if (isize >= 128) {
        osize = (int)isize - 127;
        isize = (osize + 1) / 2;
        if (isize + 1 > n) return -1;
        if (w0)
            for (int k = 0; k < osize; k += 2) {
                sm.weights[k] = ip[1 + k / 2] >> 4;
                sm.weights[k + 1] = ip[1 + k / 2] & 15;
            }
    } else {
        if (isize + 1 > n) return -1;
        // FSE_decompress_wksp, maxLog 6, into at most 255 weights
        const uint8_t *src = ip + 1;
        int max_sv = 255, tlog = 0;
        const int64_t hs = read_ncount(sm.norm, w0, &max_sv, &tlog, src, isize);
        if (hs < 0) return -1;
        if (tlog > 6) return -1;
        {   // FSE_DECOMPRESS_WKSP_SIZE(tlog, max_sv) against HUF_READ_STATS_WORKSPACE_SIZE (u32 units)
            const int64_t need = (1 + (1 << tlog)) + 1 + ((2 * (max_sv + 1) + (1 << tlog) + 8 + 3) / 4) + 128 + 1;
            const int64_t have = (1 + 64) + 1 + ((2 * 12 + 64 + 8 + 3) / 4) + 128 + 1;
            if (need > have) return -1;
        }
        d.L.sync();
        if (w0) {
            fse_spread(sm.norm, max_sv, tlog, [&](int u, int s) { sm.wt[u].sym = (uint8_t)s; });
            uint16_t *next = sm.fse_next;
            for (int s = 0; s <= max_sv; ++s) next[s] = sm.norm[s] == -1 ? 1 : (uint16_t)sm.norm[s];
            for (int u = 0; u < (1 << tlog); ++u) {
                const uint32_t x = next[sm.wt[u].sym]++;
                const int nb = tlog - highbit(x);
                sm.wt[u].nbits = (uint8_t)nb;
                sm.wt[u].next = (uint16_t)((x << nb) - (1 << tlog));
            }
        }
        d.L.sync();
        BitD b;
        if (!bit_init(b, src + hs, isize - hs)) return -1;
        uint32_t s1 = (uint32_t)bit_read(b, tlog);
        bit_reload(b);
        uint32_t s2 = (uint32_t)bit_read(b, tlog);
        bit_reload(b);
        int o = 0;
        const int omax = 255;
        for (;;) {   // FSE_decompress_usingDTable_generic's tail loop (its 4-symbol loop cannot over-read)
            if (o > omax - 2) return -1;
            {
                const WtCell c = sm.wt[s1];
                if (w0) sm.weights[o] = c.sym;
                o++;
                s1 = c.next + (uint32_t)bit_read(b, c.nbits);
            }
            if (bit_reload(b) == BIT_OVERFLOW) {
                const WtCell c = sm.wt[s2];
                if (w0) sm.weights[o] = c.sym;
                o++;
                break;
            }
            if (o > omax - 2) return -1;
            {
                const WtCell c = sm.wt[s2];
                if (w0) sm.weights[o] = c.sym;
                o++;
                s2 = c.next + (uint32_t)bit_read(b, c.nbits);
            }
            if (bit_reload(b) == BIT_OVERFLOW) {
                const WtCell c = sm.wt[s1];
                if (w0) sm.weights[o] = c.sym;
                o++;
                break;
            }
        }
        osize = o;
    }
    d.L.sync();
    uint32_t rank[HUF_LOG_MAX + 2];
    for (int k = 0; k < HUF_LOG_MAX + 2; ++k) rank[k] = 0;
    uint32_t total = 0;
    for (int k = 0; k < osize; ++k) {
        const int wgt = sm.weights[k];
        if (wgt > HUF_LOG_MAX) return -1;
        rank[wgt]++;
        total += (1u << wgt) >> 1;
    }
    if (total == 0) return -1;
    const int tlog = highbit(total) + 1;
    if (tlog > HUF_LOG_MAX) return -1;
    const uint32_t rest = (1u << tlog) - total;
    if ((1u << highbit(rest)) != rest) return -1;
    const int last_w = highbit(rest) + 1;
    rank[last_w]++;
    if (rank[1] < 2 || (rank[1] & 1)) return -1;
    const int nsym = osize + 1;
    // cells: weight 1 first, then 2, ...; within a weight by symbol
    uint32_t start[HUF_LOG_MAX + 2];
    {
        uint32_t at = 0;
        for (int wgt = 1; wgt <= tlog; ++wgt) {
            start[wgt] = at;
            at += rank[wgt] << (wgt - 1);
        }
    }
    for (int s = 0; s < nsym; ++s) {
        const int wgt = s == osize ? last_w : sm.weights[s];
        if (wgt == 0) continue;
        const uint32_t len = (1u << wgt) >> 1;
        const uint16_t cell = (uint16_t)(s | (tlog + 1 - wgt) << 8);
        for (uint32_t u = d.L.id; u < len; u += d.L.n) sm.huf[start[wgt] + u] = cell;
        start[wgt] += len;
    }
    d.L.sync();
    d.huf_log = tlog;
    return isize + 1;
}

// one Huffman stream of cnt symbols into dst; true iff decoded and consumed exactly
ZHD bool huf_stream(const Smem &sm, int tlog, const uint8_t *src, int64_t n, uint8_t *dst, int64_t cnt) {
    BitD b;
    if (!bit_init(b, src, n)) return false;
    int64_t k = 0;
    for (; k + 4 <= cnt; k += 4) {
#pragma unroll
        for (int q = 0; q < 4; ++q) {
            const uint16_t c = sm.huf[bit_look(b, tlog)];
            b.consumed += c >> 8;
            dst[k + q] = (uint8_t)c;
        }
        if (bit_reload(b) == BIT_OVERFLOW) return false;
    }
    for (; k < cnt; ++k) {
        const uint16_t c = sm.huf[bit_look(b, tlog)];
        b.consumed += c >> 8;
        dst[k] = (uint8_t)c;
        if (bit_reload(b) == BIT_OVERFLOW) return false;
    }
    bit_reload(b);
    return bit_end(b);
}

// literal section of a compressed block (ZSTD_decodeLiteralsBlock).  Sets the literals' location
// (*lit: in the input for raw, in the tail of the output for Huffman; rle >= 0: one repeated byte).
ZHD int64_t read_literals(Dec &d, const uint8_t *ip, int64_t n, int64_t op, const uint8_t **lit, int *rle,
                          int64_t *lit_n) {
    if (n < MIN_CBLOCK) return -1;
    const int type = ip[0] & 3;
    const int lh = (ip[0] >> 2) & 3;
    const int64_t room = d.cap - op < BLOCK_MAX ? d.cap - op : BLOCK_MAX;
    *rle = -1;
    if (type == 0 || type == 1) {            // raw / RLE
        int64_t hs, size;
        if (lh == 1) {
            hs = 2;
            if (type == 1 && n < 3) return -1;
            size = ld16(ip) >> 4;
        } else if (lh == 3) {
            hs = 3;
            if (n < (type == 0 ? 3 : 4)) return -1;
            size = ld24(ip) >> 4;
        } else {
            hs = 1;
            size = ip[0] >> 3;
        }
        if (size > BLOCK_MAX || size > room) return -1;
        *lit_n = size;
        if (type == 0) {
            if (hs + size > n) return -1;
            *lit = ip + hs;
            return hs + size;
        }
        *rle = ip[hs];
        return hs + 1;
    }
    if (type == 3 && d.huf_log == 0) return -1;   // treeless with no earlier table
    if (n < 5) return -1;
    const uint32_t lhc = ld32(ip);
    int64_t hs, size, csize;
    const bool single = lh == 0;
    if (lh <= 1) {
        hs = 3;
        size = (lhc >> 4) & 0x3FF;
        csize = (lhc >> 14) & 0x3FF;
    } else if (lh == 2) {
        hs = 4;
        size = (lhc >> 4) & 0x3FFF;
        csize = lhc >> 18;
    } else {
        hs = 5;
        size = (lhc >> 4) & 0x3FFFF;
        csize = (lhc >> 22) + ((int64_t)ip[4] << 10);
    }
    if (size > BLOCK_MAX) return -1;
    if (!single && size < 6) return -1;
    if (csize + hs > n) return -1;
    if (size > room) return -1;
    const uint8_t *src = ip + hs;
    int64_t sn = csize;
    if (type == 2) {
        const int64_t t = read_huffman(d, src, sn);
        if (t < 0) return -1;
        if (t >= sn) return -1;
        src += t;
        sn -= t;
    }
    uint8_t *dst = d.out + d.cap - size;     // the tail of the frame's output
    *lit = dst;
    *lit_n = size;
    Smem &sm = *d.sm;
    const int tlog = d.huf_log;
    if (single) {
        if (d.L.id == 0) sm.ok4[0] = huf_stream(sm, tlog, src, sn, dst, size);
        d.L.sync();
        const bool ok = sm.ok4[0] != 0;
        d.L.sync();
        return ok ? hs + csize : -1;
    }
    if (sn < 10) return -1;
    const int64_t l1 = ld16(src), l2 = ld16(src + 2), l3 = ld16(src + 4);
    const int64_t l4 = sn - (l1 + l2 + l3 + 6);
    if (l4 < 0 || l4 > sn) return -1;
    const int64_t seg = (size + 3) / 4;
    const int64_t len[4] = {l1, l2, l3, l4};
    for (int s = d.L.id; s < 4; s += d.L.n) {
        const int64_t at = 6 + (s > 0 ? l1 : 0) + (s > 1 ? l2 : 0) + (s > 2 ? l3 : 0);
        const int64_t cnt = s < 3 ? seg : size - 3 * seg;
        sm.ok4[s] = huf_stream(sm, tlog, src + at, len[s], dst + s * seg, cnt);
    }
    d.L.sync();
    const bool ok = sm.ok4[0] && sm.ok4[1] && sm.ok4[2] && sm.ok4[3];
    d.L.sync();
    return ok ? hs + csize : -1;
}

// one table of the sequences header (ZSTD_buildSeqTable); returns the bytes it took or -1
ZHD int64_t read_seq_table(Dec &d, int kind, int mode, const uint8_t *ip, int64_t n) {
    Smem &sm = *d.sm;
    SeqCell *tab = kind == T_LL ? sm.ll : kind == T_OF ? sm.of : sm.ml;
    const int max_sv = kind == T_LL ? 35 : kind == T_OF ? 31 : 52;
    const int max_log = kind == T_OF ? 8 : 9;
    const bool w0 = d.L.id == 0;
    if (mode == 0) {                         // predefined
        d.L.sync();
        if (w0) {
            const int msv = default_norm(kind, sm.norm);
            build_seq_table(tab, kind, sm.norm, msv, kind == T_OF ? 5 : 6, sm.fse_next);
        }
        d.L.sync();
        d.seq_log[kind] = kind == T_OF ? 5 : 6;
        return 0;
    }
    if (mode == 1) {                         // RLE
        if (n < 1) return -1;
        const int s = ip[0];
        if (s > max_sv) return -1;
        d.L.sync();
        if (w0) {
            uint32_t base;
            int extra;
            code_of(kind, s, &base, &extra);
            tab[0].base = base;
            tab[0].extra = (uint8_t)extra;
            tab[0].nbits = 0;
            tab[0].next = 0;
        }
        d.L.sync();
        d.seq_log[kind] = 0;
        return 1;
    }
    if (mode == 3) return d.fse_entropy ? 0 : -1;   // repeat
    int msv = max_sv, tlog = 0;
    d.L.sync();
    const int64_t hs = read_ncount(sm.norm, w0, &msv, &tlog, ip, n);
    if (hs < 0 || tlog > max_log) return -1;
    d.L.sync();
    if (w0) build_seq_table(tab, kind, sm.norm, msv, tlog, sm.fse_next);
    d.L.sync();
    d.seq_log[kind] = tlog;
    return hs;
}

// one compressed block at output position op; returns the bytes it wrote or -1
ZHD int64_t compressed_block(Dec &d, const uint8_t *ip, int64_t n, int64_t op) {
    const uint8_t *lit;
    int rle;
    int64_t lit_n;
    const int64_t lh = read_literals(d, ip, n, op, &lit, &rle, &lit_n);
    if (lh < 0) return -1;
    ip += lh;
    n -= lh;
    // sequences header (ZSTD_decodeSeqHeaders)
    if (n < 1) return -1;
    int64_t nseq = ip[0];
    int64_t p = 1;
    bool tables = true;
    if (nseq == 0) {
        if (n != 1) return -1;
        tables = false;
    } else if (nseq > 0x7F) {
        if (nseq == 0xFF) {
            if (p + 2 > n) return -1;
            nseq = ld16(ip + 1) + 0x7F00;
            p += 2;
        } else {
            if (p >= n) return -1;
            nseq = ((nseq - 0x80) << 8) + ip[1];
            p += 1;
        }
    }
    if (tables) {
        if (p + 1 > n) return -1;
        const int modes = ip[p];
        if (modes & 3) return -1;  // reserved bits (RFC 8878 3.1.1.3.2.1; libzstd refuses them from 1.5.6 on)
        p++;
        const int kinds[3] = {T_LL, T_OF, T_ML};
        const int m[3] = {modes >> 6, (modes >> 4) & 3, (modes >> 2) & 3};
        for (int t = 0; t < 3; ++t) {
            const int64_t r = read_seq_table(d, kinds[t], m[t], ip + p, n - p);
            if (r < 0) return -1;
            p += r;
        }
    }
    const int64_t cap_left = d.cap - op;
    if (cap_left == 0 && nseq > 0) return -1;
    uint8_t *const out = d.out;
    int64_t o = op;
    int64_t lit_at = 0;
    const bool lit_in_out = rle < 0 && lit >= out && lit < out + d.cap;
    if (nseq > 0) {
        d.fse_entropy = true;
        const Smem &sm = *d.sm;
        BitD b;
        if (!bit_init(b, ip + p, n - p)) return -1;
        uint32_t sll = (uint32_t)bit_read(b, d.seq_log[T_LL]);
        bit_reload(b);
        uint32_t sof = (uint32_t)bit_read(b, d.seq_log[T_OF]);
        bit_reload(b);
        uint32_t sml = (uint32_t)bit_read(b, d.seq_log[T_ML]);
        bit_reload(b);
        for (int64_t k = 0; k < nseq; ++k) {
            const SeqCell cl = sm.ll[sll], cm = sm.ml[sml], co = sm.of[sof];
            uint32_t off;
            const int ob = co.extra;
            const bool ll0 = cl.base == 0 && cl.extra == 0;
            if (ob > 1) {
                off = co.base + (uint32_t)bit_read(b, ob);
                d.rep[2] = d.rep[1];
                d.rep[1] = d.rep[0];
                d.rep[0] = off;
            } else if (ob == 0) {
                off = d.rep[ll0 ? 1 : 0];
                d.rep[1] = d.rep[ll0 ? 0 : 1];
                d.rep[0] = off;
            } else {
                const uint32_t v = co.base + (ll0 ? 1u : 0u) + (uint32_t)bit_read(b, 1);
                uint32_t t = v == 3 ? d.rep[0] - 1 : d.rep[v];
                t -= t == 0;   // 0 is no offset: libzstd forces -1, which fails below
                if (v != 1) d.rep[2] = d.rep[1];
                d.rep[1] = d.rep[0];
                d.rep[0] = off = t;
            }
            const int64_t ml = cm.base + (int64_t)bit_read(b, cm.extra);
            if (ob + cm.extra + cl.extra >= 57 - (9 + 9 + 8)) bit_reload(b);
            const int64_t ll = cl.base + (int64_t)bit_read(b, cl.extra);
            if (k + 1 < nseq) {
                sll = cl.next + (uint32_t)bit_read(b, cl.nbits);
                sml = cm.next + (uint32_t)bit_read(b, cm.nbits);
                sof = co.next + (uint32_t)bit_read(b, co.nbits);
            }
            bit_reload(b);
            // ZSTD_execSequence's checks
            if (ll + ml > d.cap - o) return -1;
            if (ll > lit_n - lit_at) return -1;
            if (off == 0xFFFFFFFFu || (int64_t)off > o + ll) return -1;
            // literals kept in the output's tail must not be overwritten before they are read: when they
            // would be, the block cannot end within the frame's size, and libzstd refuses it too
            if (lit_in_out && o + ll + ml + (lit_n - lit_at - ll) > d.cap) return -1;
            if (ll) {
                if (rle >= 0) {
                    for (int64_t j = d.L.id; j < ll; j += d.L.n) out[o + j] = (uint8_t)rle;
                    d.L.sync();
                } else {
                    copy_fwd(d.L, out + o, lit + lit_at, ll);
                }
            }
            o += ll;
            lit_at += ll;
            copy_match(d.L, out + o, off, ml);
            o += ml;
        }
        if (!bit_end(b)) return -1;
    }
    const int64_t last = lit_n - lit_at;
    if (last > d.cap - o) return -1;
    if (last) {
        if (rle >= 0) {
            for (int64_t j = d.L.id; j < last; j += d.L.n) out[o + j] = (uint8_t)rle;
            d.L.sync();
        } else {
            copy_fwd(d.L, out + o, lit + lit_at, last);
        }
    }
    o += last;
    return o - op;
}

// the whole frame; returns a WSTR_ZSTD_* status
ZHD int decode_frame(Dec &d) {
    const uint8_t *ip = d.in;
    const int64_t n = d.in_n;
    if (n < 6 + 3) return WSTR_ZSTD_FRAME_HEADER;
    if (ld32(ip) != 0xFD2FB528u) return WSTR_ZSTD_FRAME_HEADER;
    const int fhd = ip[4];
    const int did = fhd & 3, single = (fhd >> 5) & 1, fcs_id = fhd >> 6;
    const int did_size[4] = {0, 1, 2, 4}, fcs_size[4] = {0, 2, 4, 8};
    const int64_t hsize = 5 + !single + did_size[did] + fcs_size[fcs_id] + (single && !fcs_id);
    if (n < hsize + 3) return WSTR_ZSTD_FRAME_HEADER;
    if (fhd & 0x08) return WSTR_ZSTD_FRAME_HEADER;          // reserved bit
    int64_t p = 5;
    if (!single) {
        const int wlog = (ip[p] >> 3) + 10;
        if (wlog > 31) return WSTR_ZSTD_FRAME_HEADER;
        p++;
    }
    uint32_t dict = 0;
    if (did == 1) dict = ip[p];
    else if (did == 2) dict = ld16(ip + p);
    else if (did == 3) dict = ld32(ip + p);
    p += did_size[did];
    if (dict != 0) return WSTR_ZSTD_FRAME_HEADER;           // no dictionary is loaded
    int64_t fcs = -1;
    if (fcs_id == 0) {
        if (single) fcs = ip[p];
    } else if (fcs_id == 1) {
        fcs = ld16(ip + p) + 256;
    } else if (fcs_id == 2) {
        fcs = ld32(ip + p);
    } else {
        const uint64_t v = ld32(ip + p) | (uint64_t)ld32(ip + p + 4) << 32;
        fcs = v > (uint64_t)INT64_MAX ? INT64_MAX : (int64_t)v;
    }
    if (fhd & 0x04) return WSTR_ZSTD_UNSUPPORTED;           // content checksum: the host path
    if (fcs < 0) return WSTR_ZSTD_UNSUPPORTED;              // no content size: the host path
    if (fcs != d.cap) return WSTR_ZSTD_SIZE;
    p = hsize;
    int64_t o = 0;
    for (;;) {
        if (n - p < 3) return WSTR_ZSTD_BLOCK;
        const uint32_t bh = ld24(ip + p);
        p += 3;
        const bool last = bh & 1;
        const int type = (bh >> 1) & 3;
        const int64_t bsize = bh >> 3;
        if (type == 3) return WSTR_ZSTD_BLOCK;
        const int64_t csize = type == 1 ? 1 : bsize;
        if (csize > n - p) return WSTR_ZSTD_BLOCK;
        if (type == 0) {
            if (bsize > d.cap - o) return WSTR_ZSTD_SIZE;
            copy_fwd(d.L, d.out + o, ip + p, bsize);
            o += bsize;
        } else if (type == 1) {
            if (bsize > d.cap - o) return WSTR_ZSTD_SIZE;
            const uint8_t v = ip[p];
            for (int64_t j = d.L.id; j < bsize; j += d.L.n) d.out[o + j] = v;
            d.L.sync();
            o += bsize;
        } else {
            if (bsize > BLOCK_MAX) return WSTR_ZSTD_BLOCK;
            const int64_t w = compressed_block(d, ip + p, bsize, o);
            if (w < 0) return WSTR_ZSTD_CORRUPT;
            o += w;
        }
        p += csize;
        if (last) break;
    }
    if (o != d.cap) return WSTR_ZSTD_SIZE;
    if (p != n) return WSTR_ZSTD_TRAILING;
    return WSTR_ZSTD_OK;
}

ZHD void dec_init(Dec &d, const uint8_t *in, int64_t in_n, uint8_t *out, int64_t cap, Smem *sm, Lanes L) {
    d.in = in;
    d.in_n = in_n;
    d.out = out;
    d.cap = cap;
    d.sm = sm;
    d.L = L;
    d.huf_log = 0;
    d.seq_log[0] = d.seq_log[1] = d.seq_log[2] = 0;
    d.fse_entropy = false;
    d.rep[0] = 1;
    d.rep[1] = 4;
    d.rep[2] = 8;
}

#ifdef __CUDACC__
__global__ void __launch_bounds__(WARPS * 32) zstd_decode_kernel(const uint8_t *__restrict__ in,
                                                                 const Frame *__restrict__ frames, int n,
                                                                 int *__restrict__ queue, uint8_t *__restrict__ out,
                                                                 int32_t *__restrict__ status) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    Smem *sm = reinterpret_cast<Smem *>(smem_raw) + warp;
    for (;;) {
        int f = 0;
        if (lane == 0) f = atomicAdd(queue, 1);
        f = __shfl_sync(0xffffffffu, f, 0);
        if (f >= n) break;
        const Frame fr = frames[f];
        Dec d;
        dec_init(d, in + fr.in_off, fr.in_bytes, out + fr.out_off, fr.out_bytes, sm, Lanes{lane, 32});
        const int st = decode_frame(d);
        if (lane == 0) status[fr.index] = st;
        __syncwarp();
    }
}
#endif

}  // namespace wstr_zstd

#ifdef __CUDACC__
using namespace wstr_zstd;

// staged block: [queue counter, padding to 16 bytes][Frame x n, longest output first]
extern "C" int64_t wstr_zstd_workspace_bytes(int32_t n_frames) {
    if (n_frames < 0) return WSTR_ERR_INVALID_ARGUMENT;
    return 16 + (int64_t)sizeof(Frame) * n_frames + 256;
}

extern "C" int wstr_zstd_decode_batch(const uint8_t *d_in, const int64_t *in_off, const int64_t *in_bytes,
                                      const int64_t *out_off, const int64_t *out_bytes, int32_t n_frames,
                                      uint8_t *d_out, int32_t *d_status, void *d_workspace, int64_t workspace_bytes,
                                      void *stream) {
    if (!in_off || !in_bytes || !out_off || !out_bytes || !d_status || !d_workspace || n_frames < 0)
        return WSTR_ERR_INVALID_ARGUMENT;
    if (n_frames == 0) return WSTR_OK;
    if (!d_in || !d_out || (reinterpret_cast<uintptr_t>(d_in) & 15)) return WSTR_ERR_INVALID_ARGUMENT;
    if (workspace_bytes < wstr_zstd_workspace_bytes(n_frames)) return WSTR_ERR_WORKSPACE_TOO_SMALL;
    for (int f = 0; f < n_frames; ++f) {
        const bool ok = in_off[f] >= 0 && (in_off[f] & 15) == 0 && in_bytes[f] >= 0 && out_off[f] >= 0 &&
                        out_bytes[f] >= 0 && out_bytes[f] <= (int64_t)1 << 40;
        if (!ok) return WSTR_ERR_INVALID_ARGUMENT;
    }
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    const size_t bytes = 16 + sizeof(Frame) * (size_t)n_frames;
    void *h = nullptr, *token = nullptr;
    int rc = wstr_stage_begin(bytes, &h, &token);
    if (rc != WSTR_OK) return rc;
    int32_t *hq = static_cast<int32_t *>(h);
    hq[0] = hq[1] = hq[2] = hq[3] = 0;
    Frame *hf = reinterpret_cast<Frame *>(static_cast<char *>(h) + 16);
    // longest first by the output's power of two: a stable counting pass, O(n)
    {
        int cnt[65] = {0}, at[65];
        auto bucket = [&](int f) { return out_bytes[f] > 0 ? __builtin_clzll((unsigned long long)out_bytes[f]) : 64; };
        for (int f = 0; f < n_frames; ++f) cnt[bucket(f)]++;
        for (int b = 0, a = 0; b < 65; ++b) {
            at[b] = a;
            a += cnt[b];
        }
        for (int f = 0; f < n_frames; ++f) hf[at[bucket(f)]++] = Frame{in_off[f], in_bytes[f], out_off[f], out_bytes[f], f};
    }
    rc = wstr_stage_commit(token, d_workspace, bytes, s);
    if (rc != WSTR_OK) return rc;
    static unsigned long long attr_done = 0ull;
    int dev = 0;
    WSTR_CUDA(cudaGetDevice(&dev));
    const size_t smem = sizeof(Smem) * WARPS;
    if (!((attr_done >> (dev & 63)) & 1ull)) {
        WSTR_CUDA(cudaFuncSetAttribute(zstd_decode_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        attr_done |= 1ull << (dev & 63);
    }
    int per_sm = 0, sms = 0;
    WSTR_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, zstd_decode_kernel, WARPS * 32, smem));
    WSTR_CUDA(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
    const int want = (n_frames + WARPS - 1) / WARPS;
    const int cap = (per_sm > 0 ? per_sm : 1) * sms;
    const int grid = want < cap ? want : cap;
    char *ws = static_cast<char *>(d_workspace);
    zstd_decode_kernel<<<grid, WARPS * 32, smem, s>>>(d_in, reinterpret_cast<const Frame *>(ws + 16), n_frames,
                                                     reinterpret_cast<int *>(ws), d_out, d_status);
    WSTR_CUDA(cudaGetLastError());
    return WSTR_OK;
}
#endif
