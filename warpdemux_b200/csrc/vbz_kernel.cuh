// vbz_kernel.cuh — pod5 VBZ signal decoding: zstd frame decoder (RFC 8878) and the streamvbyte-16 row decoder.
//
// A VBZ chunk is zstd( streamvbyte16( zigzag( delta( int16 samples )))), one zstd frame per chunk.  The frame decoder
// below runs one WARP per frame: every lane walks the same bitstreams with the same state (uniform control flow, no
// broadcasts), lane-strided loops copy raw literals and matches, lane 0 writes the Huffman-decoded literals.  Compiled
// as host code (VBZ_HD without a device) the same functions run with one lane, which is how malformed input is
// rehearsed on the CPU.
//
// Supported subset (anything else is a per-frame status, never a fault):
//   one zstd frame per chunk, single-segment or with a window descriptor, with or without Frame_Content_Size;
//   raw / RLE / compressed blocks (<= 128 KiB); literals raw / RLE / Huffman 1 or 4 streams / treeless;
//   sequences with predefined / RLE / FSE / repeat tables for LL, OF, ML and the three repeat offsets.
//   Not supported: dictionaries, content checksums, skippable frames, several frames in one chunk.
// Bounded by construction: every input read is checked against the frame's byte range, every output write against
// min(limit, capacity), every loop has a bound (input bytes, table sizes, sequence count).
#pragma once
#include <cstdint>

#ifdef __CUDACC__
#define VBZ_HD __host__ __device__ __forceinline__
#else
#define VBZ_HD inline
#endif

namespace wdx {
namespace vbz {

// per-chunk status (include/wdx_b200.h: WDX_VBZ_*)
enum {
    ST_OK = 0,
    ST_BAD_MAGIC = 1,    // not a zstd frame
    ST_DICTIONARY = 2,   // the frame names a dictionary
    ST_CHECKSUM = 3,     // content checksum flag set
    ST_RESERVED = 4,     // reserved header bit, block type or field value
    ST_TRUNCATED = 5,    // the input ends inside the frame
    ST_CORRUPT = 6,      // inconsistent tables, bitstreams, offsets or sizes
    ST_TOO_LARGE = 7,    // the content does not fit its output capacity (svb16 bound in the row decoder)
    ST_FRAMES = 8,       // skippable frame, or bytes after the frame (a second frame)
    ST_SAMPLES = 9,      // row decoder: key / data lengths disagree with the chunk's `samples`
    ST_SCRATCH = 10,     // row decoder: the chunk's scratch region is too small or misaligned
};

constexpr int HUF_MAX_BITS = 11;
constexpr int LL_MAX_AL = 9, ML_MAX_AL = 9, OF_MAX_AL = 8;
constexpr int LL_MAX_SYM = 35, ML_MAX_SYM = 52, OF_MAX_SYM = 31;
constexpr int64_t BLOCK_MAX = 128 * 1024;

struct FseEntry {
    uint16_t base;
    uint8_t sym;
    uint8_t nb;
};

// one warp's decode tables (shared memory on the device)
struct Tables {
    uint16_t huf[1 << HUF_MAX_BITS];   // (symbol << 8) | code length
    FseEntry ll[1 << LL_MAX_AL], ml[1 << ML_MAX_AL], of[1 << OF_MAX_AL];
    FseEntry hw[64];                   // Huffman weights (accuracy log <= 6)
    int16_t norm[64];
    uint16_t next[64];
    uint8_t w[256];                    // Huffman weights
};

VBZ_HD void warp_sync() {
#ifdef __CUDA_ARCH__
    __syncwarp();
#endif
}

VBZ_HD int highbit(uint32_t x) {   // x > 0
#ifdef __CUDA_ARCH__
    return 31 - __clz(x);
#else
    return 31 - __builtin_clz(x);
#endif
}

VBZ_HD uint32_t rd_le(const uint8_t* p, int k) {
    uint32_t v = 0;
    for (int i = 0; i < k; i++) v |= (uint32_t)p[i] << (8 * i);
    return v;
}

// bytes [0, n) as a backward bitstream (zstd: the highest set bit of the last byte marks the end)
struct RevBits {
    const uint8_t* p;
    int64_t n;
    int64_t pos;   // bits [0, pos) unread

    VBZ_HD bool init(const uint8_t* src, int64_t nbytes) {
        p = src;
        n = nbytes;
        if (nbytes < 1 || src[nbytes - 1] == 0) return false;
        pos = 8 * (nbytes - 1) + highbit(src[nbytes - 1]);
        return true;
    }
    // bits [pos - k, pos), zeros below bit 0; k <= 32
    VBZ_HD uint32_t peek(int k) const {
        if (k == 0) return 0;
        const int64_t lo = pos - k;
        const uint64_t mask = (k == 32) ? 0xffffffffull : ((1ull << k) - 1);
        if (lo >= 0) {
            const int64_t b = lo >> 3;
            uint64_t w = 0;
            for (int i = 0; i < 5; i++)
                if (b + i < n) w |= (uint64_t)p[b + i] << (8 * i);
            return (uint32_t)((w >> (lo & 7)) & mask);
        }
        if (pos <= 0) return 0;
        uint64_t w = 0;
        for (int64_t i = 0; i < 5 && 8 * i < pos; i++) w |= (uint64_t)p[i] << (8 * i);
        w &= (1ull << pos) - 1;
        return (uint32_t)((w << (-lo)) & mask);
    }
    VBZ_HD uint32_t read(int k) {
        const uint32_t v = peek(k);
        pos -= k;
        return v;
    }
};

// FSE table description (RFC 8878 4.1.1).  Returns bytes consumed (> 0) or -status.
VBZ_HD int fse_read_ncount(const uint8_t* p, int64_t n, int max_al, int max_sym, int16_t* norm, int* nsym, int* al_out) {
    int64_t bit = 0;
    auto peek = [&](int k) -> uint32_t {
        const int64_t b = bit >> 3;
        uint32_t w = 0;
        for (int i = 0; i < 4; i++)
            if (b + i < n) w |= (uint32_t)p[b + i] << (8 * i);
        return (w >> (bit & 7)) & ((1u << k) - 1);
    };
    if (n < 1) return -ST_TRUNCATED;
    const int al = (int)peek(4) + 5;
    bit = 4;
    if (al > max_al) return -ST_CORRUPT;
    int remaining = (1 << al) + 1, threshold = 1 << al, nbits = al + 1, sym = 0;
    while (remaining > 1 && sym <= max_sym) {
        const int maxv = 2 * threshold - 1 - remaining;
        const uint32_t v = peek(nbits);
        int count;
        if ((int)(v & (threshold - 1)) < maxv) {
            count = (int)(v & (threshold - 1));
            bit += nbits - 1;
        } else {
            count = (int)(v & (2 * threshold - 1));
            if (count >= threshold) count -= maxv;
            bit += nbits;
        }
        count--;
        remaining -= count < 0 ? -count : count;
        norm[sym++] = (int16_t)count;
        if (count == 0) {
            int rep;
            do {
                rep = (int)peek(2);
                bit += 2;
                for (int k = 0; k < rep; k++) {
                    if (sym > max_sym) return -ST_CORRUPT;
                    norm[sym++] = 0;
                }
            } while (rep == 3);
        }
        if (remaining < 1) return -ST_CORRUPT;
        while (remaining < threshold) {
            nbits--;
            threshold >>= 1;
        }
        if (bit > 8 * n) return -ST_TRUNCATED;
    }
    if (remaining != 1 || bit > 8 * n) return -ST_CORRUPT;
    *nsym = sym;
    *al_out = al;
    return (int)((bit + 7) >> 3);
}

// decode table from normalised counts (RFC 8878 4.1.1 "FSE table construction"); single-threaded
VBZ_HD int fse_build(FseEntry* t, const int16_t* norm, int nsym, int al, uint16_t* next) {
    const int size = 1 << al;
    int high = size - 1;
    for (int s = 0; s < nsym; s++) {
        if (norm[s] == -1) {
            t[high--].sym = (uint8_t)s;
            next[s] = 1;
        } else {
            next[s] = (uint16_t)norm[s];
        }
    }
    const int step = (size >> 1) + (size >> 3) + 3, mask = size - 1;
    int pos = 0;
    for (int s = 0; s < nsym; s++)
        for (int i = 0; i < norm[s]; i++) {
            t[pos].sym = (uint8_t)s;
            do pos = (pos + step) & mask;
            while (pos > high);
        }
    if (pos != 0) return -ST_CORRUPT;
    for (int u = 0; u < size; u++) {
        const int s = t[u].sym;
        const uint32_t x = next[s]++;
        const int nb = al - highbit(x);
        t[u].nb = (uint8_t)nb;
        t[u].base = (uint16_t)((x << nb) - size);
    }
    return 0;
}

VBZ_HD void fse_rle(FseEntry* t, int sym) {
    t[0].sym = (uint8_t)sym;
    t[0].nb = 0;
    t[0].base = 0;
}

// predefined distributions (RFC 8878 3.1.1.3.2.2)
VBZ_HD int fse_predefined(FseEntry* t, int which, int16_t* norm, uint16_t* next) {
    static constexpr int16_t LL[36] = {4, 3, 2, 2, 2, 2, 2, 2, 2, 2, 2, 2, 2, 1, 1, 1, 2, 2, 2, 2, 2, 2, 2, 2, 2, 3, 2, 1, 1, 1, 1, 1,
                                       -1, -1, -1, -1};
    static constexpr int16_t ML[53] = {1, 4, 3, 2, 2, 2, 2, 2, 2, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1,
                                       1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, -1, -1, -1, -1, -1, -1, -1};
    static constexpr int16_t OF[29] = {1, 1, 1, 1, 1, 1, 2, 2, 2, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, -1, -1, -1, -1, -1};
    const int16_t* src = which == 0 ? LL : (which == 1 ? OF : ML);
    const int nsym = which == 0 ? 36 : (which == 1 ? 29 : 53);
    for (int s = 0; s < nsym; s++) norm[s] = src[s];
    return fse_build(t, norm, nsym, which == 1 ? 5 : 6, next);
}

// Huffman tree description (RFC 8878 4.2.1) -> T.huf.  Returns bytes consumed or -status; *max_bits = code length.
// All lanes call it; table writes are lane-strided, the FSE weight table is built by lane 0.
VBZ_HD int huf_read(const uint8_t* p, int64_t n, Tables& T, int* max_bits, int lane, int nl) {
    if (n < 1) return -ST_TRUNCATED;
    const int h = p[0];
    int nw = 0, used = 0;
    if (h >= 128) {
        nw = h - 127;
        used = 1 + (nw + 1) / 2;
        if (used > n) return -ST_TRUNCATED;
        for (int i = 0; i < nw; i++) {
            const uint8_t b = p[1 + i / 2];
            T.w[i] = (i & 1) ? (b & 15) : (b >> 4);
        }
    } else {
        used = 1 + h;
        if (used > n) return -ST_TRUNCATED;
        int nsym = 0, al = 0;
        const int hdr = fse_read_ncount(p + 1, h, 6, 12, T.norm, &nsym, &al);
        if (hdr < 0) return hdr;
        warp_sync();
        if (lane == 0) fse_build(T.hw, T.norm, nsym, al, T.next);   // cannot fail, see read_seq_table
        warp_sync();
        RevBits bs;
        if (!bs.init(p + 1 + hdr, h - hdr)) return -ST_CORRUPT;
        uint32_t s1 = bs.read(al), s2 = bs.read(al);
        // two interleaved states, as zstd's FSE_decompress: stop when a state update overruns the stream
        while (true) {
            if (nw > 253) return -ST_CORRUPT;
            FseEntry e = T.hw[s1];
            T.w[nw++] = e.sym;   // every lane writes the same value
            s1 = e.base + bs.read(e.nb);
            if (bs.pos < 0) {
                T.w[nw++] = T.hw[s2].sym;
                break;
            }
            e = T.hw[s2];
            T.w[nw++] = e.sym;
            s2 = e.base + bs.read(e.nb);
            if (bs.pos < 0) {
                T.w[nw++] = T.hw[s1].sym;
                break;
            }
        }
    }
    warp_sync();
    uint32_t total = 0;
    for (int i = 0; i < nw; i++) {
        if (T.w[i] > HUF_MAX_BITS) return -ST_CORRUPT;
        if (T.w[i]) total += 1u << (T.w[i] - 1);
    }
    if (total == 0) return -ST_CORRUPT;
    const int mb = highbit(total) + 1;
    if (mb > HUF_MAX_BITS) return -ST_CORRUPT;
    const uint32_t rest = (1u << mb) - total;
    if (rest & (rest - 1)) return -ST_CORRUPT;
    const int last_w = highbit(rest) + 1;
    if (nw + 1 > 256) return -ST_CORRUPT;
    warp_sync();
    if (lane == 0) T.w[nw] = (uint8_t)last_w;
    warp_sync();
    const int nsym = nw + 1;
    uint32_t start[HUF_MAX_BITS + 2] = {0};
    uint32_t cnt[HUF_MAX_BITS + 2] = {0};
    for (int s = 0; s < nsym; s++) cnt[T.w[s]]++;
    uint32_t acc = 0;
    for (int w = 1; w <= mb; w++) {
        start[w] = acc;
        acc += cnt[w] << (w - 1);
    }
    for (int s = 0; s < nsym; s++) {
        const int w = T.w[s];
        if (!w) continue;
        const uint32_t len = 1u << (w - 1), st = start[w];
        start[w] += len;
        const uint16_t e = (uint16_t)((s << 8) | (mb + 1 - w));
        for (uint32_t j = lane; j < len; j += nl) T.huf[st + j] = e;
    }
    warp_sync();
    *max_bits = mb;
    return used;
}

struct LitSrc {
    int type;             // 0 raw, 1 RLE, 2 Huffman
    const uint8_t* raw;   // raw literals / RLE byte
    int64_t size;         // regenerated size
    int64_t used;
    // Huffman: up to 4 streams, consumed in order
    int nstreams, cur;
    const uint8_t* sp[4];
    int64_t sn[4];
    int64_t quota[4];
    int64_t left;         // literals left in the current stream
    RevBits bs;
    int mb;
};

VBZ_HD int lit_next_stream(LitSrc& L) {
    // the finished stream must be consumed exactly
    if (L.cur >= 0 && L.bs.pos != 0) return -ST_CORRUPT;
    L.cur++;
    if (L.cur >= L.nstreams) return -ST_CORRUPT;
    if (!L.bs.init(L.sp[L.cur], L.sn[L.cur])) return -ST_CORRUPT;
    L.left = L.quota[L.cur];
    return 0;
}

VBZ_HD int lit_huf_one(LitSrc& L, const Tables& T, uint8_t* sym) {
    while (L.left == 0) {
        const int rc = lit_next_stream(L);
        if (rc) return rc;
    }
    const uint16_t e = T.huf[L.bs.peek(L.mb)];
    L.bs.pos -= e & 0xff;
    if (L.bs.pos < 0) return -ST_CORRUPT;
    L.left--;
    *sym = (uint8_t)(e >> 8);
    return 0;
}

struct Out {
    uint8_t* out;
    int64_t pos;
    int64_t stop;     // min(limit, capacity)
    bool cap_bound;   // stop comes from the capacity (writing past it means the content is too large)
};

// literals -> output.  Returns 0, 1 (output stop reached) or -status.
VBZ_HD int emit_literals(LitSrc& L, const Tables& T, Out& o, int64_t count, int lane, int nl) {
    if (count > L.size - L.used) return -ST_CORRUPT;
    int64_t k = count;
    int done = 0;
    if (o.pos + k > o.stop) {
        if (o.cap_bound) return -ST_TOO_LARGE;
        k = o.stop - o.pos;
        done = 1;
    }
    if (L.type == 0) {
        for (int64_t i = lane; i < k; i += nl) o.out[o.pos + i] = L.raw[L.used + i];
    } else if (L.type == 1) {
        const uint8_t v = L.raw[0];
        for (int64_t i = lane; i < k; i += nl) o.out[o.pos + i] = v;
    } else {
        for (int64_t i = 0; i < k; i++) {
            uint8_t s;
            const int rc = lit_huf_one(L, T, &s);
            if (rc) return rc;
            if (lane == 0) o.out[o.pos + i] = s;
        }
    }
    L.used += k;
    o.pos += k;
    return done;
}

VBZ_HD int emit_match(Out& o, int64_t off, int64_t len, int lane, int nl) {
    if (off < 1 || off > o.pos) return -ST_CORRUPT;
    int64_t k = len;
    int done = 0;
    if (o.pos + k > o.stop) {
        if (o.cap_bound) return -ST_TOO_LARGE;
        k = o.stop - o.pos;
        done = 1;
    }
    warp_sync();   // the bytes copied from were written by any lane
    const int64_t src = o.pos - off;
    for (int64_t i = lane; i < k; i += nl) o.out[o.pos + i] = o.out[src + (i < off ? i : i % off)];
    warp_sync();
    o.pos += k;
    return done;
}

struct FrameState {
    int huf_bits;                  // 0: no Huffman table yet (treeless literals are corrupt)
    int al_ll, al_of, al_ml;       // -1: no table yet (repeat mode is corrupt)
    uint32_t rep[3];
};

// literals section at p (n bytes left in the block).  Returns bytes consumed or -status.
VBZ_HD int64_t read_literals(const uint8_t* p, int64_t n, Tables& T, FrameState& F, LitSrc& L, int lane, int nl) {
    if (n < 1) return -ST_CORRUPT;
    const int type = p[0] & 3, sf = (p[0] >> 2) & 3;
    L.used = 0;
    if (type < 2) {
        int64_t rs, hs;
        if (sf == 0 || sf == 2) {
            rs = p[0] >> 3;
            hs = 1;
        } else if (sf == 1) {
            if (n < 2) return -ST_CORRUPT;
            rs = (p[0] >> 4) + ((int64_t)p[1] << 4);
            hs = 2;
        } else {
            if (n < 3) return -ST_CORRUPT;
            rs = (p[0] >> 4) + ((int64_t)p[1] << 4) + ((int64_t)p[2] << 12);
            hs = 3;
        }
        if (rs > BLOCK_MAX) return -ST_CORRUPT;
        const int64_t body = type == 0 ? rs : 1;
        if (hs + body > n) return -ST_CORRUPT;
        L.type = type;
        L.raw = p + hs;
        L.size = rs;
        return hs + body;
    }
    int64_t rs, cs, hs;
    int ns = sf == 0 ? 1 : 4;
    if (sf < 2) {
        if (n < 3) return -ST_CORRUPT;
        const uint32_t v = rd_le(p, 3);
        rs = (v >> 4) & 0x3ff;
        cs = (v >> 14) & 0x3ff;
        hs = 3;
    } else if (sf == 2) {
        if (n < 4) return -ST_CORRUPT;
        const uint32_t v = rd_le(p, 4);
        rs = (v >> 4) & 0x3fff;
        cs = (v >> 18) & 0x3fff;
        hs = 4;
    } else {
        if (n < 5) return -ST_CORRUPT;
        const uint64_t v = rd_le(p, 4) | ((uint64_t)p[4] << 32);
        rs = (int64_t)((v >> 4) & 0x3ffff);
        cs = (int64_t)((v >> 22) & 0x3ffff);
        hs = 5;
    }
    if (rs > BLOCK_MAX || hs + cs > n) return -ST_CORRUPT;
    const uint8_t* q = p + hs;
    int64_t qn = cs;
    if (type == 2) {
        int mb = 0;
        const int used = huf_read(q, qn, T, &mb, lane, nl);
        if (used < 0) return used == -ST_TRUNCATED ? -ST_CORRUPT : used;
        F.huf_bits = mb;
        q += used;
        qn -= used;
    } else if (F.huf_bits == 0) {
        return -ST_CORRUPT;
    }
    L.type = 2;
    L.size = rs;
    L.mb = F.huf_bits;
    L.nstreams = ns;
    L.cur = -1;
    L.left = 0;
    if (ns == 1) {
        L.sp[0] = q;
        L.sn[0] = qn;
        L.quota[0] = rs;
    } else {
        if (qn < 6) return -ST_CORRUPT;
        const int64_t s1 = rd_le(q, 2), s2 = rd_le(q + 2, 2), s3 = rd_le(q + 4, 2);
        const int64_t s4 = qn - 6 - s1 - s2 - s3;
        if (s4 < 1) return -ST_CORRUPT;
        const int64_t seg = (rs + 3) / 4;
        if (rs - 3 * seg < 0) return -ST_CORRUPT;
        const uint8_t* b = q + 6;
        L.sp[0] = b; L.sn[0] = s1;
        L.sp[1] = b + s1; L.sn[1] = s2;
        L.sp[2] = b + s1 + s2; L.sn[2] = s3;
        L.sp[3] = b + s1 + s2 + s3; L.sn[3] = s4;
        L.quota[0] = L.quota[1] = L.quota[2] = seg;
        L.quota[3] = rs - 3 * seg;
    }
    return hs + cs;
}

// one of the three sequence tables (built by lane 0; fse_build cannot fail on counts that fse_read_ncount accepted:
// they sum to the table size, so the spread returns to 0).  Returns bytes consumed or -status.
VBZ_HD int read_seq_table(const uint8_t* p, int64_t n, int mode, int which, FseEntry* t, int* al, Tables& T, int lane) {
    const int max_al = which == 1 ? OF_MAX_AL : LL_MAX_AL, max_sym = which == 0 ? LL_MAX_SYM : (which == 1 ? OF_MAX_SYM : ML_MAX_SYM);
    int used = 0;
    if (mode == 0) {
        if (lane == 0) fse_predefined(t, which, T.norm, T.next);
        *al = which == 1 ? 5 : 6;
    } else if (mode == 1) {
        if (n < 1 || p[0] > max_sym) return -ST_CORRUPT;
        if (lane == 0) fse_rle(t, p[0]);
        *al = 0;
        used = 1;
    } else if (mode == 2) {
        int nsym = 0, a = 0;
        used = fse_read_ncount(p, n, max_al, max_sym, T.norm, &nsym, &a);
        if (used < 0) return -ST_CORRUPT;
        warp_sync();
        if (lane == 0) fse_build(t, T.norm, nsym, a, T.next);
        *al = a;
    } else if (*al < 0) {
        return -ST_CORRUPT;   // repeat mode without a previous table
    }
    warp_sync();   // T.norm / T.next are reused by the next table
    return used;
}

VBZ_HD int decode_sequences(const uint8_t* p, int64_t n, Tables& T, FrameState& F, LitSrc& L, Out& o, int lane, int nl) {
    static constexpr uint32_t LL_BASE[36] = {0, 1, 2, 3, 4, 5, 6, 7, 8, 9, 10, 11, 12, 13, 14, 15, 16, 18, 20, 22, 24, 28, 32, 40,
                                             48, 64, 128, 256, 512, 1024, 2048, 4096, 8192, 16384, 32768, 65536};
    static constexpr uint8_t LL_BITS[36] = {0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 1, 1, 1, 1, 2, 2, 3, 3,
                                            4, 6, 7, 8, 9, 10, 11, 12, 13, 14, 15, 16};
    static constexpr uint32_t ML_BASE[53] = {3, 4, 5, 6, 7, 8, 9, 10, 11, 12, 13, 14, 15, 16, 17, 18, 19, 20, 21, 22, 23, 24, 25, 26,
                                             27, 28, 29, 30, 31, 32, 33, 34, 35, 37, 39, 41, 43, 47, 51, 59, 67, 83, 99, 131, 259, 515,
                                             1027, 2051, 4099, 8195, 16387, 32771, 65539};
    static constexpr uint8_t ML_BITS[53] = {0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0,
                                            0, 0, 0, 0, 0, 1, 1, 1, 1, 2, 2, 3, 3, 4, 4, 5, 7, 8, 9, 10, 11, 12, 13, 14, 15, 16};
    if (n < 1) return -ST_CORRUPT;
    int64_t nseq, q;
    if (p[0] < 128) {
        nseq = p[0];
        q = 1;
    } else if (p[0] < 255) {
        if (n < 2) return -ST_CORRUPT;
        nseq = ((int64_t)(p[0] - 128) << 8) + p[1];
        q = 2;
    } else {
        if (n < 3) return -ST_CORRUPT;
        nseq = p[1] + ((int64_t)p[2] << 8) + 0x7f00;
        q = 3;
    }
    if (nseq == 0) {
        if (q != n) return -ST_CORRUPT;
        return emit_literals(L, T, o, L.size - L.used, lane, nl);
    }
    if (q >= n) return -ST_CORRUPT;
    const int modes = p[q++];
    if (modes & 3) return -ST_RESERVED;
    int used = read_seq_table(p + q, n - q, (modes >> 6) & 3, 0, T.ll, &F.al_ll, T, lane);
    if (used < 0) return used;
    q += used;
    used = read_seq_table(p + q, n - q, (modes >> 4) & 3, 1, T.of, &F.al_of, T, lane);
    if (used < 0) return used;
    q += used;
    used = read_seq_table(p + q, n - q, (modes >> 2) & 3, 2, T.ml, &F.al_ml, T, lane);
    if (used < 0) return used;
    q += used;
    warp_sync();
    RevBits bs;
    if (!bs.init(p + q, n - q)) return -ST_CORRUPT;
    uint32_t sll = bs.read(F.al_ll), sof = bs.read(F.al_of), sml = bs.read(F.al_ml);
    for (int64_t i = 0; i < nseq; i++) {
        const FseEntry eo = T.of[sof], em = T.ml[sml], el = T.ll[sll];
        const int ofc = eo.sym;
        if (ofc > OF_MAX_SYM || em.sym > ML_MAX_SYM || el.sym > LL_MAX_SYM) return -ST_CORRUPT;
        const uint64_t ofv = (1ull << ofc) + bs.read(ofc);
        const int64_t ml = ML_BASE[em.sym] + bs.read(ML_BITS[em.sym]);
        const int64_t ll = LL_BASE[el.sym] + bs.read(LL_BITS[el.sym]);
        if (i + 1 < nseq) {
            sll = el.base + bs.read(el.nb);
            sml = em.base + bs.read(em.nb);
            sof = eo.base + bs.read(eo.nb);
        }
        if (bs.pos < 0) return -ST_CORRUPT;
        uint64_t off;
        if (ofv > 3) {
            off = ofv - 3;
            F.rep[2] = F.rep[1];
            F.rep[1] = F.rep[0];
            F.rep[0] = (uint32_t)off;
        } else {
            const int idx = (int)ofv + (ll == 0 ? 1 : 0);   // 1..4
            if (idx == 1) {
                off = F.rep[0];
            } else if (idx == 2) {
                off = F.rep[1];
                F.rep[1] = F.rep[0];
                F.rep[0] = (uint32_t)off;
            } else {
                off = idx == 3 ? F.rep[2] : (uint64_t)F.rep[0] - 1;
                if (off == 0) return -ST_CORRUPT;
                F.rep[2] = F.rep[1];
                F.rep[1] = F.rep[0];
                F.rep[0] = (uint32_t)off;
            }
        }
        int rc = emit_literals(L, T, o, ll, lane, nl);
        if (rc) return rc;
        rc = emit_match(o, (int64_t)off, ml, lane, nl);
        if (rc) return rc;
    }
    if (bs.pos != 0) return -ST_CORRUPT;
    return emit_literals(L, T, o, L.size - L.used, lane, nl);
}

// One frame: src[0, n) -> out[0, produced).  Decoding stops once min(limit, cap) bytes exist; content beyond `cap`
// when limit > cap, or a Frame_Content_Size above content_max, is ST_TOO_LARGE.  Returns the status.
VBZ_HD int decode_frame(const uint8_t* src, int64_t n, uint8_t* out, int64_t cap, int64_t limit, int64_t content_max,
                        int64_t* produced, Tables& T, int lane, int nl) {
    *produced = 0;
    if (n < 4) return ST_TRUNCATED;
    const uint32_t magic = rd_le(src, 4);
    if ((magic & 0xfffffff0u) == 0x184d2a50u) return ST_FRAMES;
    if (magic != 0xfd2fb528u) return ST_BAD_MAGIC;
    if (n < 5) return ST_TRUNCATED;
    const int fhd = src[4];
    const int fcs_flag = fhd >> 6, single = (fhd >> 5) & 1, did_flag = fhd & 3;
    if (fhd & 8) return ST_RESERVED;
    if (fhd & 4) return ST_CHECKSUM;
    int64_t p = 5;
    if (!single) p++;
    const int did_size = did_flag == 3 ? 4 : did_flag;
    const int fcs_size = fcs_flag == 0 ? single : (1 << fcs_flag);
    if (p + did_size + fcs_size > n) return ST_TRUNCATED;
    if (did_size && rd_le(src + p, did_size) != 0) return ST_DICTIONARY;
    p += did_size;
    int64_t fcs = -1;
    if (fcs_size) {
        uint64_t v = rd_le(src + p, fcs_size < 4 ? fcs_size : 4);
        if (fcs_size == 8) v |= (uint64_t)rd_le(src + p + 4, 4) << 32;
        if (fcs_size == 2) v += 256;
        if (v > (uint64_t)INT64_MAX) return ST_TOO_LARGE;
        fcs = (int64_t)v;
        p += fcs_size;
    }
    if (fcs > content_max) return ST_TOO_LARGE;
    Out o{out, 0, limit < cap ? limit : cap, limit > cap};
    if (fcs >= 0 && fcs > cap && o.cap_bound) return ST_TOO_LARGE;
    FrameState F{0, -1, -1, -1, {1, 4, 8}};
    while (true) {
        if (o.pos >= o.stop && !o.cap_bound) {
            *produced = o.pos;
            return ST_OK;
        }
        if (p + 3 > n) return ST_TRUNCATED;
        const uint32_t bh = rd_le(src + p, 3);
        p += 3;
        const int last = bh & 1, bt = (bh >> 1) & 3;
        const int64_t bsz = bh >> 3;
        if (bt == 3) return ST_RESERVED;
        if (bsz > BLOCK_MAX) return ST_CORRUPT;
        const int64_t in_sz = bt == 1 ? 1 : bsz;
        if (p + in_sz > n) return ST_TRUNCATED;
        const int64_t block_start = o.pos;
        int rc = 0;
        if (bt < 2) {
            LitSrc L{};
            L.type = bt;
            L.raw = src + p;
            L.size = bsz;
            rc = emit_literals(L, T, o, bsz, lane, nl);
        } else {
            LitSrc L{};
            const int64_t used = read_literals(src + p, bsz, T, F, L, lane, nl);
            if (used < 0) return (int)-used;
            rc = decode_sequences(src + p + used, bsz - used, T, F, L, o, lane, nl);
        }
        if (rc < 0) return -rc;
        if (rc == 1) {
            *produced = o.pos;
            return ST_OK;
        }
        if (o.pos - block_start > BLOCK_MAX) return ST_CORRUPT;
        p += in_sz;
        if (last) break;
    }
    warp_sync();
    if (fcs >= 0 && o.pos != fcs) return ST_CORRUPT;
    if (p != n) return ST_FRAMES;
    *produced = o.pos;
    return ST_OK;
}

// ---- streamvbyte-16 -> int16 samples ------------------------------------------------------------------------------
// Decoded chunk layout: ceil(s/8) key bytes (one bit per sample, LSB first: 0 = 1 data byte, 1 = 2 bytes little endian),
// then the data bytes.  Value u -> zig-zag -> delta; the running sum restarts at 0 for every chunk and wraps like int16.

// bytes of the first t samples' data, given their key bytes (the bits of samples >= t masked off)
VBZ_HD int svb16_key_width(uint8_t key, int nsamp) {   // nsamp in [0, 8]
    const uint32_t m = nsamp >= 8 ? 0xffu : ((1u << nsamp) - 1);
#ifdef __CUDA_ARCH__
    return nsamp + __popc(key & m);
#else
    return nsamp + __builtin_popcount(key & m);
#endif
}

// nsamp (<= 8) samples from data at byte d (widths from key), zig-zag decoded and summed into `acc` (int16 wrap);
// writes the running sums to out.  Returns the number of data bytes used.
VBZ_HD int svb16_decode8(const uint8_t* data, uint8_t key, int nsamp, uint16_t acc, int16_t* out) {
    int d = 0;
    for (int i = 0; i < nsamp; i++) {
        uint32_t u = data[d++];
        if ((key >> i) & 1) u |= (uint32_t)data[d++] << 8;
        const int32_t zz = (int32_t)(u >> 1) ^ -(int32_t)(u & 1);
        acc = (uint16_t)(acc + (uint16_t)zz);
        out[i] = (int16_t)acc;
    }
    return d;
}

VBZ_HD uint16_t svb16_delta_sum8(const uint8_t* data, uint8_t key, int nsamp) {
    int d = 0;
    uint16_t acc = 0;
    for (int i = 0; i < nsamp; i++) {
        uint32_t u = data[d++];
        if ((key >> i) & 1) u |= (uint32_t)data[d++] << 8;
        acc = (uint16_t)(acc + (uint16_t)((int32_t)(u >> 1) ^ -(int32_t)(u & 1)));
    }
    return acc;
}

}  // namespace vbz
}  // namespace wdx
