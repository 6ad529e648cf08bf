// LZ4 frame format (magic 0x184D2204) with LZ4 blocks: Kafka compression codec 3 of a RecordBatch's records section.
//
// Written __host__ __device__ so that the CPU test build compiles the same source.  Message format v2 writes the frame
// as published, with the correct header checksum.  Every flag combination a producer can set is accepted:
//   independent or linked blocks, block checksums on / off, content size present / absent, content checksum on / off,
//   uncompressed blocks (bit 31 of the block size), block maximum 64 KB, 256 KB, 1 MB or 4 MB.
// Rejected: a wrong version or reserved bit, a DictID, a wrong header-checksum byte, offset 0, an offset reaching before
// the frame's output (before the block's output when blocks are independent), a literal run past the end of its block,
// a block expanding past its block maximum or past the output slot, a wrong XXH32 block or content checksum, a stored
// content size that disagrees with the blocks, and bytes after the frame.
//
// ck_lz4_frame<false> is the size pass: it walks the tokens only (no output, no checksums) and returns the decompressed
// size; ck_lz4_frame<true> decodes into a slot of exactly that size and checks every checksum.
#ifndef CK_LZ4_CUH
#define CK_LZ4_CUH

#define CK_XXH_P1 2654435761u
#define CK_XXH_P2 2246822519u
#define CK_XXH_P3 3266489917u
#define CK_XXH_P4 668265263u
#define CK_XXH_P5 374761393u

CK_HD u32 ck_rotl32(u32 x, u32 r) { return (x << r) | (x >> (32u - r)); }
CK_HD u32 ck_xxh_round(u32 acc, u32 in) { acc += in * CK_XXH_P2; return ck_rotl32(acc, 13) * CK_XXH_P1; }

// XXH32 of p[0..n) with seed 0
CK_HD u32 ck_xxh32(const u8* p, u32 n) {
    const u8* end = p + n;
    u32 h;
    if (n >= 16) {
        u32 v1 = CK_XXH_P1 + CK_XXH_P2, v2 = CK_XXH_P2, v3 = 0, v4 = 0u - CK_XXH_P1;
        for (; p + 16 <= end; p += 16) {
            v1 = ck_xxh_round(v1, ck_le32(p)); v2 = ck_xxh_round(v2, ck_le32(p + 4));
            v3 = ck_xxh_round(v3, ck_le32(p + 8)); v4 = ck_xxh_round(v4, ck_le32(p + 12));
        }
        h = ck_rotl32(v1, 1) + ck_rotl32(v2, 7) + ck_rotl32(v3, 12) + ck_rotl32(v4, 18);
    } else {
        h = CK_XXH_P5;
    }
    h += n;
    for (; p + 4 <= end; p += 4) h = ck_rotl32(h + ck_le32(p) * CK_XXH_P3, 17) * CK_XXH_P4;
    for (; p < end; p++) h = ck_rotl32(h + (u32)*p * CK_XXH_P5, 11) * CK_XXH_P1;
    h ^= h >> 15; h *= CK_XXH_P2; h ^= h >> 13; h *= CK_XXH_P3; h ^= h >> 16;
    return h;
}

// one compressed block src[0..n) whose output starts at dst[op]; the output may not pass dst[lim] and a match may not
// reach before dst[lo].  W = false: no bytes are written (size pass).
template <bool W>
CK_HD bool ck_lz4_block(const u8* src, u32 n, u8* dst, u32& op, u32 lim, u32 lo) {
    u32 ip = 0;
    if (!n) return false;
    for (;;) {
        u32 tok = src[ip++];
        u32 lit = tok >> 4;
        if (lit == 15) {
            u32 b;
            do { if (ip >= n) return false; b = src[ip++]; lit += b; } while (b == 255 && lit < 0x7fffffffu);
        }
        if (lit > n - ip || lit > lim - op) return false;
        if (W) for (u32 k = 0; k < lit; k++) dst[op + k] = src[ip + k];
        ip += lit; op += lit;
        if (ip == n) return true;                                    // the last sequence has no match
        if (ip + 2 > n) return false;
        u32 off = (u32)src[ip] | ((u32)src[ip + 1] << 8);
        ip += 2;
        if (off == 0 || off > op - lo) return false;
        u32 ml = tok & 15u;
        if (ml == 15) {
            u32 b;
            do { if (ip >= n) return false; b = src[ip++]; ml += b; } while (b == 255 && ml < 0x7fffffffu);
        }
        ml += 4;
        if (ml > lim - op) return false;
        if (W) { const u8* from = dst + op - off; u8* to = dst + op; for (u32 k = 0; k < ml; k++) to[k] = from[k]; }
        op += ml;
        if (ip >= n) return false;                                   // a block ends with literals
    }
}

// the frame src[0..n).  W = false: size pass, out_size = decompressed size.  W = true: decode into dst[0..out_size).
template <bool W>
CK_HD bool ck_lz4_frame(const u8* src, u32 n, u8* dst, u32& out_size) {
    if (n < 7 || ck_le32(src) != 0x184D2204u) return false;
    u32 flg = src[4], bd = src[5];
    if ((flg >> 6) != 1 || (flg & 2u) || (flg & 1u) || (bd & 0x8fu)) return false;     // version 01, reserved, DictID
    u32 bsize_id = (bd >> 4) & 7u;
    if (bsize_id < 4) return false;
    u32 bmax = 1u << (8 + 2 * bsize_id);                                              // 4: 64 KB ... 7: 4 MB
    bool indep = flg & 0x20u, bsum = flg & 0x10u, csize = flg & 0x08u, csum = flg & 0x04u;
    u32 pos = 6;
    unsigned long long stored = 0;
    if (csize) {
        if (n < 15) return false;
        for (int k = 7; k >= 0; k--) stored = (stored << 8) | src[pos + k];
        pos += 8;
    }
    if (((ck_xxh32(src + 4, pos - 4) >> 8) & 0xffu) != src[pos]) return false;        // header checksum
    pos++;
    u32 cap = W ? out_size : 0x7fffffffu;
    u32 op = 0;
    for (;;) {
        if (pos + 4 > n) return false;
        u32 bs = ck_le32(src + pos);
        pos += 4;
        if (!bs) break;                                                               // EndMark
        bool raw = bs >> 31;
        bs &= 0x7fffffffu;
        if (bs > bmax || bs > n - pos) return false;
        if (bsum && (n - pos - bs < 4 || (W && ck_xxh32(src + pos, bs) != ck_le32(src + pos + bs)))) return false;
        u32 lim = cap - op < bmax ? cap : op + bmax;                                  // the block's own maximum, and the slot
        if (raw) {
            if (bs > lim - op) return false;
            if (W) for (u32 k = 0; k < bs; k++) dst[op + k] = src[pos + k];
            op += bs;
        } else if (!ck_lz4_block<W>(src + pos, bs, dst, op, lim, indep ? op : 0u)) {
            return false;
        }
        pos += bs + (bsum ? 4u : 0u);
    }
    if (csum) {
        if (pos + 4 > n) return false;
        if (W && ck_xxh32(dst, op) != ck_le32(src + pos)) return false;
        pos += 4;
    }
    if (pos != n) return false;                                                       // nothing may follow the frame
    if (csize && stored != op) return false;
    if (W) return op == out_size;
    out_size = op;
    return true;
}

#endif  // CK_LZ4_CUH
