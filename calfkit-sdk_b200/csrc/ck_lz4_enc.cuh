// LZ4 block encoder, and the greedy LZ77 parse it shares with the DEFLATE encoder (ck_deflate.cuh): Kafka compression
// codec 3 on the produce side.  Written __host__ __device__ like the decoders, so that the CPU test build compiles the
// same source.  One call compresses one chunk of at most 64 KB; the caller owns the hash table (1 << bits entries of u32,
// initialised here, so that the output depends on the input alone).
//
// Parse: one probe per position into a hash table of 4-byte values (the most recent position wins), a match is taken
// when its first 4 bytes agree and is extended byte by byte; one position inside every match is re-entered.  After 64
// misses in a row the parse skips ahead faster (1 + misses / 64 bytes), which keeps incompressible input cheap.
//
// Block rules (LZ4 Block Format): the last 5 bytes are literals, no match starts in the last 12 bytes, offsets 1..65535.
// A chunk whose compressed form is not smaller than itself is stored raw (bit 31 of the block size).
#ifndef CK_LZ4_ENC_CUH
#define CK_LZ4_ENC_CUH

#define CK_LZ_EMPTY 0xffffffffu
#define CK_LZ4_TAB_BITS 12
#define CK_LZ4_FLG 0x60u             // version 01, independent blocks, no checksums, no content size
#define CK_LZ4_BD 0x40u              // 64 KB block maximum
#define CK_LZ4_HC 0x82u              // (XXH32(60 40) >> 8) & 0xff

CK_HD u32 ck_lz_hash(u32 v, u32 bits) { return (v * 2654435761u) >> (32u - bits); }

// greedy parse of w[start..end): positions are relative to the window base w, and w[0..start) is history that matches may
// reach into (no further than max_dist).  A match starts below mf_end (<= end - 3), ends at or before m_end and is at most
// max_len long.  The sink gets f.seq(literal start, literal length, offset, match length) in order, the last call with
// match length 0, and may stop the parse by clearing f.ok.
template <class Sink>
CK_HD void ck_lz_parse(const u8* w, u32 start, u32 end, u32 mf_end, u32 m_end, u32 max_dist, u32 max_len, u32* tab, u32 bits,
                       Sink& f) {
    for (u32 i = 0; i < (1u << bits); i++) tab[i] = CK_LZ_EMPTY;
    for (u32 p = start > max_dist ? start - max_dist : 0; p < start && p + 4 <= end; p++) tab[ck_lz_hash(ck_le32(w + p), bits)] = p;
    u32 anchor = start, ip = start, miss = 0;
    while (ip < mf_end) {
        u32 cur = ck_le32(w + ip);
        u32 h = ck_lz_hash(cur, bits), cand = tab[h];
        tab[h] = ip;
        if (cand != CK_LZ_EMPTY && ip - cand <= max_dist && ck_le32(w + cand) == cur) {
            u32 lim = m_end - ip < max_len ? m_end - ip : max_len, ml = 4;
            while (ml < lim && w[cand + ml] == w[ip + ml]) ml++;
            f.seq(anchor, ip - anchor, ip - cand, ml);
            if (!f.ok) return;
            ip += ml; anchor = ip; miss = 0;
            if (ip - 2 < mf_end) tab[ck_lz_hash(ck_le32(w + ip - 2), bits)] = ip - 2;
        } else {
            ip += 1 + (miss++ >> 6);
        }
    }
    f.seq(anchor, end - anchor, 0, 0);
}

// LZ4 sequences into dst[0..cap); ok = false as soon as the next sequence would not fit
struct ck_lz4_sink {
    const u8* w; u8* dst; u32 op, cap; bool ok;
    CK_HD void seq(u32 lp, u32 ll, u32 off, u32 ml) {
        u32 m = ml ? ml - 4 : 0;
        u32 need = 1 + (ll >= 15 ? (ll - 15) / 255 + 1 : 0) + ll + (ml ? 2 + (m >= 15 ? (m - 15) / 255 + 1 : 0) : 0);
        if (need > cap - op) { ok = false; return; }
        dst[op++] = (u8)(((ll < 15 ? ll : 15) << 4) | (m < 15 ? m : 15));
        if (ll >= 15) { u32 r = ll - 15; for (; r >= 255; r -= 255) dst[op++] = 255; dst[op++] = (u8)r; }
        for (u32 k = 0; k < ll; k++) dst[op + k] = w[lp + k];
        op += ll;
        if (!ml) return;
        dst[op++] = (u8)off; dst[op++] = (u8)(off >> 8);
        if (m >= 15) { u32 r = m - 15; for (; r >= 255; r -= 255) dst[op++] = 255; dst[op++] = (u8)r; }
    }
};

// one LZ4 frame block for src[0..n), n <= 64 KB: the 4-byte block size, then the compressed block, or the raw bytes when
// compressing does not make them smaller.  Returns the bytes written (at most n + 4).  tab: 1 << CK_LZ4_TAB_BITS entries.
CK_HD u32 ck_lz4_enc_block(const u8* src, u32 n, u8* dst, u32* tab) {
    ck_lz4_sink f; f.w = src; f.dst = dst + 4; f.op = 0; f.cap = n ? n - 1 : 0; f.ok = n > 0;
    if (f.ok) ck_lz_parse(src, 0, n, n >= 13 ? n - 12 : 0, n >= 5 ? n - 5 : 0, 65535u, 0xffffffffu, tab, CK_LZ4_TAB_BITS, f);
    u32 bs = f.op;
    if (!f.ok) { for (u32 k = 0; k < n; k++) dst[4 + k] = src[k]; bs = n | 0x80000000u; }
    dst[0] = (u8)bs; dst[1] = (u8)(bs >> 8); dst[2] = (u8)(bs >> 16); dst[3] = (u8)(bs >> 24);
    return 4 + (bs & 0x7fffffffu);
}

// the frame around the blocks: magic + descriptor + header checksum (7 bytes) and the end mark (4 bytes)
CK_HD void ck_lz4_frame_head(u8* d) { d[0] = 0x04; d[1] = 0x22; d[2] = 0x4d; d[3] = 0x18; d[4] = CK_LZ4_FLG; d[5] = CK_LZ4_BD; d[6] = CK_LZ4_HC; }
#define CK_LZ4_HEAD 7u
#define CK_LZ4_TAIL 4u

#endif  // CK_LZ4_ENC_CUH
