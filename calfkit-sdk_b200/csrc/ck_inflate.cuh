// gzip (RFC 1952) around DEFLATE (RFC 1951): Kafka compression codec 1 of a RecordBatch's records section.
//
// Written __host__ __device__ (like the walker) so that the CPU test build compiles the same source.  One call decodes
// one gzip member into a slot whose size the caller took from the trailer's ISIZE (ck_gzip_isize) beforehand:
//   header   ID1 ID2 = 1f 8b, CM = 8; FEXTRA / FNAME / FCOMMENT / FHCRC are skipped (the header CRC is not checked);
//            reserved flag bits set -> rejected
//   blocks   stored, fixed Huffman, dynamic Huffman; a distance may reach back to the first byte of the member's output
//   trailer  CRC-32 (IEEE) of the output and ISIZE must both match, and the output must fill the slot exactly
// A records section is exactly ONE member: bytes after its trailer make the frame bad.  (RFC 1952 allows concatenated
// members, but no Kafka producer writes them, and accepting them would let a frame carry data its ISIZE does not cover.)
//
// Huffman codes are decoded canonically: per code length, how many codes there are and the symbols in code order
// (count[16] / sym[]); a symbol costs one step per bit of its code.  State lives in the calling thread.
#ifndef CK_INFLATE_CUH
#define CK_INFLATE_CUH

#define CK_INF_MAXBITS 15
#define CK_INF_NLIT 288
#define CK_INF_NDIST 32

struct ck_inf_bits {
    const u8* p; u32 n, pos;                      // input p[0..n); pos = next byte to load (may run past n: zeros are loaded)
    unsigned long long buf; u32 cnt;
    CK_HD u32 need(u32 k) {                       // the next k bits (k <= 32), LSB first, not consumed
        while (cnt < k) {
            u32 b = pos < n ? p[pos] : 0u;
            pos++;
            buf |= (unsigned long long)b << cnt; cnt += 8;
        }
        return (u32)(buf & ((1ull << k) - 1));
    }
    CK_HD void drop(u32 k) { buf >>= k; cnt -= k; }
    CK_HD u32 get(u32 k) { u32 v = need(k); drop(k); return v; }
    CK_HD void align() { u32 r = cnt & 7u; drop(r); }           // to the next byte boundary of the input
    CK_HD u32 byte_pos() const { return pos - cnt / 8u; }       // input position of the next unconsumed whole byte
    CK_HD bool over() const { return (unsigned long long)pos * 8u - cnt > (unsigned long long)n * 8u; }   // consumed past the end
};

struct ck_inf_huff { unsigned short count[CK_INF_MAXBITS + 1]; unsigned short sym[CK_INF_NLIT]; };

// canonical code from code lengths.  0 = complete; 1 = incomplete; -1 = over-subscribed.
CK_HD int ck_inf_build(ck_inf_huff& h, const unsigned char* len, u32 n) {
    for (u32 b = 0; b <= CK_INF_MAXBITS; b++) h.count[b] = 0;
    for (u32 s = 0; s < n; s++) h.count[len[s]]++;
    unsigned short offs[CK_INF_MAXBITS + 1];
    int left = 1;
    offs[1] = 0;
    for (u32 b = 1; b <= CK_INF_MAXBITS; b++) {
        left = 2 * left - h.count[b];
        if (left < 0) return -1;
        if (b < CK_INF_MAXBITS) offs[b + 1] = offs[b] + h.count[b];
    }
    for (u32 s = 0; s < n; s++) if (len[s]) h.sym[offs[len[s]]++] = (unsigned short)s;
    return left > 0 ? 1 : 0;
}
// zlib's rule: an incomplete code is acceptable only when it is a single code of one bit (or no code at all)
CK_HD bool ck_inf_usable(const ck_inf_huff& h, int r) {
    if (r < 0) return false;
    if (r == 0) return true;
    u32 used = 0;
    for (u32 b = 1; b <= CK_INF_MAXBITS; b++) used += h.count[b];
    return used == 0 || (used == 1 && h.count[1] == 1);
}

// one symbol, or -1 for a code that is not in the table
CK_HD int ck_inf_decode(ck_inf_bits& in, const ck_inf_huff& h) {
    u32 bits = in.need(CK_INF_MAXBITS);
    int code = 0, first = 0, index = 0;
    for (u32 b = 1; b <= CK_INF_MAXBITS; b++) {
        code |= (int)((bits >> (b - 1)) & 1u);
        int c = h.count[b];
        if (code - first < c) { in.drop(b); return h.sym[index + code - first]; }
        index += c; first += c; first <<= 1; code <<= 1;
    }
    return -1;
}

// literal / length and distance codes of one block until end-of-block; false on any error
CK_HD bool ck_inf_codes(ck_inf_bits& in, const ck_inf_huff& lit, const ck_inf_huff& dist, u8* dst, u32 cap, u32& op) {
    for (;;) {
        int s = ck_inf_decode(in, lit);
        if (s < 0 || in.over()) return false;
        if (s < 256) {
            if (op >= cap) return false;
            dst[op++] = (u8)s;
            continue;
        }
        if (s == 256) return true;
        s -= 257;
        if (s >= 29) return false;                                   // 286, 287: no such length
        u32 len;
        if (s < 8) len = (u32)s + 3;
        else if (s == 28) len = 258;
        else { u32 e = (u32)(s - 4) / 4; len = ((4u + ((u32)s & 3u)) << e) + 3u + in.get(e); }
        int d = ck_inf_decode(in, dist);
        if (d < 0 || d >= 30) return false;                          // 30, 31: no such distance
        u32 dd;
        if (d < 4) dd = (u32)d + 1;
        else { u32 e = (u32)d / 2 - 1; dd = ((2u + ((u32)d & 1u)) << e) + 1u + in.get(e); }
        if (in.over() || dd > op || len > cap - op) return false;
        const u8* from = dst + op - dd;
        u8* to = dst + op;
        for (u32 k = 0; k < len; k++) to[k] = from[k];               // byte order matters: a match may overlap itself
        op += len;
    }
}

CK_HD u32 ck_le32(const u8* p) { return (u32)p[0] | ((u32)p[1] << 8) | ((u32)p[2] << 16) | ((u32)p[3] << 24); }

// the decompressed size a gzip member declares (ISIZE, its last four bytes); false if it cannot be a gzip member or
// declares more than DEFLATE can expand n bytes to (258 bytes per bit of input: 1032:1)
CK_HD bool ck_gzip_isize(const u8* src, u32 n, u32& isize) {
    if (n < 18 || src[0] != 0x1f || src[1] != 0x8b || src[2] != 8) return false;
    isize = ck_le32(src + n - 4);
    return (unsigned long long)isize <= 1032ull * n;
}

// skip the member header; position of the DEFLATE stream, or 0 on error
CK_HD u32 ck_gzip_header(const u8* src, u32 n) {
    if (n < 18 || src[0] != 0x1f || src[1] != 0x8b || src[2] != 8) return 0;
    u8 flg = src[3];
    if (flg & 0xe0) return 0;                                        // reserved bits
    u32 pos = 10;                                                    // MTIME XFL OS
    if (flg & 4) {                                                   // FEXTRA
        if (pos + 2 > n) return 0;
        u32 xlen = (u32)src[pos] | ((u32)src[pos + 1] << 8);
        pos += 2 + xlen;
        if (pos > n) return 0;
    }
    if (flg & 8) { while (pos < n && src[pos]) pos++; if (pos >= n) return 0; pos++; }    // FNAME
    if (flg & 16) { while (pos < n && src[pos]) pos++; if (pos >= n) return 0; pos++; }   // FCOMMENT
    if (flg & 2) pos += 2;                                           // FHCRC
    return pos + 8 <= n ? pos : 0;
}

// inflate the member src[0..n) into dst[0..cap), cap = its ISIZE.  crc_tab: slicing-by-4 tables of CK_CRC32_POLY.
// true iff the member is well formed, fills dst exactly, its CRC-32 and ISIZE match and nothing follows it.
CK_HD bool ck_gunzip(const u8* src, u32 n, u8* dst, u32 cap, const u32* crc_tab) {
    u32 start = ck_gzip_header(src, n);
    if (!start) return false;
    ck_inf_bits in; in.p = src; in.n = n - 8; in.pos = start; in.buf = 0; in.cnt = 0;   // the trailer is not DEFLATE input
    ck_inf_huff lit, dist;
    u32 op = 0;
    u32 last;
    do {
        last = in.get(1);
        u32 type = in.get(2);
        if (in.over()) return false;
        if (type == 0) {                                             // stored
            in.align();
            u32 p = in.byte_pos();
            in.buf = 0; in.cnt = 0; in.pos = p;
            if (p + 4 > in.n) return false;
            u32 len = (u32)src[p] | ((u32)src[p + 1] << 8), nlen = (u32)src[p + 2] | ((u32)src[p + 3] << 8);
            if ((len ^ 0xffffu) != nlen) return false;
            p += 4;
            if (len > in.n - p || len > cap - op) return false;
            for (u32 k = 0; k < len; k++) dst[op + k] = src[p + k];
            op += len; in.pos = p + len;
        } else if (type == 1) {                                      // fixed Huffman
            unsigned char l[CK_INF_NLIT];
            u32 s = 0;
            for (; s < 144; s++) l[s] = 8;
            for (; s < 256; s++) l[s] = 9;
            for (; s < 280; s++) l[s] = 7;
            for (; s < CK_INF_NLIT; s++) l[s] = 8;
            ck_inf_build(lit, l, CK_INF_NLIT);
            for (s = 0; s < 30; s++) l[s] = 5;
            ck_inf_build(dist, l, 30);
            if (!ck_inf_codes(in, lit, dist, dst, cap, op)) return false;
        } else if (type == 2) {                                      // dynamic Huffman
            u32 nlen = in.get(5) + 257, ndist = in.get(5) + 1, ncode = in.get(4) + 4;
            if (in.over() || nlen > 286 || ndist > 30) return false;
            const unsigned char order[19] = {16, 17, 18, 0, 8, 7, 9, 6, 10, 5, 11, 4, 12, 3, 13, 2, 14, 1, 15};
            unsigned char l[CK_INF_NLIT + CK_INF_NDIST];
            for (u32 k = 0; k < 19; k++) l[order[k]] = k < ncode ? (unsigned char)in.get(3) : 0;
            if (in.over() || ck_inf_build(lit, l, 19) != 0) return false;   // the code-length code must be complete
            u32 k = 0;
            while (k < nlen + ndist) {
                int s = ck_inf_decode(in, lit);
                if (s < 0 || in.over()) return false;
                if (s < 16) { l[k++] = (unsigned char)s; continue; }
                u32 rep; unsigned char v = 0;
                if (s == 16) { if (!k) return false; v = l[k - 1]; rep = 3 + in.get(2); }
                else if (s == 17) rep = 3 + in.get(3);
                else rep = 11 + in.get(7);
                if (in.over() || k + rep > nlen + ndist) return false;
                while (rep--) l[k++] = v;
            }
            if (!l[256]) return false;                               // no end-of-block code
            if (!ck_inf_usable(lit, ck_inf_build(lit, l, nlen))) return false;
            if (!ck_inf_usable(dist, ck_inf_build(dist, l + nlen, ndist))) return false;
            if (!ck_inf_codes(in, lit, dist, dst, cap, op)) return false;
        } else {
            return false;
        }
        if (in.over()) return false;
    } while (!last);
    in.align();
    u32 p = in.byte_pos();
    if (p != n - 8 || op != cap) return false;                       // exactly one member, exactly ISIZE bytes
    if (ck_le32(src + p + 4) != cap) return false;
    return ck_crc_span(crc_tab, dst, cap) == ck_le32(src + p);
}

#endif  // CK_INFLATE_CUH
