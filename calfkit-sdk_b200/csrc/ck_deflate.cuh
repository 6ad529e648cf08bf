// DEFLATE (RFC 1951) encoder for the gzip members of Kafka compression codec 1 on the produce side.  Written
// __host__ __device__ like the decoder (ck_inflate.cuh), so that the CPU test build compiles the same source.
//
// A section is compressed in independent 64 KB chunks, as pigz does: each chunk becomes ONE non-final block with dynamic
// Huffman codes followed by an empty stored block (so that the next chunk starts on a byte), or non-final stored blocks
// when those are smaller.  Matches come from the greedy parse of ck_lz4_enc.cuh (minimum 4, maximum 258 bytes, distance up
// to 32 KB) and may reach into the previous chunk of the same section, whose bytes the caller passes as history.  The
// parse runs twice: once to count symbols, once to write them, so no symbol buffer is needed.
//
// Huffman code lengths are optimal (in-place Moffat-Katajainen over symbols sorted by frequency), then limited to 15 bits
// (7 for the code-length code) by pushing long codes up to the limit and lengthening the shortest codes until the Kraft
// sum is 1 again.  Every code has at least two symbols, so every code is complete.
#ifndef CK_DEFLATE_CUH
#define CK_DEFLATE_CUH

#include "ck_lz4_enc.cuh"

#define CK_DFL_TAB_BITS 13
#define CK_DFL_CHUNK 65536u
#define CK_GZ_HEAD 10u               // 1f 8b 08 00 00000000 00 ff
#define CK_GZ_TAIL 10u               // final empty fixed block 03 00, CRC-32, ISIZE

struct ck_bitw {
    u8* p; u32 op; unsigned long long buf; u32 cnt;
    CK_HD void put(u32 v, u32 n) {                       // n <= 32 bits, LSB first
        buf |= (unsigned long long)v << cnt; cnt += n;
        while (cnt >= 8) { p[op++] = (u8)buf; buf >>= 8; cnt -= 8; }
    }
    CK_HD void align() { if (cnt) put(0, 8 - cnt); }
};

CK_HD u32 ck_bitrev(u32 c, u32 n) { u32 r = 0; for (u32 k = 0; k < n; k++) { r = (r << 1) | (c & 1u); c >>= 1; } return r; }
CK_HD u32 ck_log2(u32 v) { u32 r = 0; while (v >>= 1) r++; return r; }

// length 3..258 -> symbol 257..285, extra bits, extra value
CK_HD void ck_dfl_len(u32 len, u32& sym, u32& eb, u32& ev) {
    u32 l = len - 3;
    if (len == 258) { sym = 285; eb = 0; ev = 0; }
    else if (l < 8) { sym = 257 + l; eb = 0; ev = 0; }
    else { u32 e = ck_log2(l) - 2; sym = 257 + 4 * (e + 1) + ((l >> e) & 3u); eb = e; ev = l & ((1u << e) - 1); }
}
// distance 1..32768 -> symbol 0..29, extra bits, extra value
CK_HD void ck_dfl_dist(u32 d, u32& sym, u32& eb, u32& ev) {
    u32 v = d - 1;
    if (v < 4) { sym = v; eb = 0; ev = 0; }
    else { u32 lg = ck_log2(v); sym = 2 * lg + ((v >> (lg - 1)) & 1u); eb = lg - 1; ev = v & ((1u << eb) - 1); }
}

// code lengths len[0..n) (<= maxbits) for freq[0..n), n <= 288; sym / a: scratch of n entries
CK_HD void ck_huff_lengths(const u32* freq, u32 n, u32 maxbits, u8* len, unsigned short* sym, u32* a) {
    u32 m = 0;
    for (u32 s = 0; s < n; s++) { len[s] = 0; if (freq[s]) sym[m++] = (unsigned short)s; }
    for (u32 s = 0; m < 2 && s < n; s++) if (!freq[s] && (m == 0 || sym[0] != s)) sym[m++] = (unsigned short)s;   // pair a lone symbol
    for (u32 i = 1; i < m; i++) {                       // insertion sort by (frequency, symbol)
        unsigned short v = sym[i]; u32 fv = freq[v]; u32 j = i;
        while (j > 0 && (freq[sym[j - 1]] > fv || (freq[sym[j - 1]] == fv && sym[j - 1] > v))) { sym[j] = sym[j - 1]; j--; }
        sym[j] = v;
    }
    for (u32 i = 0; i < m; i++) a[i] = freq[sym[i]] ? freq[sym[i]] : 1u;
    // Moffat-Katajainen: a[] ascending frequencies -> code lengths, in place
    a[0] += a[1];
    u32 root = 0, leaf = 2;
    for (u32 next = 1; next < m - 1; next++) {
        if (leaf >= m || a[root] < a[leaf]) { a[next] = a[root]; a[root++] = next; } else a[next] = a[leaf++];
        if (leaf >= m || (root < next && a[root] < a[leaf])) { a[next] += a[root]; a[root++] = next; } else a[next] += a[leaf++];
    }
    a[m - 2] = 0;
    for (int next = (int)m - 3; next >= 0; next--) a[next] = a[a[next]] + 1;
    int avbl = 1, used = 0, dpth = 0, r = (int)m - 2, nx = (int)m - 1;
    while (avbl > 0) {
        while (r >= 0 && (int)a[r] == dpth) { used++; r--; }
        while (avbl > used) { a[nx--] = (u32)dpth; avbl--; }
        avbl = 2 * used; dpth++; used = 0;
    }
    // limit to maxbits: a[] is now non-increasing; count per length, fold the long ones, restore the Kraft sum
    u32 num[33] = {0};
    for (u32 i = 0; i < m; i++) num[a[i] > 32 ? 32 : a[i]]++;
    for (u32 l = maxbits + 1; l <= 32; l++) { num[maxbits] += num[l]; num[l] = 0; }
    unsigned long long total = 0;
    for (u32 l = 1; l <= maxbits; l++) total += (unsigned long long)num[l] << (maxbits - l);
    while (total != (1ull << maxbits)) {
        num[maxbits]--;
        for (u32 l = maxbits - 1; l > 0; l--) if (num[l]) { num[l]--; num[l + 1] += 2; break; }
        total--;
    }
    u32 j = 0;                                          // the rarest symbols get the longest codes
    for (u32 l = maxbits; l > 0; l--) for (u32 k = 0; k < num[l]; k++) len[sym[j++]] = (u8)l;
}

// canonical codes, bit-reversed for LSB-first output
CK_HD void ck_huff_codes(const u8* len, u32 n, unsigned short* code) {
    u32 cnt[16] = {0}, next[16];
    for (u32 s = 0; s < n; s++) cnt[len[s]]++;
    cnt[0] = 0;
    u32 c = 0;
    for (u32 b = 1; b < 16; b++) { c = (c + cnt[b - 1]) << 1; next[b] = c; }
    for (u32 s = 0; s < n; s++) code[s] = len[s] ? (unsigned short)ck_bitrev(next[len[s]]++, len[s]) : 0;
}

struct ck_dfl_tables {
    u32 lf[286], df[30], cf[19];
    u8 ll[286 + 30], cl[19];                            // literal / length lengths, then distance lengths (contiguous)
    unsigned short lc[286], dc[30], cc[19];
    unsigned short rle[286 + 30];                       // code-length symbols: sym | extra << 5
    unsigned short sym[288]; u32 a[288];
    u32 hlit, hdist, hclen, nrle;
};

// counts symbols (emit = false) or writes them (emit = true)
struct ck_dfl_sink {
    const u8* w; ck_dfl_tables* t; ck_bitw* bw; bool emit, ok;
    CK_HD void lit(u32 b) { if (emit) bw->put(t->lc[b], t->ll[b]); else t->lf[b]++; }
    CK_HD void seq(u32 lp, u32 ll, u32 off, u32 ml) {
        for (u32 k = 0; k < ll; k++) lit(w[lp + k]);
        if (!ml) return;
        u32 s, eb, ev, ds, deb, dev;
        ck_dfl_len(ml, s, eb, ev); ck_dfl_dist(off, ds, deb, dev);
        if (emit) { bw->put(t->lc[s], t->ll[s]); bw->put(ev, eb); bw->put(t->dc[ds], t->ll[286 + ds]); bw->put(dev, deb); }
        else { t->lf[s]++; t->df[ds]++; }
    }
};

CK_HD void ck_dfl_parse(const u8* w, u32 start, u32 end, u32* tab, ck_dfl_sink& f) {
    ck_lz_parse(w, start, end, end >= start + 4 ? end - 3 : start, end, 32768u, 258u, tab, CK_DFL_TAB_BITS, f);
}

// one chunk w[start..end) (end - start <= 64 KB) whose history w[0..start) matches may reach into (the caller passes at
// most 32 KB of it).  dst gets the chunk's blocks, starting and ending on a byte; returns their size, at most
// (end - start) + 5 * ceil((end - start) / 65535).  tab: 1 << CK_DFL_TAB_BITS entries; t: scratch.
CK_HD u32 ck_deflate_chunk(const u8* w, u32 start, u32 end, u8* dst, u32* tab, ck_dfl_tables& t) {
    u32 n = end - start;
    for (u32 s = 0; s < 286; s++) t.lf[s] = 0;
    for (u32 s = 0; s < 30; s++) t.df[s] = 0;
    for (u32 s = 0; s < 19; s++) t.cf[s] = 0;
    ck_bitw bw; bw.p = dst; bw.op = 0; bw.buf = 0; bw.cnt = 0;
    ck_dfl_sink f; f.w = w; f.t = &t; f.bw = &bw; f.emit = false; f.ok = true;
    ck_dfl_parse(w, start, end, tab, f);
    t.lf[256] = 1;                                      // end of block
    ck_huff_lengths(t.lf, 286, 15, t.ll, t.sym, t.a);
    ck_huff_lengths(t.df, 30, 15, t.ll + 286, t.sym, t.a);
    t.hlit = 286; while (t.hlit > 257 && !t.ll[t.hlit - 1]) t.hlit--;
    t.hdist = 30; while (t.hdist > 1 && !t.ll[286 + t.hdist - 1]) t.hdist--;
    // run-length code of the hlit + hdist lengths (runs may cross from the literal into the distance lengths)
    u8 seqv[286 + 30];
    u32 total = t.hlit + t.hdist;
    for (u32 i = 0; i < t.hlit; i++) seqv[i] = t.ll[i];
    for (u32 i = 0; i < t.hdist; i++) seqv[t.hlit + i] = t.ll[286 + i];
    t.nrle = 0;
    for (u32 i = 0; i < total;) {
        u32 v = seqv[i], run = 1;
        while (i + run < total && seqv[i + run] == v) run++;
        u32 r = run;
        if (v == 0) {
            while (r >= 11) { u32 k = r < 138 ? r : 138; t.rle[t.nrle++] = (unsigned short)(18 | (k - 11) << 5); r -= k; }
            if (r >= 3) { t.rle[t.nrle++] = (unsigned short)(17 | (r - 3) << 5); r = 0; }
            while (r) { t.rle[t.nrle++] = 0; r--; }
        } else {
            t.rle[t.nrle++] = (unsigned short)v; r--;
            while (r >= 3) { u32 k = r < 6 ? r : 6; t.rle[t.nrle++] = (unsigned short)(16 | (k - 3) << 5); r -= k; }
            while (r) { t.rle[t.nrle++] = (unsigned short)v; r--; }
        }
        i += run;
    }
    for (u32 i = 0; i < t.nrle; i++) t.cf[t.rle[i] & 31u]++;
    ck_huff_lengths(t.cf, 19, 7, t.cl, t.sym, t.a);
    const unsigned char order[19] = {16, 17, 18, 0, 8, 7, 9, 6, 10, 5, 11, 4, 12, 3, 13, 2, 14, 1, 15};
    t.hclen = 19; while (t.hclen > 4 && !t.cl[order[t.hclen - 1]]) t.hclen--;
    // exact size of the dynamic block
    unsigned long long bits = 3 + 14 + 3ull * t.hclen;
    const u8 cl_extra[3] = {2, 3, 7};
    for (u32 s = 0; s < 19; s++) bits += (unsigned long long)t.cf[s] * (t.cl[s] + (s >= 16 ? cl_extra[s - 16] : 0u));
    for (u32 s = 0; s < 286; s++) {
        if (!t.lf[s]) continue;
        u32 eb = 0;
        if (s >= 265 && s < 285) eb = (s - 261) / 4;
        bits += (unsigned long long)t.lf[s] * (t.ll[s] + eb);
    }
    for (u32 s = 0; s < 30; s++) if (t.df[s]) bits += (unsigned long long)t.df[s] * (t.ll[286 + s] + (s >= 4 ? s / 2 - 1 : 0u));
    unsigned long long dyn = (bits + 3 + 7) / 8 + 4;    // + the empty stored block: 3 bits, pad to a byte, 00 00 ff ff
    unsigned long long stored = n + 5ull * ((n + 65534) / 65535);
    if (dyn > stored) {
        for (u32 p = 0; p < n;) {                       // not final, stored
            u32 k = n - p < 65535 ? n - p : 65535;
            u8* d = dst + bw.op;
            d[0] = 0; d[1] = (u8)k; d[2] = (u8)(k >> 8); d[3] = (u8)~k; d[4] = (u8)(~k >> 8);
            for (u32 i = 0; i < k; i++) d[5 + i] = w[start + p + i];
            bw.op += 5 + k; p += k;
        }
        return bw.op;
    }
    ck_huff_codes(t.ll, 286, t.lc);
    ck_huff_codes(t.ll + 286, 30, t.dc);
    ck_huff_codes(t.cl, 19, t.cc);
    bw.put(0, 1); bw.put(2, 2);                         // not final, dynamic
    bw.put(t.hlit - 257, 5); bw.put(t.hdist - 1, 5); bw.put(t.hclen - 4, 4);
    for (u32 k = 0; k < t.hclen; k++) bw.put(t.cl[order[k]], 3);
    for (u32 i = 0; i < t.nrle; i++) {
        u32 s = t.rle[i] & 31u, x = t.rle[i] >> 5;
        bw.put(t.cc[s], t.cl[s]);
        if (s >= 16) bw.put(x, cl_extra[s - 16]);
    }
    f.emit = true;
    ck_dfl_parse(w, start, end, tab, f);
    bw.put(t.lc[256], t.ll[256]);
    bw.put(0, 3); bw.align();                           // empty stored block: the next chunk starts on a byte
    bw.put(0, 16); bw.put(0xffff, 16);
    return bw.op;
}

CK_HD void ck_gzip_head(u8* d) { d[0] = 0x1f; d[1] = 0x8b; d[2] = 8; for (u32 k = 3; k < 9; k++) d[k] = 0; d[9] = 0xff; }
// after the last chunk: the empty final fixed-Huffman block, CRC-32 and ISIZE of the section
CK_HD void ck_gzip_tail(u8* d, u32 crc, u32 isize) {
    d[0] = 3; d[1] = 0;
    for (u32 k = 0; k < 4; k++) { d[2 + k] = (u8)(crc >> (8 * k)); d[6 + k] = (u8)(isize >> (8 * k)); }
}

#endif  // CK_DEFLATE_CUH
