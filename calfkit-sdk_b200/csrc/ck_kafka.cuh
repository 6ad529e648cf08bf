// Kafka RecordBatch v2 framing on the device (SURVEY.md section 8f row 1).
//
// Reference: done by aiokafka underneath broker.subscriber(...) / broker.publish(...) (calfkit/worker/worker.py:45-53,
// calfkit/nodes/base.py:82-87; faststream[kafka] -> aiokafka, third-party, absent from the image).  Format restated in
// oracle/kafka_batch.py from the published protocol (message format v2) and pinned there to known-answer vectors.
//
// decode (a fetch response's record set = concatenated frames, copied to HBM as it arrived):
//   ck_rb_crc_kernel     warp per batch: CRC32C (Castagnoli) of the covered bytes [21, end) — every lane runs a
//                        slicing-by-4 table CRC over its own contiguous chunk, the 32 partial CRCs are folded with
//                        GF(2) polynomial arithmetic (crc(A||B) = crc(A) * x^(8|B|) mod P  xor  crc(B));
//   ck_rb_split_kernel   thread per batch: hop from record to record (each starts with its own varint length)
//   ck_rb_fields_kernel  thread per record: zig-zag varints -> key span, value span, the `correlation_id` header span
// The walker then reads every value where it lies inside the raw buffer (ck_view.len): no per-record slicing on the host.
// Compressed frames (gzip = codec 1, ck_inflate.cuh; LZ4 = codec 3, ck_lz4.cuh), only when a fetch holds any:
//   ck_rb_csize_kernel       thread per frame: decompressed size (gzip ISIZE / LZ4 token walk); scan -> 16-byte slots
//   ck_rb_decompress_kernel  thread per frame: decode into the slot after the submitted bytes; the split then reads there
//
// encode (produce): the payloads of one topic-partition (an index list the producer side already has) become one frame:
//   ck_rb_size_kernel    thread per record: encoded size (varints depend on the record's offsetDelta = its rank)
//   (scan)               -> byte offset of every record inside the frame
//   ck_rb_write_kernel   warp per record: varint header, key, value, the two headers calfkit's publishes carry
//   ck_rb_header_kernel + ck_rb_crc_chunks/fold: the 61-byte batch header, CRC32C over the frame in 16 KB chunks
// encode runs (produce, every topic-partition of a step; codec 0 none, 1 gzip, 3 LZ4):
//   ck_rbs_split_kernel      warp per group: greedy split to max_bytes with exact in-frame sizes -> offsetDelta, size, opens
//   (scans) + ck_rbs_index_kernel / ck_rbs_layout_kernel: record offsets, frame of every record, 64 KB chunks per frame
//   ck_rb_write_kernel       the records, straight into the frames (codec 0) or into a plaintext scratch
//   ck_rbs_compress_kernel   thread per 64 KB chunk (ck_lz4_enc.cuh / ck_deflate.cuh) into a slot of worst-case size
//   (scans) + ck_rbs_copy_kernel / ck_rbs_header_kernel / ck_rbs_crc_kernel: assembly, headers, gzip CRC-32 fold, CRC32C
// Worst-case section for P bytes of records: LZ4 11 + P + 4 ceil(P / 64 KB), gzip 20 + P + 10 ceil(P / 64 KB).
#ifndef CK_KAFKA_CUH
#define CK_KAFKA_CUH

#include "ck_walk.cuh"            // u8 / u32 and CK_HD (the CRC and checksum cores below also build on the host)

#define CK_CRC_POLY 0x82F63B78u      // CRC32C (Castagnoli), reflected: the RecordBatch CRC
#define CK_CRC32_POLY 0xEDB88320u    // CRC-32 (IEEE 802.3), reflected: the gzip trailer (ck_inflate.cuh)
#define CK_RB_HEADER 61u
#define CK_RB_CRC_FROM 21u

// ---- CRC32C / CRC-32 -------------------------------------------------------------------------------------------------
// four 256-entry tables (slicing-by-4) for the reflected polynomial `poly`, built in shared memory by the block itself
// (by the calling thread alone in the host test build)
CK_HD void ck_crc_tables(u32* t /* [4][256] */, u32 poly = CK_CRC_POLY) {
#if defined(__CUDA_ARCH__)
    const u32 i0 = threadIdx.x, step = blockDim.x;
#else
    const u32 i0 = 0, step = 1;
#endif
    for (u32 i = i0; i < 256; i += step) {
        u32 c = i;
#pragma unroll
        for (int k = 0; k < 8; k++) c = (c >> 1) ^ ((c & 1u) ? poly : 0u);
        t[i] = c;
    }
#if defined(__CUDA_ARCH__)
    __syncthreads();
#endif
    for (u32 i = i0; i < 256; i += step) {
        u32 c = t[i];
#pragma unroll
        for (int k = 1; k < 4; k++) { c = (c >> 8) ^ t[c & 0xffu]; t[k * 256 + i] = c; }
    }
#if defined(__CUDA_ARCH__)
    __syncthreads();
#endif
}
// finalised CRC of p[0..n) (init / xor-out all ones) for the polynomial the tables were built for
CK_HD u32 ck_crc_span(const u32* __restrict__ t, const u8* __restrict__ p, u32 n) {
    u32 c = 0xffffffffu;
    while (n && ((uintptr_t)p & 3u)) { c = t[(c ^ *p++) & 0xffu] ^ (c >> 8); n--; }
    const u32* w = (const u32*)p;
    for (; n >= 4; n -= 4) {
#if defined(__CUDA_ARCH__)
        c ^= __ldg(w++);
#else
        c ^= *w++;
#endif
        c = t[768 + (c & 0xffu)] ^ t[512 + ((c >> 8) & 0xffu)] ^ t[256 + ((c >> 16) & 0xffu)] ^ t[c >> 24];
    }
    p = (const u8*)w;
    while (n--) c = t[(c ^ *p++) & 0xffu] ^ (c >> 8);
    return ~c;
}

#include "ck_inflate.cuh"
#include "ck_lz4.cuh"
#include "ck_deflate.cuh"

#if defined(__CUDACC__)
// a(x) * b(x) mod P(x), reflected representation (bit 31 = x^0); poly: the reflected polynomial, as for ck_crc_tables
__device__ __forceinline__ u32 ck_gf_mul(u32 a, u32 b, u32 poly = CK_CRC_POLY) {
    u32 p = 0;
#pragma unroll 4
    for (u32 m = 0x80000000u; m; m >>= 1) {
        if (a & m) p ^= b;
        b = (b & 1u) ? (b >> 1) ^ poly : b >> 1;
    }
    return p;
}
// x^(8 n) mod P
__device__ __forceinline__ u32 ck_gf_xpow8(unsigned long long n, u32 poly = CK_CRC_POLY) {
    u32 p = 0x80000000u;                       // x^0
    u32 sq = 0x00800000u;                      // x^8
    while (n) { if (n & 1ull) p = ck_gf_mul(sq, p, poly); sq = ck_gf_mul(sq, sq, poly); n >>= 1; }
    return p;
}
__device__ __forceinline__ u32 ck_crc_combine(u32 crc_a, u32 crc_b, u32 xpow_len_b, u32 poly = CK_CRC_POLY) {
    return ck_gf_mul(xpow_len_b, crc_a, poly) ^ crc_b;
}

// CRC32C of one span by one warp (all lanes return it): lane 0 takes the odd-sized head so that every other lane holds
// exactly `chunk` bytes and the tree fold shifts by multiples of one precomputed power
__device__ __forceinline__ u32 ck_crc32c_warp(const u32* __restrict__ t, const u8* __restrict__ p, u32 n, u32 lane) {
    u32 chunk = (n >> 5) & ~3u;
    u32 head = n - 31u * chunk;
    u32 c = lane == 0 ? ck_crc_span(t, p, head) : (chunk ? ck_crc_span(t, p + head + (lane - 1) * chunk, chunk) : 0u);
    if (!chunk) return __shfl_sync(0xffffffffu, c, 0);
    u32 xp = ck_gf_xpow8(chunk);               // x^(8 chunk); squared at every level: right blocks hold 1, 2, 4, 8, 16 chunks
#pragma unroll
    for (u32 s = 1; s < 32; s <<= 1) {
        u32 right = __shfl_down_sync(0xffffffffu, c, s);
        if ((lane & (2 * s - 1)) == 0) c = ck_crc_combine(c, right, xp);
        xp = ck_gf_mul(xp, xp);
    }
    return __shfl_sync(0xffffffffu, c, 0);
}

__device__ __forceinline__ u32 ck_be32(const u8* p) { return ((u32)p[0] << 24) | ((u32)p[1] << 16) | ((u32)p[2] << 8) | p[3]; }
__device__ __forceinline__ void ck_put_be32(u8* p, u32 v) { p[0] = v >> 24; p[1] = v >> 16; p[2] = v >> 8; p[3] = v; }
__device__ __forceinline__ void ck_put_be64(u8* p, unsigned long long v) { ck_put_be32(p, (u32)(v >> 32)); ck_put_be32(p + 4, (u32)v); }

// ---- decode -------------------------------------------------------------------------------------------------------------
// batch_bad[b] / rec_bad[i]: why a frame (and every record in it) was refused
#define CK_RB_BAD 1u          // CRC32C, framing or decompression failure
#define CK_RB_BAD_CODEC 2u    // a compression codec the device does not decode (snappy = 2, zstd = 4, 5-7 unassigned)
#define CK_RB_GZIP 1u
#define CK_RB_LZ4 3u
__device__ __forceinline__ bool ck_rb_codec_decoded(u32 codec) { return codec == 0 || codec == CK_RB_GZIP || codec == CK_RB_LZ4; }

// batch_off[b] .. batch_off[b+1]: frame b inside buf (indexed by the host: the frames chain through their own length field)
__global__ void __launch_bounds__(256)
ck_rb_crc_kernel(const u8* __restrict__ buf, const long long* __restrict__ batch_off, u32 nb, u32* __restrict__ batch_bad) {
    __shared__ u32 t[1024];
    ck_crc_tables(t);
    u32 w = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
    if (w >= nb) return;
    const u8* f = buf + batch_off[w];
    u32 flen = (u32)(batch_off[w + 1] - batch_off[w]);
    u32 bad = 0;
    if (flen < CK_RB_HEADER || f[16] != 2) bad = CK_RB_BAD;                            // not magic 2
    else {
        u32 c = ck_crc32c_warp(t, f + CK_RB_CRC_FROM, flen - CK_RB_CRC_FROM, lane);
        if (c != ck_be32(f + 17)) bad = CK_RB_BAD;
        else if (!ck_rb_codec_decoded(f[22] & 7u)) bad = CK_RB_BAD_CODEC;
    }
    if (lane == 0) batch_bad[w] = bad;
}

__device__ __forceinline__ bool ck_varint(const u8* __restrict__ p, u32& pos, u32 end, long long& out) {
    unsigned long long u = 0; u32 shift = 0;
    for (;;) {
        if (pos >= end || shift > 63) return false;
        u8 b = p[pos++];
        u |= (unsigned long long)(b & 0x7f) << shift;
        if (!(b & 0x80)) break;
        shift += 7;
    }
    out = (long long)(u >> 1) ^ -(long long)(u & 1);
    return true;
}

// thread per batch: where does each record start.  rec_base[b] = records in the batches before b (host prefix sum of
// the recordsCount header fields).  The records of batch b are the section sec_off[b] .. + sec_len[b] of buf: the raw
// bytes after the header, or for a compressed batch its decompressed slot; sec_off = nullptr means every batch is
// uncompressed (the section is the rest of the frame).  A batch whose records do not exactly fill its section is bad.
__global__ void __launch_bounds__(128)
ck_rb_split_kernel(const u8* __restrict__ buf, const long long* __restrict__ batch_off, const u32* __restrict__ rec_base, u32 nb,
                   const long long* __restrict__ sec_off, const u32* __restrict__ sec_len,
                   u32* __restrict__ batch_bad, long long* __restrict__ rec_pos, u32* __restrict__ rec_batch) {
    u32 b = blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= nb) return;
    u32 r0 = rec_base[b], cnt = rec_base[b + 1] - r0;
    long long base = sec_off ? sec_off[b] : batch_off[b] + CK_RB_HEADER;
    u32 slen = sec_off ? sec_len[b] : (u32)(batch_off[b + 1] - batch_off[b]) - CK_RB_HEADER;
    const u8* f = buf + base;
    u32 pos = 0;
    bool ok = !batch_bad[b];
    for (u32 k = 0; k < cnt; k++) {
        rec_batch[r0 + k] = b;
        if (!ok) { rec_pos[r0 + k] = -1; continue; }
        rec_pos[r0 + k] = base + pos;
        long long len;
        if (!ck_varint(f, pos, slen, len) || len < 0 || pos + (u32)len > slen) { ok = false; rec_pos[r0 + k] = -1; continue; }
        pos += (u32)len;
    }
    if (ok && pos != slen) ok = false;
    if (!ok && !batch_bad[b]) batch_bad[b] = CK_RB_BAD;
}

// thread per batch, compressed fetches only (after the CRC kernel): the decompressed size of every compressed batch that
// passed its CRC — gzip: the trailer's ISIZE (checked after the inflate); LZ4: a walk over the block headers and tokens,
// cross-checked against a stored content size.  dlen[b] = 0 for the others; a batch whose size cannot be had is bad.
__global__ void __launch_bounds__(128)
ck_rb_csize_kernel(const u8* __restrict__ buf, const long long* __restrict__ batch_off, u32 nb, u32* __restrict__ batch_bad,
                   u32* __restrict__ dlen) {
    u32 b = blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= nb) return;
    const u8* f = buf + batch_off[b];
    u32 codec = f[22] & 7u, n = 0;
    if (!batch_bad[b] && codec) {
        const u8* src = f + CK_RB_HEADER;
        u32 slen = (u32)(batch_off[b + 1] - batch_off[b]) - CK_RB_HEADER;
        bool ok = codec == CK_RB_GZIP ? ck_gzip_isize(src, slen, n) : ck_lz4_frame<false>(src, slen, nullptr, n);
        if (!ok || n > 0x7fff0000u) { batch_bad[b] = CK_RB_BAD; n = 0; }
    }
    dlen[b] = n;
}

// thread per batch: decompress every compressed batch into its slot dbase + slot[b] (exclusive scan of dlen rounded up
// to 16) and give every batch its records section for the split.  A batch that does not decode is bad.
__global__ void __launch_bounds__(128)
ck_rb_decompress_kernel(u8* __restrict__ buf, const long long* __restrict__ batch_off, u32 nb, long long dbase,
                        const long long* __restrict__ slot, const u32* __restrict__ dlen, u32* __restrict__ batch_bad,
                        long long* __restrict__ sec_off, u32* __restrict__ sec_len) {
    __shared__ u32 t[1024];
    ck_crc_tables(t, CK_CRC32_POLY);
    u32 b = blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= nb) return;
    long long fo = batch_off[b];
    const u8* f = buf + fo;
    u32 flen = (u32)(batch_off[b + 1] - fo);
    u32 codec = flen >= CK_RB_HEADER ? f[22] & 7u : 0u;
    if (!codec || batch_bad[b]) { sec_off[b] = fo + CK_RB_HEADER; sec_len[b] = flen >= CK_RB_HEADER ? flen - CK_RB_HEADER : 0u; return; }
    u32 n = dlen[b];
    u8* dst = buf + dbase + slot[b];
    const u8* src = f + CK_RB_HEADER;
    bool ok = codec == CK_RB_GZIP ? ck_gunzip(src, flen - CK_RB_HEADER, dst, n, t) : ck_lz4_frame<true>(src, flen - CK_RB_HEADER, dst, n);
    if (!ok) batch_bad[b] = CK_RB_BAD;
    sec_off[b] = dbase + slot[b]; sec_len[b] = n;
}

// thread per record
__global__ void __launch_bounds__(128)
ck_rb_fields_kernel(const u8* __restrict__ buf, long long buf_len, const long long* __restrict__ rec_pos, const u32* __restrict__ rec_batch,
                    const u32* __restrict__ batch_bad, u32 n,
                    long long* __restrict__ val_off, u32* __restrict__ val_len, long long* __restrict__ key_off, int* __restrict__ key_len,
                    long long* __restrict__ corr_off, int* __restrict__ corr_len, u32* __restrict__ rec_bad) {
    u32 i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    val_off[i] = 0; val_len[i] = 0; key_off[i] = 0; key_len[i] = -1; corr_off[i] = 0; corr_len[i] = -1;
    long long rp = rec_pos[i];
    if (rp < 0 || batch_bad[rec_batch[i]]) { u32 why = batch_bad[rec_batch[i]]; rec_bad[i] = why ? why : CK_RB_BAD; return; }
    const u8* p = buf + rp;
    u32 end = (u32)min((long long)0x7fffffff, buf_len - rp), pos = 0;
    long long len, t;
    bool ok = ck_varint(p, pos, end, len);
    u32 rec_end = pos + (u32)len;
    if (ok) end = rec_end;
    pos += 1;                                                   // attributes
    ok = ok && ck_varint(p, pos, end, t) && ck_varint(p, pos, end, t);       // timestampDelta, offsetDelta
    ok = ok && ck_varint(p, pos, end, t);                       // key
    if (ok && t >= 0) { key_off[i] = rp + pos; key_len[i] = (int)t; pos += (u32)t; }
    ok = ok && pos <= end && ck_varint(p, pos, end, t);         // value
    if (ok && t >= 0) { val_off[i] = rp + pos; val_len[i] = (u32)t; pos += (u32)t; }
    long long nh = 0;
    ok = ok && pos <= end && ck_varint(p, pos, end, nh);
    for (long long hcount = 0; ok && hcount < nh; hcount++) {
        long long kl, vl;
        ok = ck_varint(p, pos, end, kl) && kl >= 0 && pos + (u32)kl <= end;
        if (!ok) break;
        u32 kpos = pos; pos += (u32)kl;
        ok = ck_varint(p, pos, end, vl);
        if (!ok) break;
        bool is_corr = (kl == 14);                              // "correlation_id" (FastStream's header)
        const char* want = "correlation_id";
        for (u32 b = 0; is_corr && b < 14; b++) is_corr = (p[kpos + b] == (u8)want[b]);
        if (vl >= 0) { if (is_corr) { corr_off[i] = rp + pos; corr_len[i] = (int)vl; } pos += (u32)vl; }
        ok = pos <= end;
    }
    ok = ok && pos == rec_end;
    rec_bad[i] = ok ? 0u : 1u;
    if (!ok) { val_len[i] = 0; }
}

__global__ void __launch_bounds__(256)
ck_rb_mark_bad_kernel(const u32* __restrict__ rec_bad, u32 n, u32* __restrict__ cols, u32 stride) {
    u32 i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n && rec_bad[i]) cols[(size_t)CK_COL_STATUS * stride + i] = CK_BAD_FRAME;
}

// ---- encode -------------------------------------------------------------------------------------------------------------
__device__ __forceinline__ u32 ck_varint_size(long long v) {
    unsigned long long u = ((unsigned long long)v << 1) ^ (unsigned long long)(v >> 63);
    u32 n = 1;
    while (u >= 0x80) { u >>= 7; n++; }
    return n;
}
__device__ __forceinline__ u32 ck_put_varint(u8* p, long long v) {
    unsigned long long u = ((unsigned long long)v << 1) ^ (unsigned long long)(v >> 63);
    u32 n = 0;
    while (u >= 0x80) { p[n++] = (u8)(u | 0x80); u >>= 7; }
    p[n++] = (u8)u;
    return n;
}
// what calfkit's publishes carry (SURVEY.md Appendix A): key = correlation id bytes when keyed, headers
// content-type: application/json and correlation_id (FastStream)
#define CK_RB_CT_HDR 30u             // varint(12) "content-type" varint(16) "application/json" = 1 + 12 + 1 + 16
struct ck_rb_rec { u32 body_len, key_len, corr_len, val_len; };

__device__ __forceinline__ ck_rb_rec ck_rb_measure(u32 rank, u32 val_len, u32 corr_len, bool keyed) {
    ck_rb_rec r; r.val_len = val_len; r.corr_len = corr_len; r.key_len = keyed ? corr_len : 0xffffffffu;
    u32 body = 1 + 1 + ck_varint_size(rank);                                    // attributes, timestampDelta 0, offsetDelta
    body += keyed ? ck_varint_size(corr_len) + corr_len : 1;                    // key (or null)
    body += ck_varint_size(val_len) + val_len;
    body += 1 + CK_RB_CT_HDR + (1 + 14 + ck_varint_size(corr_len) + corr_len);  // 2 headers
    r.body_len = body;
    return r;
}

// idx[k] = index into the publish table of the k-th record of this topic-partition (its offsetDelta = k)
__global__ void __launch_bounds__(256)
ck_rb_size_kernel(const ck_pub* __restrict__ pubs, const u32* __restrict__ idx, u32 n, const u32* __restrict__ pay_len,
                  const u32* __restrict__ cols, u32 stride, u32* __restrict__ sizes) {
    u32 k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= n) return;
    ck_pub p = pubs[idx[k]];
    ck_rb_rec r = ck_rb_measure(k, pay_len[p.payload], cols[(size_t)CK_COL_CORR_LEN * stride + p.record], p.has_key != 0);
    sizes[k] = ck_varint_size(r.body_len) + r.body_len;
}

// warp per record; corr bytes are the raw JSON string content of deps.correlation_id (ids without escapes: the hashing
// rule of ck_murmur2_key applies to escaped ones — those are rejected here by the host side before encoding).
// Record k goes to frame + hdr * (fid[k] + 1) + rec_off[k] with offsetDelta delta[k]; fid / delta = nullptr: one frame
// (record k at frame + hdr + rec_off[k], offsetDelta k).  hdr = 0 writes bare records sections back to back.
__global__ void __launch_bounds__(256)
ck_rb_write_kernel(ck_view vw, const ck_pub* __restrict__ pubs, const u32* __restrict__ idx, u32 n, const u32* __restrict__ pay_len,
                   const long long* __restrict__ out_off, const u8* __restrict__ out, const u32* __restrict__ cols, u32 stride,
                   const long long* __restrict__ rec_off, u8* __restrict__ frame, const u32* __restrict__ delta = nullptr,
                   const u32* __restrict__ fid = nullptr, u32 hdr = CK_RB_HEADER) {
    u32 k = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
    if (k >= n) return;
    ck_pub p = pubs[idx[k]];
    u32 rl; const u8* rec = ck_rec(vw, p.record, rl);
    u32 co = cols[(size_t)CK_COL_CORR_OFF * stride + p.record], cl = cols[(size_t)CK_COL_CORR_LEN * stride + p.record];
    u32 od = delta ? delta[k] : k;
    ck_rb_rec r = ck_rb_measure(od, pay_len[p.payload], cl, p.has_key != 0);
    u8* d = frame + (unsigned long long)hdr * (fid ? fid[k] + 1ull : 1ull) + rec_off[k];
    u32 pos = 0, vpos = 0, kpos = 0, cpos = 0;
    // every lane computes the same layout; lane 0 writes the small pieces, the warp copies key / value / header value
    u8 tmp[10];
    u32 m = ck_put_varint(tmp, r.body_len); if (lane == 0) for (u32 b = 0; b < m; b++) d[pos + b] = tmp[b]; pos += m;
    if (lane == 0) { d[pos] = 0; d[pos + 1] = 0; } pos += 2;                                  // attributes, timestampDelta = 0
    m = ck_put_varint(tmp, od); if (lane == 0) for (u32 b = 0; b < m; b++) d[pos + b] = tmp[b]; pos += m;
    if (p.has_key) { m = ck_put_varint(tmp, cl); if (lane == 0) for (u32 b = 0; b < m; b++) d[pos + b] = tmp[b]; pos += m; kpos = pos; pos += cl; }
    else { if (lane == 0) d[pos] = 1; pos += 1; }                                             // zig-zag(-1) = null key
    m = ck_put_varint(tmp, r.val_len); if (lane == 0) for (u32 b = 0; b < m; b++) d[pos + b] = tmp[b]; pos += m; vpos = pos; pos += r.val_len;
    if (lane == 0) {
        d[pos] = 4;                                                                           // 2 headers
        d[pos + 1] = 24; const char* a = "content-type"; for (u32 b = 0; b < 12; b++) d[pos + 2 + b] = (u8)a[b];
        d[pos + 14] = 32; const char* j = "application/json"; for (u32 b = 0; b < 16; b++) d[pos + 15 + b] = (u8)j[b];
        d[pos + 31] = 28; const char* c = "correlation_id"; for (u32 b = 0; b < 14; b++) d[pos + 32 + b] = (u8)c[b];
    }
    pos += 1 + CK_RB_CT_HDR + 15;
    m = ck_put_varint(tmp, cl); if (lane == 0) for (u32 b = 0; b < m; b++) d[pos + b] = tmp[b]; pos += m; cpos = pos;
    if (p.has_key) for (u32 b = lane; b < cl; b += 32) d[kpos + b] = rec[co + b];
    for (u32 b = lane; b < cl; b += 32) d[cpos + b] = rec[co + b];
    ck_warp_copy(d + vpos, out + out_off[p.payload], r.val_len, lane);
}

// frame header (everything but the crc), by one thread
__global__ void ck_rb_header_kernel(u8* __restrict__ frame, const long long* __restrict__ rec_off, u32 n, long long base_offset,
                                    long long timestamp_ms, long long* __restrict__ frame_len_out) {
    if (threadIdx.x || blockIdx.x) return;
    unsigned long long total = CK_RB_HEADER + (unsigned long long)rec_off[n];
    ck_put_be64(frame, (unsigned long long)base_offset);
    ck_put_be32(frame + 8, (u32)(total - 12));
    ck_put_be32(frame + 12, 0);                              // partitionLeaderEpoch
    frame[16] = 2;
    frame[21] = 0; frame[22] = 0;                            // attributes: no compression, CreateTime
    ck_put_be32(frame + 23, n - 1);                          // lastOffsetDelta
    ck_put_be64(frame + 27, (unsigned long long)timestamp_ms);
    ck_put_be64(frame + 35, (unsigned long long)timestamp_ms);
    ck_put_be64(frame + 43, ~0ull);                          // producerId -1
    frame[51] = 0xff; frame[52] = 0xff;                      // producerEpoch -1
    ck_put_be32(frame + 53, 0xffffffffu);                    // baseSequence -1
    ck_put_be32(frame + 57, n);
    *frame_len_out = (long long)total;
}

// CRC32C of a large frame: one warp per 16 KB chunk of the covered bytes, then one warp folds the partials
#define CK_RB_CRC_CHUNK 16384u
__global__ void __launch_bounds__(256)
ck_rb_crc_chunks_kernel(const u8* __restrict__ frame, const long long* __restrict__ frame_len, u32* __restrict__ partial) {
    __shared__ u32 t[1024];
    ck_crc_tables(t);
    u32 w = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
    unsigned long long covered = (unsigned long long)*frame_len - CK_RB_CRC_FROM;
    unsigned long long start = (unsigned long long)w * CK_RB_CRC_CHUNK;
    if (start >= covered) return;
    u32 len = (u32)min((unsigned long long)CK_RB_CRC_CHUNK, covered - start);
    u32 c = ck_crc32c_warp(t, frame + CK_RB_CRC_FROM + start, len, lane);
    if (lane == 0) partial[w] = c;
}
__global__ void ck_rb_crc_fold_kernel(u8* __restrict__ frame, const long long* __restrict__ frame_len, const u32* __restrict__ partial) {
    if (blockIdx.x || threadIdx.x) return;
    unsigned long long covered = (unsigned long long)*frame_len - CK_RB_CRC_FROM;
    u32 nchunks = (u32)((covered + CK_RB_CRC_CHUNK - 1) / CK_RB_CRC_CHUNK);
    u32 xp = ck_gf_xpow8(CK_RB_CRC_CHUNK);
    u32 c = 0;                                               // crc of the empty prefix
    for (u32 k = 0; k < nchunks; k++) {
        unsigned long long start = (unsigned long long)k * CK_RB_CRC_CHUNK;
        u32 len = (u32)min((unsigned long long)CK_RB_CRC_CHUNK, covered - start);
        c = ck_crc_combine(c, partial[k], len == CK_RB_CRC_CHUNK ? xp : ck_gf_xpow8(len));
    }
    ck_put_be32(frame + 17, c);
}

// ---- encode: runs of frames, compressed or not (ck_encode_recordbatches) ------------------------------------------------
// Records of group g = idx[group_off[g] .. group_off[g+1]) (one topic-partition each) become a run of frames: a frame takes
// the group's next records while 61 + their encoded sizes <= max_bytes, and always at least one.  offsetDelta is the
// position inside the frame, so a record's size depends on where its frame starts: the split measures exact sizes.
__device__ __forceinline__ u32 ck_rbs_size(const ck_pub* __restrict__ pubs, const u32* __restrict__ idx, u32 k, u32 d,
                                           const u32* __restrict__ pay_len, const u32* __restrict__ cols, u32 stride) {
    ck_pub p = pubs[idx[k]];
    ck_rb_rec r = ck_rb_measure(d, pay_len[p.payload], cols[(size_t)CK_COL_CORR_LEN * stride + p.record], p.has_key != 0);
    return ck_varint_size(r.body_len) + r.body_len;
}

// warp per group, 32 records per step: sizes at the open frame's positions, a prefix sum, one ballot for the first record
// that does not fit.  Writes per record its offsetDelta, its size and whether it opens a frame.
__global__ void __launch_bounds__(256)
ck_rbs_split_kernel(const ck_pub* __restrict__ pubs, const u32* __restrict__ idx, const u32* __restrict__ group_off, u32 n_groups,
                    const u32* __restrict__ pay_len, const u32* __restrict__ cols, u32 stride, u32 max_bytes,
                    u32* __restrict__ delta, u32* __restrict__ sizes, u32* __restrict__ opens) {
    u32 g = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
    if (g >= n_groups) return;
    u32 end = group_off[g + 1], s = group_off[g], pos = s;             // s: first record of the open frame
    unsigned long long acc = CK_RB_HEADER;
    while (pos < end) {
        u32 k = pos + lane;
        unsigned long long inc = k < end ? ck_rbs_size(pubs, idx, k, k - s, pay_len, cols, stride) : 0ull;
        u32 sz = (u32)inc;
#pragma unroll
        for (u32 o = 1; o < 32; o <<= 1) { unsigned long long t = __shfl_up_sync(0xffffffffu, inc, o); if (lane >= o) inc += t; }
        u32 over = __ballot_sync(0xffffffffu, k < end && acc + inc > max_bytes);
        u32 take = over ? __ffs(over) - 1 : min(32u, end - pos);
        if (take == 0 && pos == s) take = 1;                            // a record larger than the limit: a frame of its own
        if (lane < take) { delta[k] = k - s; sizes[k] = sz; opens[k] = k == s; }
        acc += take ? __shfl_sync(0xffffffffu, inc, take - 1) : 0ull;
        pos += take;
        if (over) { s = pos; acc = CK_RB_HEADER; }                      // the frame is full: the next one opens at pos
    }
}

// thread per record: its frame (opens_x = exclusive scan of opens), and the first record of every frame
__global__ void __launch_bounds__(256)
ck_rbs_index_kernel(const u32* __restrict__ opens, const long long* __restrict__ opens_x, u32 n, u32 nf, u32* __restrict__ fid,
                    u32* __restrict__ frame_first) {
    u32 k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k == 0) frame_first[nf] = n;
    if (k >= n) return;
    u32 f = (u32)opens_x[k] + opens[k] - 1;
    fid[k] = f;
    if (opens[k]) frame_first[f] = k;
}

// thread per frame: records section size and 64 KB chunk count; uncompressed frames also get their place in the output
// (frame_off[nf] = total), since their size is known here
#define CK_RBS_CHUNK 65536u
__global__ void __launch_bounds__(256)
ck_rbs_layout_kernel(const u32* __restrict__ frame_first, const long long* __restrict__ rec_off, u32 nf, u32 codec,
                     u32* __restrict__ nchunks, long long* __restrict__ frame_off) {
    u32 f = blockIdx.x * blockDim.x + threadIdx.x;
    if (f > nf) return;
    long long s0 = rec_off[frame_first[f]];
    if (!codec) { frame_off[f] = s0 + (long long)CK_RB_HEADER * f; return; }
    if (f == nf) return;
    long long sec = rec_off[frame_first[f + 1]] - s0;
    nchunks[f] = (u32)((sec + CK_RBS_CHUNK - 1) / CK_RBS_CHUNK);
}

// the frame of chunk c: the last f with chunk_base[f] <= c
__device__ __forceinline__ u32 ck_rbs_frame_of(const long long* __restrict__ base, u32 nf, unsigned long long c) {
    u32 lo = 0, hi = nf;                                               // base[lo] <= c < base[hi]
    while (hi - lo > 1) { u32 mid = (lo + hi) >> 1; if ((unsigned long long)base[mid] <= c) lo = mid; else hi = mid; }
    return lo;
}

// one thread per chunk, grid-stride over a fixed pool of threads (each owns a hash table and DEFLATE scratch): chunk c of
// frame f is plain[start, end) with start = the frame's section start + 64 KB * (c - chunk_base[f]).  Its compressed form
// goes to the slot plain-offset + 64 * c of `slots` (never larger than the chunk + 64 bytes), its size to csz[c], and for
// gzip its CRC-32 to ccrc[c].  Chunks c in [*n_chunks, cmax) get size 0 (the scan after this runs over the host's bound).
__global__ void __launch_bounds__(128)
ck_rbs_compress_kernel(const u8* __restrict__ plain, const long long* __restrict__ rec_off, const u32* __restrict__ frame_first,
                       const long long* __restrict__ chunk_base, u32 nf, const unsigned long long* __restrict__ n_chunks, u32 cmax,
                       u32 codec, u8* __restrict__ slots, u32* __restrict__ csz, u32* __restrict__ ccrc, u32* __restrict__ tabs,
                       ck_dfl_tables* __restrict__ dtabs) {
    __shared__ u32 t[1024];
    ck_crc_tables(t, CK_CRC32_POLY);
    u32 tid = blockIdx.x * blockDim.x + threadIdx.x, nt = gridDim.x * blockDim.x;
    unsigned long long nc = *n_chunks;
    u32* tab = tabs + ((size_t)tid << CK_DFL_TAB_BITS);
    for (u32 c = tid; c < cmax; c += nt) {
        if (c >= nc) { csz[c] = 0; continue; }
        u32 f = ck_rbs_frame_of(chunk_base, nf, c);
        long long s0 = rec_off[frame_first[f]], s1 = rec_off[frame_first[f + 1]];
        long long start = s0 + (long long)(c - chunk_base[f]) * CK_RBS_CHUNK;
        u32 n = (u32)min((long long)CK_RBS_CHUNK, s1 - start);
        u8* dst = slots + start + 64ll * c;
        if (codec == CK_RB_LZ4) {
            csz[c] = ck_lz4_enc_block(plain + start, n, dst, tab);
        } else {
            long long lo = start - s0 > 32768 ? start - 32768 : s0;    // history: up to 32 KB of the same section
            csz[c] = ck_deflate_chunk(plain + lo, (u32)(start - lo), (u32)(start - lo) + n, dst, tab, dtabs[tid]);
            ccrc[c] = ck_crc_span(t, plain + start, n);
        }
    }
}

// thread per frame: compressed frame size = header + codec header + its chunks + codec trailer
__global__ void __launch_bounds__(256)
ck_rbs_fsize_kernel(const long long* __restrict__ chunk_base, const long long* __restrict__ chunk_off, u32 nf, u32 codec,
                    u32* __restrict__ fsize) {
    u32 f = blockIdx.x * blockDim.x + threadIdx.x;
    if (f >= nf) return;
    long long cs = chunk_off[chunk_base[f + 1]] - chunk_off[chunk_base[f]];
    fsize[f] = CK_RB_HEADER + (u32)cs + (codec == CK_RB_LZ4 ? CK_LZ4_HEAD + CK_LZ4_TAIL : CK_GZ_HEAD + CK_GZ_TAIL);
}

// warp per chunk: slot -> its place in the frame
__global__ void __launch_bounds__(256)
ck_rbs_copy_kernel(const u8* __restrict__ slots, const long long* __restrict__ rec_off, const u32* __restrict__ frame_first,
                   const long long* __restrict__ chunk_base, const long long* __restrict__ chunk_off, u32 nf,
                   const unsigned long long* __restrict__ n_chunks, u32 codec, const long long* __restrict__ frame_off, u8* __restrict__ out) {
    unsigned long long c = (blockIdx.x * (unsigned long long)blockDim.x + threadIdx.x) >> 5;
    u32 lane = threadIdx.x & 31;
    if (c >= *n_chunks) return;
    u32 f = ck_rbs_frame_of(chunk_base, nf, c);
    long long start = rec_off[frame_first[f]] + (long long)(c - chunk_base[f]) * CK_RBS_CHUNK;
    u32 head = codec == CK_RB_LZ4 ? CK_LZ4_HEAD : CK_GZ_HEAD;
    u8* dst = out + frame_off[f] + CK_RB_HEADER + head + (chunk_off[c] - chunk_off[chunk_base[f]]);
    ck_warp_copy(dst, slots + start + 64ll * c, (u32)(chunk_off[c + 1] - chunk_off[c]), lane);
}

// thread per frame: the 61-byte header (everything but the CRC32C), the codec's header and trailer (gzip: CRC-32 of the
// section folded from the per-chunk CRCs), and the frame's group.  Frame f of group g: baseOffset = base_offsets[g] +
// the records of g in earlier frames.
__global__ void __launch_bounds__(128)
ck_rbs_header_kernel(u8* __restrict__ out, const long long* __restrict__ frame_off, const u32* __restrict__ frame_first,
                     const long long* __restrict__ rec_off, u32 nf, const u32* __restrict__ group_off, u32 n_groups,
                     const long long* __restrict__ base_offsets, long long timestamp_ms, u32 codec,
                     const long long* __restrict__ chunk_base, const u32* __restrict__ ccrc, u32* __restrict__ frame_group) {
    u32 f = blockIdx.x * blockDim.x + threadIdx.x;
    if (f >= nf) return;
    u32 k0 = frame_first[f], cnt = frame_first[f + 1] - k0;
    u32 lo = 0, hi = n_groups;                                         // the group holding k0: last g with group_off[g] <= k0
    while (hi - lo > 1) { u32 mid = (lo + hi) >> 1; if (group_off[mid] <= k0) lo = mid; else hi = mid; }
    u8* fr = out + frame_off[f];
    unsigned long long flen = (unsigned long long)(frame_off[f + 1] - frame_off[f]);
    ck_put_be64(fr, (unsigned long long)((base_offsets ? base_offsets[lo] : 0ll) + (k0 - group_off[lo])));
    ck_put_be32(fr + 8, (u32)(flen - 12));
    ck_put_be32(fr + 12, 0);                                 // partitionLeaderEpoch
    fr[16] = 2;
    fr[21] = 0; fr[22] = (u8)codec;                          // attributes: codec, CreateTime
    ck_put_be32(fr + 23, cnt - 1);                           // lastOffsetDelta
    ck_put_be64(fr + 27, (unsigned long long)timestamp_ms);
    ck_put_be64(fr + 35, (unsigned long long)timestamp_ms);
    ck_put_be64(fr + 43, ~0ull);                             // producerId -1
    fr[51] = 0xff; fr[52] = 0xff;                            // producerEpoch -1
    ck_put_be32(fr + 53, 0xffffffffu);                       // baseSequence -1
    ck_put_be32(fr + 57, cnt);
    frame_group[f] = lo;
    if (codec == CK_RB_LZ4) {
        ck_lz4_frame_head(fr + CK_RB_HEADER);
        ck_put_be32(fr + flen - CK_LZ4_TAIL, 0);             // EndMark
    } else if (codec == CK_RB_GZIP) {
        long long s0 = rec_off[k0], sec = rec_off[frame_first[f + 1]] - s0;
        u32 crc = 0, xfull = ck_gf_xpow8(CK_RBS_CHUNK, CK_CRC32_POLY);
        for (long long c = chunk_base[f]; c < chunk_base[f + 1]; c++) {
            long long len = min((long long)CK_RBS_CHUNK, sec - (c - chunk_base[f]) * (long long)CK_RBS_CHUNK);
            crc = ck_crc_combine(crc, ccrc[c], len == CK_RBS_CHUNK ? xfull : ck_gf_xpow8((unsigned long long)len, CK_CRC32_POLY), CK_CRC32_POLY);
        }
        ck_gzip_head(fr + CK_RB_HEADER);
        ck_gzip_tail(fr + flen - CK_GZ_TAIL, crc, (u32)sec);
    }
}

// warp per frame: CRC32C of the covered bytes [21, end) of every frame
__global__ void __launch_bounds__(256)
ck_rbs_crc_kernel(u8* __restrict__ out, const long long* __restrict__ frame_off, u32 nf) {
    __shared__ u32 t[1024];
    ck_crc_tables(t);
    u32 w = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
    if (w >= nf) return;
    u8* fr = out + frame_off[w];
    u32 c = ck_crc32c_warp(t, fr + CK_RB_CRC_FROM, (u32)(frame_off[w + 1] - frame_off[w]) - CK_RB_CRC_FROM, lane);
    if (lane == 0) ck_put_be32(fr + 17, c);
}

#endif  // __CUDACC__
#endif  // CK_KAFKA_CUH
