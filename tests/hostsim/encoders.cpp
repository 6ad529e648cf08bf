// TEST INFRASTRUCTURE ONLY.  Compiles the device encoders of compressed Kafka record batches (csrc/ck_lz4_enc.cuh,
// csrc/ck_deflate.cuh, written __host__ __device__) with g++ into their own library, together with the decoders
// (codecs.cpp), so that every output can be checked against zlib, the LZ4 restatement and the host build of the device
// decoders under AddressSanitizer / UBSan.  A section is assembled here as the device assembles it: 64 KB chunks, each
// compressed on its own (a gzip chunk may reach 32 KB back into the previous one), between the codec's header and trailer.
#include "codecs.cpp"             // the decoders and ck_kafka.cuh: one translation unit

static u32 g_crc32e[1024];
static bool g_crce_ready = false;

// worst-case section size for n bytes of input (the bound the header comment of ck_kafka.cuh states)
extern "C" uint64_t ck_host_enc_bound(uint32_t n, uint32_t codec) {
    uint64_t chunks = (n + CK_DFL_CHUNK - 1) / CK_DFL_CHUNK;
    return codec == 3 ? CK_LZ4_HEAD + CK_LZ4_TAIL + n + 4 * chunks : CK_GZ_HEAD + CK_GZ_TAIL + n + 10 * chunks;
}

// codec 3: one LZ4 frame; codec 1: one gzip member.  Returns the section size, or 0 if cap is too small.
extern "C" uint64_t ck_host_encode(const uint8_t* src, uint32_t n, uint32_t codec, uint8_t* dst, uint64_t cap) {
    if (!g_crce_ready) { ck_crc_tables(g_crc32e, CK_CRC32_POLY); g_crce_ready = true; }
    uint64_t bound = ck_host_enc_bound(n, codec);
    if (cap < bound) return 0;
    std::vector<uint8_t> in(src, src + n), out(bound);
    std::vector<u32> tab(1u << CK_DFL_TAB_BITS);
    ck_dfl_tables* t = new ck_dfl_tables;
    uint64_t op = 0;
    if (codec == 3) { ck_lz4_frame_head(out.data()); op = CK_LZ4_HEAD; }
    else { ck_gzip_head(out.data()); op = CK_GZ_HEAD; }
    for (u32 s = 0; s < n; s += CK_DFL_CHUNK) {
        u32 e = n - s < CK_DFL_CHUNK ? n : s + CK_DFL_CHUNK;
        // the chunk's own buffer: history + chunk only, so that a read outside them is a sanitizer report
        u32 lo = codec == 3 ? s : (s > 32768 ? s - 32768 : 0);
        std::vector<uint8_t> win(in.begin() + lo, in.begin() + e);
        if (codec == 3) op += ck_lz4_enc_block(win.data(), e - s, out.data() + op, tab.data());
        else op += ck_deflate_chunk(win.data(), s - lo, e - lo, out.data() + op, tab.data(), *t);
    }
    delete t;
    if (codec == 3) { memset(out.data() + op, 0, 4); op += CK_LZ4_TAIL; }
    else { ck_gzip_tail(out.data() + op, n ? ck_crc_span(g_crc32e, in.data(), n) : 0u, n); op += CK_GZ_TAIL; }
    memcpy(dst, out.data(), op);
    return op;
}
