// TEST INFRASTRUCTURE ONLY.  Compiles the device decoders of compressed Kafka record batches (csrc/ck_inflate.cuh,
// csrc/ck_lz4.cuh, written __host__ __device__) with g++ into their own library, so that they can be checked against
// zlib and the LZ4 restatement on the CPU, under AddressSanitizer / UBSan, without touching the walker's test build.
#include <cstdint>
#include <cstring>
#include <vector>
#include "../../calfkit-sdk_b200/csrc/ck_kafka.cuh"

static u32 g_crc32[1024];
static bool g_crc_ready = false;

// 1 = accepted (dst[0..cap) written, cap = ISIZE); 0 = rejected.  The member is copied to a buffer of exactly n bytes and
// the output to one of exactly cap bytes, so that any read or write outside them is a sanitizer report.
extern "C" int ck_host_gunzip(const uint8_t* src, uint32_t n, uint8_t* dst, uint32_t cap) {
    if (!g_crc_ready) { ck_crc_tables(g_crc32, CK_CRC32_POLY); g_crc_ready = true; }
    std::vector<uint8_t> in(src, src + n), out(cap ? cap : 1);
    bool ok = ck_gunzip(in.data(), n, out.data(), cap, g_crc32);
    if (ok && cap) memcpy(dst, out.data(), cap);
    return ok ? 1 : 0;
}
extern "C" int ck_host_gzip_isize(const uint8_t* src, uint32_t n, uint32_t* isize) {
    std::vector<uint8_t> in(src, src + n);
    return ck_gzip_isize(in.data(), n, *isize) ? 1 : 0;
}
extern "C" int ck_host_lz4_size(const uint8_t* src, uint32_t n, uint32_t* size) {
    std::vector<uint8_t> in(src, src + n);
    return ck_lz4_frame<false>(in.data(), n, nullptr, *size) ? 1 : 0;
}
extern "C" int ck_host_lz4_decode(const uint8_t* src, uint32_t n, uint8_t* dst, uint32_t cap) {
    std::vector<uint8_t> in(src, src + n), out(cap ? cap : 1);
    u32 sz = cap;
    bool ok = ck_lz4_frame<true>(in.data(), n, out.data(), sz);
    if (ok && cap) memcpy(dst, out.data(), cap);
    return ok ? 1 : 0;
}
