// C-ABI of libcalfkit_b200.so: handle, device buffers, stream, kernel launches.
// See include/calfkit_b200.h for the contract and the reference call sites each entry replaces.
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <string>
#include <vector>

#include "../../include/calfkit_b200.h"
#include "ck_kernels.cuh"

static_assert(sizeof(ck_publish) == sizeof(ck_pub), "ck_publish must mirror ck_pub");

#define CK_LIT_CAP (256 * 1024)
#define CK_PAD 256   // tail padding of every byte buffer (readers may touch a few bytes past a span)

static thread_local std::string g_create_error;

struct ck_handle {
    int device = 0;
    cudaStream_t stream = nullptr;
    cudaStream_t xstream = nullptr; cudaEvent_t x_ev0 = nullptr, x_ev1 = nullptr;   // high-priority side stream of the exchange
    std::string err;
    uint64_t max_in = 0, max_out = 0, max_aux = 0;
    uint32_t max_records = 0, max_payloads = 0, max_pubs = 0;
    // device buffers
    u8* d_in = nullptr; long long* d_in_off = nullptr;
    u8* d_out = nullptr; long long* d_out_off = nullptr;
    u8* d_aux = nullptr; long long* d_aux_off = nullptr; u8* d_glue = nullptr;
    u8* d_ovl = nullptr; long long* d_ovl_off = nullptr; u32* d_ovl_len = nullptr; ck_canon_ctl* d_canon_ctl = nullptr; u32* d_canon_list = nullptr; ck_elem* d_elems = nullptr; u32 elem_cap = 0; u32* d_cand = nullptr; uint2* d_hist_skip = nullptr;
    uint64_t max_ovl = 0;
    u32* d_cols = nullptr; ck_out_desc* d_descs = nullptr; u32* d_pay_len = nullptr; ck_pub* d_pubs = nullptr;
    unsigned long long* d_tile_sum = nullptr; unsigned long long* d_grand = nullptr;
    u8* d_lit = nullptr; ck_tool_cfg* d_tool_cfg = nullptr; ck_agent_cfg* d_agent_cfg = nullptr;
    u32* d_counts = nullptr; long long* d_slot_base = nullptr; u32* d_agent_tables = nullptr;
    bool agent_set = false; ck_agent_cfg h_agent_cfg{};
    u32* d_topic_hist = nullptr;
    // aggregation gate (allocated by ck_gate_create)
    ck_gate gate{}; bool gate_set = false; u32* d_rec_entry = nullptr;
    // peer exchange (ck_comm_create)
    u8* d_recv = nullptr; ck_xpeers peers{}; void* peer_opened[CK_X_MAXWORLD] = {nullptr}; u32 comm_rank = 0, comm_world = 0, max_fwd = 0, x_nb = 0;
    unsigned long long region_stride = 0, region_data_cap = 0; u32* d_x_overflow = nullptr; bool comm_ready = false;
    // publish grouping (allocated on first use)
    u32 *d_g_hist = nullptr, *d_g_o1 = nullptr, *d_g_o2 = nullptr, *d_g_keys = nullptr; long long* d_g_base = nullptr; unsigned long long *d_g_tile = nullptr, *d_g_grand = nullptr;
    bool grouped = false; bool opt_bucket = false; const u32* cur_perm = nullptr;
    // Kafka record-batch framing (allocated on first use)
    long long *d_rb_batch_off = nullptr, *d_rb_rec_pos = nullptr, *d_rb_key_off = nullptr, *d_rb_corr_off = nullptr, *d_rb_rec_off = nullptr, *d_rb_frame_len = nullptr;
    u32 *d_rb_rec_base = nullptr, *d_rb_batch_bad = nullptr, *d_rb_rec_batch = nullptr, *d_rb_val_len = nullptr, *d_rb_rec_bad = nullptr, *d_rb_idx = nullptr, *d_rb_sizes = nullptr, *d_rb_partial = nullptr;
    int *d_rb_key_len = nullptr, *d_rb_corr_len = nullptr; u8* d_rb_frame = nullptr; uint64_t rb_frame_cap = 0; uint32_t rb_n = 0;
    long long *d_rb_slot = nullptr, *d_rb_sec_off = nullptr; u32 *d_rb_dlen = nullptr, *d_rb_sec_len = nullptr;   // compressed batches
    uint64_t rb_dbase = 0, rb_dlen = 0;      // decompressed sections of the last fetch: d_in[rb_dbase .. + rb_dlen)
    // runs of frames on the produce side (ck_encode_recordbatches, allocated on first use)
    u32 *d_rbs_idx = nullptr, *d_rbs_goff = nullptr, *d_rbs_delta = nullptr, *d_rbs_size = nullptr, *d_rbs_open = nullptr, *d_rbs_fid = nullptr;
    u32 *d_rbs_ffirst = nullptr, *d_rbs_nch = nullptr, *d_rbs_csz = nullptr, *d_rbs_ccrc = nullptr, *d_rbs_fsize = nullptr, *d_rbs_fgroup = nullptr, *d_rbs_tabs = nullptr;
    long long *d_rbs_base = nullptr, *d_rbs_recoff = nullptr, *d_rbs_openx = nullptr, *d_rbs_foff = nullptr, *d_rbs_cbase = nullptr, *d_rbs_coff = nullptr;
    u8 *d_rbs_plain = nullptr, *d_rbs_slots = nullptr, *d_rbs_out = nullptr; ck_dfl_tables* d_rbs_dtabs = nullptr;
    unsigned long long *d_rbs_tile = nullptr, *d_rbs_grand = nullptr, *h_rbs = nullptr;   // h_rbs: pinned
    uint64_t rbs_plain_cap = 0, rbs_out_cap = 0, rbs_chunk_cap = 0, rbs_total = 0; uint32_t rbs_pool = 0, rbs_nf = 0;
    // exchange planning (allocated on first use)
    u32* d_x_hist = nullptr; long long* d_x_base = nullptr; unsigned long long* d_x_nbytes = nullptr;
    long long *d_x_src_off = nullptr, *d_x_len = nullptr, *d_x_dst_off = nullptr; u32 *d_x_len32 = nullptr, *d_x_pub = nullptr;
    unsigned long long *d_x_tile = nullptr, *d_x_grand = nullptr, *d_x_grand2 = nullptr; long long* h_x = nullptr;   // h_x: pinned
    // topic table
    ck_topic_table tab{}; u32 *d_tab_hash = nullptr, *d_tab_off = nullptr, *d_tab_len = nullptr; int32_t* d_tab_id = nullptr; u8* d_tab_names = nullptr;
    uint32_t num_partitions = 0, hist_cap = 0;
    // current batch
    const u8* cur_in = nullptr; const long long* cur_in_off = nullptr; const u32* cur_len = nullptr;
    uint32_t n = 0, n_payloads = 0, n_pubs = 0;
    bool tool_set = false; ck_tool_cfg h_tool_cfg{};
    unsigned long long n_launch = 0;
    unsigned long long* h_grand = nullptr;   // pinned
    // profiling: asynchronous event pairs around every kernel, read back (and summed) on demand so
    // that timing the kernels does not serialise the stream during a timed region
    bool profile = false;
    std::vector<cudaEvent_t> ev_pool;                    // 2 events per recorded launch
    std::vector<int> ev_kernel;                          // kernel id of each recorded pair
    size_t ev_used = 0;
    float k_ms[CK_NUM_KERNELS] = {0}; uint32_t k_n[CK_NUM_KERNELS] = {0};
};

#define CUDA_TRY(h, call) do { cudaError_t e_ = (call); if (e_ != cudaSuccess) { \
    char b_[512]; snprintf(b_, sizeof b_, "%s failed: %s (%s:%d)", #call, cudaGetErrorString(e_), __FILE__, __LINE__); \
    (h)->err = b_; return 1; } } while (0)

#define CKL(h) (h)->n_launch++,          // every kernel launch is counted (ck_launch_count: bench.py's gpu_launches)
static int fail(ck_handle* h, const char* msg) { h->err = msg; return 1; }

struct KTimer {
    ck_handle* h; int k; size_t slot;
    KTimer(ck_handle* hh, int kk) : h(hh), k(kk), slot(0) {
        if (!h->profile) return;
        if (h->ev_used + 2 > h->ev_pool.size()) {
            for (int j = 0; j < 64; j++) { cudaEvent_t e; cudaEventCreate(&e); h->ev_pool.push_back(e); }
        }
        slot = h->ev_used; h->ev_used += 2; h->ev_kernel.push_back(k);
        cudaEventRecord(h->ev_pool[slot], h->stream);
    }
    ~KTimer() { if (h->profile) cudaEventRecord(h->ev_pool[slot + 1], h->stream); }
};
static void profile_collect(ck_handle* h) {
    cudaStreamSynchronize(h->stream);
    for (size_t p = 0; p * 2 < h->ev_used; p++) {
        float ms = 0;
        if (cudaEventElapsedTime(&ms, h->ev_pool[2 * p], h->ev_pool[2 * p + 1]) == cudaSuccess) { h->k_ms[h->ev_kernel[p]] += ms; h->k_n[h->ev_kernel[p]]++; }
    }
    h->ev_used = 0; h->ev_kernel.clear();
}

extern "C" int ck_version(void) { return 1; }

extern "C" const char* ck_last_error(ck_handle* h) { return h ? h->err.c_str() : g_create_error.c_str(); }

extern "C" int ck_create(int device, uint64_t max_in_bytes, uint64_t max_out_bytes, uint32_t max_records,
                         uint32_t max_payloads, uint64_t max_aux_bytes, ck_handle** out) {
    *out = nullptr;
    ck_handle* h = new ck_handle();
    auto bail = [&](const char* what, cudaError_t e) {
        char b[512]; snprintf(b, sizeof b, "ck_create: %s: %s", what, cudaGetErrorString(e));
        g_create_error = b; ck_destroy(h); return 1;
    };
    cudaError_t e;
    h->device = device;
    if ((e = cudaSetDevice(device)) != cudaSuccess) return bail("cudaSetDevice", e);
    cudaDeviceProp prop;
    if ((e = cudaGetDeviceProperties(&prop, device)) != cudaSuccess) return bail("cudaGetDeviceProperties", e);
    if (prop.major != 10) { g_create_error = "ck_create: this library is built for sm_100a (B200) only"; ck_destroy(h); return 1; }
    if ((e = cudaStreamCreateWithFlags(&h->stream, cudaStreamNonBlocking)) != cudaSuccess) return bail("cudaStreamCreate", e);
    {   // the canonicaliser is (boundedly) recursive: give device threads room for its frames
        size_t cur = 0; cudaDeviceGetLimit(&cur, cudaLimitStackSize);
        if (cur < 12 * 1024 && (e = cudaDeviceSetLimit(cudaLimitStackSize, 12 * 1024)) != cudaSuccess) return bail("cudaDeviceSetLimit(stack)", e);
    }
    h->max_in = max_in_bytes; h->max_out = max_out_bytes; h->max_aux = max_aux_bytes; h->max_records = max_records;
    h->max_payloads = max_payloads > max_records ? max_payloads : max_records; h->max_pubs = 2 * h->max_payloads;
#define ALLOC(p, bytes) if ((e = cudaMalloc((void**)&(p), (bytes))) != cudaSuccess) return bail("cudaMalloc " #p, e)
    ALLOC(h->d_in, max_in_bytes + CK_PAD);
    ALLOC(h->d_in_off, sizeof(long long) * ((size_t)max_records + 1));
    ALLOC(h->d_out, max_out_bytes + CK_PAD);
    ALLOC(h->d_out_off, sizeof(long long) * ((size_t)h->max_payloads + 1));
    ALLOC(h->d_aux, max_aux_bytes + CK_PAD);
    ALLOC(h->d_aux_off, sizeof(long long) * ((size_t)max_records + 1));
    ALLOC(h->d_glue, (size_t)CK_GLUE_STRIDE * h->max_payloads + CK_PAD);
    h->max_ovl = max_in_bytes;
    ALLOC(h->d_ovl, h->max_ovl + CK_PAD);
    ALLOC(h->d_ovl_off, sizeof(long long) * ((size_t)max_records + 1));
    ALLOC(h->d_ovl_len, sizeof(u32) * (size_t)max_records);
    ALLOC(h->d_canon_ctl, sizeof(ck_canon_ctl));
    ALLOC(h->d_canon_list, sizeof(u32) * (size_t)max_records);
    // list elements of long records walked one per thread: a message of a history is rarely shorter than a few hundred bytes
    // (a full list only means the remaining ones are walked inside their record's warp)
    { unsigned long long cap = max_in_bytes / 256 + 1024; if (cap > 0x7fffffffull) cap = 0x7fffffffull; h->elem_cap = (u32)cap; }
    ALLOC(h->d_elems, sizeof(ck_elem) * (size_t)h->elem_cap);
    ALLOC(h->d_cand, sizeof(u32) * (size_t)max_records);
    ALLOC(h->d_hist_skip, sizeof(uint2) * (size_t)max_records);
    ALLOC(h->d_cols, sizeof(u32) * (size_t)CK_NUM_COLS * max_records);
    ALLOC(h->d_descs, sizeof(ck_out_desc) * (size_t)h->max_payloads);
    ALLOC(h->d_pay_len, sizeof(u32) * (size_t)h->max_payloads);
    ALLOC(h->d_pubs, sizeof(ck_pub) * (size_t)h->max_pubs);
    ALLOC(h->d_tile_sum, sizeof(unsigned long long) * ((size_t)h->max_payloads / CK_SCAN_TILE + 2));
    ALLOC(h->d_grand, sizeof(unsigned long long));
    ALLOC(h->d_lit, CK_LIT_CAP + CK_PAD);
    ALLOC(h->d_tool_cfg, sizeof(ck_tool_cfg));
    ALLOC(h->d_agent_cfg, sizeof(ck_agent_cfg));
    ALLOC(h->d_counts, sizeof(u32) * (size_t)max_records);
    ALLOC(h->d_slot_base, sizeof(long long) * ((size_t)max_records + 1));
    h->hist_cap = 4096;
    ALLOC(h->d_topic_hist, sizeof(u32) * h->hist_cap);
#undef ALLOC
    cudaMemsetAsync(h->d_in + max_in_bytes, 0, CK_PAD, h->stream);
    cudaMemsetAsync(h->d_topic_hist, 0, sizeof(u32) * h->hist_cap, h->stream);
    if ((e = cudaMallocHost((void**)&h->h_grand, sizeof(unsigned long long))) != cudaSuccess) return bail("cudaMallocHost", e);
    if ((e = cudaStreamSynchronize(h->stream)) != cudaSuccess) return bail("init sync", e);
    *out = h;
    return 0;
}

extern "C" void ck_destroy(ck_handle* h) {
    if (!h) return;
    cudaSetDevice(h->device);
    if (h->stream) cudaStreamSynchronize(h->stream);
    void* ptrs[] = {h->d_in, h->d_in_off, h->d_out, h->d_out_off, h->d_aux, h->d_aux_off, h->d_glue, h->d_ovl, h->d_ovl_off, h->d_ovl_len, h->d_canon_ctl, h->d_canon_list, h->d_elems, h->d_cand, h->d_hist_skip, h->d_cols, h->d_descs, h->d_pay_len,
                    h->d_pubs, h->d_tile_sum, h->d_grand, h->d_lit, h->d_tool_cfg, h->d_agent_cfg, h->d_counts, h->d_slot_base, h->d_agent_tables, h->d_topic_hist, h->d_tab_hash, h->d_tab_off,
                    h->d_tab_len, h->d_tab_id, h->d_tab_names, h->d_x_hist, h->d_x_base, h->d_x_nbytes, h->d_x_src_off, h->d_x_len, h->d_x_dst_off,
                    h->d_x_len32, h->d_x_pub, h->d_x_tile, h->d_x_grand, h->d_x_grand2};
    for (void* p : ptrs) if (p) cudaFree(p);
    void* gptrs[] = {h->gate.keys, h->gate.vals, h->gate.entries, h->gate.slots, h->gate.arena, h->gate.ctr, h->d_rec_entry,
                     h->d_rb_batch_off, h->d_rb_rec_pos, h->d_rb_key_off, h->d_rb_corr_off, h->d_rb_rec_off, h->d_rb_frame_len, h->d_rb_rec_base, h->d_rb_batch_bad,
                     h->d_g_hist, h->d_g_o1, h->d_g_o2, h->d_g_keys, h->d_g_base, h->d_g_tile, h->d_g_grand,
                     h->d_rb_rec_batch, h->d_rb_val_len, h->d_rb_rec_bad, h->d_rb_idx, h->d_rb_sizes, h->d_rb_partial, h->d_rb_key_len, h->d_rb_corr_len, h->d_rb_frame,
                     h->d_rb_slot, h->d_rb_sec_off, h->d_rb_dlen, h->d_rb_sec_len,
                     h->d_rbs_idx, h->d_rbs_goff, h->d_rbs_delta, h->d_rbs_size, h->d_rbs_open, h->d_rbs_fid, h->d_rbs_ffirst, h->d_rbs_nch,
                     h->d_rbs_csz, h->d_rbs_ccrc, h->d_rbs_fsize, h->d_rbs_fgroup, h->d_rbs_tabs, h->d_rbs_base, h->d_rbs_recoff, h->d_rbs_openx,
                     h->d_rbs_foff, h->d_rbs_cbase, h->d_rbs_coff, h->d_rbs_plain, h->d_rbs_slots, h->d_rbs_out, h->d_rbs_dtabs, h->d_rbs_tile,
                     h->d_rbs_grand};
    for (void* p : gptrs) if (p) cudaFree(p);
    if (h->h_rbs) cudaFreeHost(h->h_rbs);
    for (u32 d = 0; d < CK_X_MAXWORLD; d++) if (h->peer_opened[d]) cudaIpcCloseMemHandle(h->peer_opened[d]);
    if (h->d_recv) cudaFree(h->d_recv);
    if (h->d_x_overflow) cudaFree(h->d_x_overflow);
    if (h->h_grand) cudaFreeHost(h->h_grand);
    if (h->h_x) cudaFreeHost(h->h_x);
    for (cudaEvent_t e : h->ev_pool) cudaEventDestroy(e);
    if (h->xstream) { cudaStreamSynchronize(h->xstream); cudaStreamDestroy(h->xstream); }
    if (h->x_ev0) cudaEventDestroy(h->x_ev0);
    if (h->x_ev1) cudaEventDestroy(h->x_ev1);
    if (h->stream) cudaStreamDestroy(h->stream);
    delete h;
}

static u32 host_fnv1a(const u8* p, u32 n) { u32 h = 2166136261u; for (u32 i = 0; i < n; i++) h = (h ^ p[i]) * 16777619u; return h ? h : 1u; }

extern "C" int ck_register_topics(ck_handle* h, const uint8_t* names, const uint32_t* offsets, uint32_t n,
                                  const int32_t* ids, uint32_t num_partitions) {
    cudaSetDevice(h->device);
    u32 cap = 64;
    while (cap < 4 * n) cap <<= 1;
    std::vector<u32> th(cap, 0), toff(cap, 0), tlen(cap, 0);
    std::vector<int32_t> tid(cap, -1);
    for (u32 i = 0; i < n; i++) {
        if (ids[i] < 0) return fail(h, "ck_register_topics: ids must be >= 0");
        u32 len = offsets[i + 1] - offsets[i];
        u32 hh = host_fnv1a(names + offsets[i], len);
        u32 slot = hh & (cap - 1);
        while (th[slot] != 0) {
            if (th[slot] == hh && tlen[slot] == len && memcmp(names + toff[slot], names + offsets[i], len) == 0) break;   // duplicate name: last wins
            slot = (slot + 1) & (cap - 1);
        }
        th[slot] = hh; toff[slot] = offsets[i]; tlen[slot] = len; tid[slot] = ids[i];
    }
    CUDA_TRY(h, cudaStreamSynchronize(h->stream));
    void* olds[] = {h->d_tab_hash, h->d_tab_off, h->d_tab_len, h->d_tab_id, h->d_tab_names};
    for (void* p : olds) if (p) cudaFree(p);
    h->d_tab_hash = h->d_tab_off = h->d_tab_len = nullptr; h->d_tab_id = nullptr; h->d_tab_names = nullptr;
    u32 total = n ? offsets[n] : 0;
    CUDA_TRY(h, cudaMalloc((void**)&h->d_tab_hash, sizeof(u32) * cap));
    CUDA_TRY(h, cudaMalloc((void**)&h->d_tab_off, sizeof(u32) * cap));
    CUDA_TRY(h, cudaMalloc((void**)&h->d_tab_len, sizeof(u32) * cap));
    CUDA_TRY(h, cudaMalloc((void**)&h->d_tab_id, sizeof(int32_t) * cap));
    CUDA_TRY(h, cudaMalloc((void**)&h->d_tab_names, (size_t)total + CK_PAD));
    CUDA_TRY(h, cudaMemcpy(h->d_tab_hash, th.data(), sizeof(u32) * cap, cudaMemcpyHostToDevice));
    CUDA_TRY(h, cudaMemcpy(h->d_tab_off, toff.data(), sizeof(u32) * cap, cudaMemcpyHostToDevice));
    CUDA_TRY(h, cudaMemcpy(h->d_tab_len, tlen.data(), sizeof(u32) * cap, cudaMemcpyHostToDevice));
    CUDA_TRY(h, cudaMemcpy(h->d_tab_id, tid.data(), sizeof(int32_t) * cap, cudaMemcpyHostToDevice));
    if (total) CUDA_TRY(h, cudaMemcpy(h->d_tab_names, names, total, cudaMemcpyHostToDevice));
    h->tab.cap = cap; h->tab.hash = h->d_tab_hash; h->tab.id = h->d_tab_id; h->tab.name_off = h->d_tab_off;
    h->tab.name_len = h->d_tab_len; h->tab.names = h->d_tab_names;
    h->num_partitions = num_partitions;
    return 0;
}

extern "C" int ck_set_tool_node(ck_handle* h, int32_t publish_topic_id, uint32_t nparts, const uint32_t* kinds,
                                const uint8_t* blob, const uint32_t* part_offsets) {
    cudaSetDevice(h->device);
    if (nparts > CK_TPL_MAX_PARTS) return fail(h, "ck_set_tool_node: too many template parts");
    std::vector<u8> pool;
    auto put = [&](const char* s, uint32_t out[2]) { out[0] = (u32)pool.size(); out[1] = (u32)strlen(s); pool.insert(pool.end(), s, s + strlen(s)); };
    ck_tool_cfg c{};
    c.publish_topic_id = publish_topic_id;
    put(",\"", c.lit_comma_q); put("\"", c.lit_q); put("\":{\"return_value\":", c.lit_open);
    put(",\"content\":null,\"metadata\":{\"tool_call_id\":\"", c.lit_mid); put("\"},\"kind\":\"tool-return\"}", c.lit_close);
    put("{\"return_value\":", c.lit_value_open);
    c.tpl_nparts = nparts;
    for (u32 k = 0; k < nparts; k++) {
        c.tpl_kind[k] = kinds[k]; c.tpl_off[k] = (u32)pool.size(); c.tpl_len[k] = part_offsets[k + 1] - part_offsets[k];
        pool.insert(pool.end(), blob + part_offsets[k], blob + part_offsets[k + 1]);
    }
    if (pool.size() > CK_LIT_CAP) return fail(h, "ck_set_tool_node: literal pool overflow");
    CUDA_TRY(h, cudaStreamSynchronize(h->stream));
    CUDA_TRY(h, cudaMemcpy(h->d_lit, pool.data(), pool.size(), cudaMemcpyHostToDevice));
    CUDA_TRY(h, cudaMemcpy(h->d_tool_cfg, &c, sizeof c, cudaMemcpyHostToDevice));
    h->h_tool_cfg = c; h->tool_set = true;
    return 0;
}

static ck_view view_of(ck_handle* h) {
    ck_view v; v.in = h->cur_in; v.off = h->cur_in_off; v.ovl = h->d_ovl; v.ovl_off = h->d_ovl_off; v.ovl_len = h->d_ovl_len;
    v.canon_ctl = h->d_canon_ctl; v.canon_list = h->d_canon_list; v.len = h->cur_len; v.perm = h->cur_perm; v.elems = h->d_elems; v.elem_cap = h->elem_cap; v.hist_skip = h->d_hist_skip;
    return v;
}

static int run_scan(ck_handle* h, const u32* len, u32 n, long long* out_off, u32 pad,
                    unsigned long long* tile_sum = nullptr, unsigned long long* grand = nullptr);

static int group_alloc(ck_handle* h) {
    u32 nb_max = (h->max_pubs + CK_G_BLOCK - 1) / CK_G_BLOCK;
    if (!h->d_g_hist) {
        size_t nh = 64 * (size_t)nb_max;
        CUDA_TRY(h, cudaMalloc((void**)&h->d_g_hist, sizeof(u32) * nh));
        CUDA_TRY(h, cudaMalloc((void**)&h->d_g_base, sizeof(long long) * (nh + 1)));
        CUDA_TRY(h, cudaMalloc((void**)&h->d_g_o1, sizeof(u32) * ((size_t)h->max_pubs + 1)));
        CUDA_TRY(h, cudaMalloc((void**)&h->d_g_o2, sizeof(u32) * ((size_t)h->max_pubs + 1)));
        CUDA_TRY(h, cudaMalloc((void**)&h->d_g_keys, sizeof(u32) * CK_G_KEYS));
        CUDA_TRY(h, cudaMalloc((void**)&h->d_g_tile, sizeof(unsigned long long) * (nh / CK_SCAN_TILE + 2)));
        CUDA_TRY(h, cudaMalloc((void**)&h->d_g_grand, sizeof(unsigned long long)));
    }
    return 0;
}

// stable two-pass radix sort of indices 0..n-1 by a 12-bit key -> d_g_o2 (and per-key counts in d_g_keys)
template <class KeyFn>
static int group_sort(ck_handle* h, KeyFn keyf, u32 n, int timer) {
    CUDA_TRY(h, cudaMemsetAsync(h->d_g_keys, 0, sizeof(u32) * CK_G_KEYS, h->stream));
    if (!n) return 0;
    u32 nb = (n + CK_G_BLOCK - 1) / CK_G_BLOCK;
    {
        KTimer t(h, timer);
        CKL(h) ck_group_count_kernel<0, KeyFn><<<nb, CK_G_BLOCK, 0, h->stream>>>(keyf, nullptr, n, h->d_g_hist, h->d_g_keys);
        CUDA_TRY(h, cudaGetLastError());
    }
    if (run_scan(h, h->d_g_hist, 64 * nb, h->d_g_base, 0, h->d_g_tile, h->d_g_grand)) return 1;
    {
        KTimer t(h, timer);
        CKL(h) ck_group_scatter_kernel<0, KeyFn><<<nb, CK_G_BLOCK, 0, h->stream>>>(keyf, nullptr, n, h->d_g_base, h->d_g_o1);
        CKL(h) ck_group_count_kernel<6, KeyFn><<<nb, CK_G_BLOCK, 0, h->stream>>>(keyf, h->d_g_o1, n, h->d_g_hist, h->d_g_keys);
        CUDA_TRY(h, cudaGetLastError());
    }
    if (run_scan(h, h->d_g_hist, 64 * nb, h->d_g_base, 0, h->d_g_tile, h->d_g_grand)) return 1;
    {
        KTimer t(h, timer);
        CKL(h) ck_group_scatter_kernel<6, KeyFn><<<nb, CK_G_BLOCK, 0, h->stream>>>(keyf, h->d_g_o1, n, h->d_g_base, h->d_g_o2);
        CUDA_TRY(h, cudaGetLastError());
    }
    return 0;
}

// decode = walk every submitted record; re-emit the ones that are valid but not canonical into the overlay
// (count -> scan -> write) and walk those again in their canonical spelling
static int launch_decode(ck_handle* h) {
    static int mode = -1;
    if (mode < 0) { const char* e = getenv("CK_WALKER"); mode = (e && !strcmp(e, "global")) ? 2 : 0; }   // development A/B switch
    u32 n = h->n;
    if (!n) return 0;
    ck_view v = view_of(h);
    CUDA_TRY(h, cudaMemsetAsync(h->d_ovl_off, 0xff, sizeof(long long) * (size_t)n, h->stream));      // no overlays yet
    CUDA_TRY(h, cudaMemsetAsync(h->d_canon_ctl, 0, sizeof(ck_canon_ctl), h->stream));
    h->cur_perm = nullptr;
    if (h->opt_bucket && n > 64) {
        if (group_alloc(h)) return 1;
        ck_key_len kf; kf.v = v;
        if (group_sort(h, kf, n, CK_K_WALK)) return 1;
        h->cur_perm = h->d_g_o2;
        v = view_of(h);
    }
    if (mode == 2) v.hist_skip = nullptr;                    // A/B walker: no pre-scan, every list walked in place
    if (mode != 2) {
        // records of CK_HIST_MIN bytes or more, one warp each: structural pre-scan; message_history listed message by message
        // for the element pass, or (long records that are long for another reason) the whole record walked by the warp.
        // Both kernels exit at once when there are no such records.
        KTimer t(h, CK_K_WALK_LONG);
        CKL(h) ck_classify_kernel<<<(n + 255) / 256, 256, 0, h->stream>>>(v, n, h->d_cand);
        u32 lblocks = (n + CK_LONG_WARPS - 1) / CK_LONG_WARPS; if (lblocks > 148 * CK_LONG_MINB) lblocks = 148 * CK_LONG_MINB;
        CKL(h) ck_walk_long_kernel<<<lblocks, 32 * CK_LONG_WARPS, CK_LONG_WARPS * sizeof(ck_long_index), h->stream>>>(v, h->d_cols, n, h->d_cand, h->d_hist_skip);
        CUDA_TRY(h, cudaGetLastError());
    }
    {
        KTimer t(h, CK_K_WALK);
        if (mode == 2) CKL(h) ck_walk_global_kernel<<<(n + 127) / 128, 128, 0, h->stream>>>(v, n, h->d_cols, n, 0);
        else CKL(h) ck_walk_kernel<<<(n + 127) / 128, 128, CK_WALK_THREADS * CK_WIN_STRIDE, h->stream>>>(v, n, h->d_cols, n, 0);
        CUDA_TRY(h, cudaGetLastError());
    }
    {
        // the history messages listed by the pre-scan or deferred by the long walker, one thread each (exits at once when
        // there are none)
        KTimer t(h, CK_K_WALK_ELEMS);
        CKL(h) ck_walk_elems_kernel<<<148 * CK_WALK_MINB, CK_WALK_THREADS, CK_WALK_THREADS * CK_WIN_STRIDE, h->stream>>>(v, h->d_cols, n);
        CUDA_TRY(h, cudaGetLastError());
    }
    {
        // the records the walker listed (usually none: both kernels exit at once) are re-emitted canonically into the
        // overlay and walked again in that spelling
        KTimer t(h, CK_K_CANON);
        u32 blocks = (n + 63) / 64; if (blocks > 148 * 8) blocks = 148 * 8;
        CKL(h) ck_canon_kernel<<<blocks, 64, 0, h->stream>>>(v, n, h->d_cols, n, h->d_ovl, (long long)h->max_ovl, h->d_ovl_off, h->d_ovl_len);
        CKL(h) ck_rewalk_list_kernel<<<blocks, 64, 0, h->stream>>>(v, n, h->d_cols, n);
        CUDA_TRY(h, cudaGetLastError());
    }
    return 0;
}

extern "C" int ck_submit(ck_handle* h, const uint8_t* host_in, const int64_t* host_off, uint32_t n) {
    cudaSetDevice(h->device);
    if (n > h->max_records) return fail(h, "ck_submit: batch has more records than max_records");
    uint64_t nbytes = n ? (uint64_t)(host_off[n] - host_off[0]) : 0;
    if (n && host_off[0] != 0) return fail(h, "ck_submit: offsets must start at 0");
    if (nbytes > h->max_in) return fail(h, "ck_submit: batch larger than max_in_bytes");
    CUDA_TRY(h, cudaMemcpyAsync(h->d_in, host_in, nbytes, cudaMemcpyHostToDevice, h->stream));
    CUDA_TRY(h, cudaMemcpyAsync(h->d_in_off, host_off, sizeof(long long) * ((size_t)n + 1), cudaMemcpyHostToDevice, h->stream));
    CUDA_TRY(h, cudaMemsetAsync(h->d_in + nbytes, 0, 16, h->stream));
    h->cur_in = h->d_in; h->cur_in_off = h->d_in_off; h->cur_len = nullptr; h->n = n; h->n_payloads = 0; h->n_pubs = 0;
    return launch_decode(h);
}

extern "C" int ck_submit_device(ck_handle* h, const uint8_t* dev_in, const int64_t* dev_off, uint32_t n) {
    cudaSetDevice(h->device);
    if (n > h->max_records) return fail(h, "ck_submit_device: batch has more records than max_records");
    h->cur_in = dev_in; h->cur_in_off = (const long long*)dev_off; h->cur_len = nullptr; h->n = n; h->n_payloads = 0; h->n_pubs = 0;
    return launch_decode(h);
}

static int run_scan(ck_handle* h, const u32* len, u32 n, long long* out_off, u32 pad,
                    unsigned long long* tile_sum, unsigned long long* grand) {
    KTimer t(h, CK_K_SCAN);
    if (!tile_sum) { tile_sum = h->d_tile_sum; grand = h->d_grand; }
    u32 ntiles = (n + CK_SCAN_TILE - 1) / CK_SCAN_TILE;
    if (n) {
        CKL(h) ck_scan_tiles_kernel<<<ntiles, CK_SCAN_BLOCK, 0, h->stream>>>(len, n, tile_sum, pad);
        CKL(h) ck_scan_sums_kernel<<<1, CK_SCAN_BLOCK, 0, h->stream>>>(tile_sum, ntiles, grand);
        CKL(h) ck_scan_apply_kernel<<<ntiles, CK_SCAN_BLOCK, 0, h->stream>>>(len, n, tile_sum, out_off, pad);
    }
    CUDA_TRY(h, cudaGetLastError());
    return 0;
}

static int scan_emit(ck_handle* h, u32 npay, const u8* aux) {
    if (run_scan(h, h->d_pay_len, npay, h->d_out_off, 15)) return 1;   // payloads start 16-byte aligned
    {
        KTimer t(h, CK_K_EMIT);
        if (npay) {
            u32 warps_per_block = 256 / 32;
            CKL(h) ck_emit_kernel<<<(npay + warps_per_block - 1) / warps_per_block, 256, 0, h->stream>>>(
                view_of(h), h->d_lit, aux, h->d_glue, h->d_descs, h->d_out_off, npay, h->d_out, (long long)h->max_out);
        }
        CUDA_TRY(h, cudaGetLastError());
    }
    h->n_payloads = npay;
    return 0;
}

extern "C" int ck_tool_args(ck_handle* h) {
    cudaSetDevice(h->device);
    if (!h->tool_set) return fail(h, "ck_tool_args: call ck_set_tool_node first");
    {
        KTimer t(h, CK_K_PLAN);
        if (h->n) CKL(h) ck_plan_tool_kernel<<<(h->n + 127) / 128, 128, 0, h->stream>>>(view_of(h), h->n, h->d_cols, h->n,
            h->d_tool_cfg, h->d_lit, nullptr, nullptr, h->d_glue, 0, h->d_descs, h->d_pay_len, h->d_pubs);
        CUDA_TRY(h, cudaGetLastError());
    }
    h->n_pubs = 0;
    return scan_emit(h, h->n, nullptr);
}

// plan (modes 1 / 2) staged through shared memory, publishes routed in the same kernel (ck_plan2.cuh)
static int launch_plan2(ck_handle* h, const u8* aux, const long long* aux_off, int mode) {
    static bool attr_set = false;
    if (!attr_set) {
        CUDA_TRY(h, cudaFuncSetAttribute(ck_plan_tool2_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)CK_P2_SMEM));
        attr_set = true;
    }
    KTimer t(h, CK_K_PLAN);
    if (h->n) CKL(h) ck_plan_tool2_kernel<<<(h->n + CK_P2_THREADS - 1) / CK_P2_THREADS, CK_P2_THREADS, CK_P2_SMEM, h->stream>>>(
        view_of(h), h->n, h->d_cols, h->n, h->d_tool_cfg, h->d_lit, aux_off, aux, h->d_glue, mode, h->d_descs, h->d_pay_len, h->d_pubs,
        h->tab, h->num_partitions, h->d_topic_hist, h->hist_cap);
    CUDA_TRY(h, cudaGetLastError());
    return 0;
}

static int tool_plan_common(ck_handle* h, const u8* aux, const long long* aux_off) {
    if (!h->tool_set) return fail(h, "ck_tool_plan: call ck_set_tool_node first");
    if (h->h_tool_cfg.tpl_nparts == 0 && aux_off == nullptr) return fail(h, "ck_tool_plan: node has no device template, host results required");
    if (launch_plan2(h, aux, aux_off, 1)) return 1;
    // NOTE: payload sizes are bounded by in + per-record constant; the caller sizes max_out accordingly
    if (scan_emit(h, h->n, aux)) return 1;
    h->n_pubs = 2 * h->n;
    return 0;
}

extern "C" int ck_tool_plan(ck_handle* h, const uint8_t* host_aux, const int64_t* host_aux_off) {
    cudaSetDevice(h->device);
    if (host_aux_off) {
        uint64_t nb = (uint64_t)host_aux_off[h->n];
        if (nb > h->max_aux) return fail(h, "ck_tool_plan: results larger than max_aux_bytes");
        CUDA_TRY(h, cudaMemcpyAsync(h->d_aux, host_aux, nb, cudaMemcpyHostToDevice, h->stream));
        CUDA_TRY(h, cudaMemcpyAsync(h->d_aux_off, host_aux_off, sizeof(long long) * ((size_t)h->n + 1), cudaMemcpyHostToDevice, h->stream));
        return tool_plan_common(h, h->d_aux, h->d_aux_off);
    }
    return tool_plan_common(h, nullptr, nullptr);
}

// ReturnCall of the state as it is on the wire (Agent final output): pop the frame, publish to the
// callback topic and to publish_topic (nodes/base.py:105-118, worker/worker.py:52-53)
extern "C" int ck_return_plan(ck_handle* h) {
    cudaSetDevice(h->device);
    if (!h->tool_set) return fail(h, "ck_return_plan: call ck_set_tool_node (publish topic) first");
    if (launch_plan2(h, nullptr, nullptr, 2)) return 1;
    if (scan_emit(h, h->n, nullptr)) return 1;
    h->n_pubs = 2 * h->n;
    return 0;
}

// client reply decode: payload i = the output value of reply i (see ck_reply_plan_kernel)
extern "C" int ck_reply_plan(ck_handle* h, uint32_t mode) {
    cudaSetDevice(h->device);
    if (mode > 2) return fail(h, "ck_reply_plan: mode must be 0 (auto), 1 (text) or 2 (data)");
    {
        KTimer t(h, CK_K_PLAN);
        if (h->n) CKL(h) ck_reply_plan_kernel<<<(h->n + 127) / 128, 128, 0, h->stream>>>(view_of(h), h->n, h->d_cols, h->n, mode, h->d_glue,
                                                                               h->d_descs, h->d_pay_len);
        CUDA_TRY(h, cudaGetLastError());
    }
    if (scan_emit(h, h->n, nullptr)) return 1;
    h->n_pubs = 0;
    return 0;
}

extern "C" int ck_tool_plan_device(ck_handle* h, const uint8_t* dev_aux, const int64_t* dev_aux_off) {
    cudaSetDevice(h->device);
    return tool_plan_common(h, dev_aux, (const long long*)dev_aux_off);
}

extern "C" int ck_set_agent_node(ck_handle* h, int32_t publish_topic_id, const uint8_t* agent_name, uint32_t agent_name_len,
                                 const uint8_t* callback_topic, uint32_t callback_len,
                                 const uint8_t* tool_names, const uint32_t* tool_name_off,
                                 const uint8_t* tool_topics, const uint32_t* tool_topic_off, uint32_t ntools) {
    // agent_name / callback_topic / tool topics are spliced into JSON strings: the caller passes them
    // already JSON-escaped (the Python binding does); tool_names are compared against raw JSON bytes.
    cudaSetDevice(h->device);
    std::vector<u8> pool;
    auto puts = [&](const std::string& s, uint32_t out[2]) { out[0] = (u32)pool.size(); out[1] = (u32)s.size(); pool.insert(pool.end(), s.begin(), s.end()); };
    ck_agent_cfg c{};
    c.publish_topic_id = publish_topic_id;
    c.ntools = ntools;
    std::string an((const char*)agent_name, agent_name_len), cb((const char*)callback_topic, callback_len);
    puts(",", c.lit_comma);
    puts("\",\"" + an + "\"],\"frame_id\":\"", c.lit_mid);
    puts("\",\"overrides\":null}", c.lit_tail);
    puts("{\"target_topic\":\"" + cb + "\",\"callback_topic\":\"", c.lit_tc_head);
    puts("\",\"input_args\":null,\"frame_id\":\"", c.lit_tc_mid);
    c.self_topic_id = -1;
    std::vector<u32> tab(6 * (size_t)ntools);
    for (u32 k = 0; k < ntools; k++) {
        std::string nm((const char*)tool_names + tool_name_off[k], tool_name_off[k + 1] - tool_name_off[k]);
        std::string tp((const char*)tool_topics + tool_topic_off[k], tool_topic_off[k + 1] - tool_topic_off[k]);
        uint32_t sp[2];
        puts(nm, sp); tab[k] = sp[0]; tab[ntools + k] = sp[1];
        puts("{\"target_topic\":\"" + tp + "\",\"callback_topic\":\"" + cb + "\",\"input_args\":[\"", sp);
        tab[2 * ntools + k] = sp[0]; tab[3 * ntools + k] = sp[1];
        // registered id of the tool's topic, if any (host-side probe of the same table the device uses is
        // not needed: ids are resolved by the route kernel when this is 0xffffffff)
        tab[4 * ntools + k] = 0xffffffffu;
        { std::vector<u64> pad(nm.size() / 8 + 4, 0ull);          // 8-byte aligned, padded: the reader loads whole aligned words
          memcpy((u8*)pad.data() + 8, nm.data(), nm.size());
          GRd hr; hr.init((const u8*)pad.data() + 8, (u32)nm.size());
          tab[5 * ntools + k] = ck_hash_span(hr, 0, (u32)nm.size()); }    // the device compares it with ck_hash_span of the name in the record
    }
    if (pool.size() > CK_LIT_CAP) return fail(h, "ck_set_agent_node: literal pool overflow");
    CUDA_TRY(h, cudaStreamSynchronize(h->stream));
    if (h->d_agent_tables) { cudaFree(h->d_agent_tables); h->d_agent_tables = nullptr; }
    CUDA_TRY(h, cudaMalloc((void**)&h->d_agent_tables, sizeof(u32) * (tab.size() + 1)));
    CUDA_TRY(h, cudaMemcpy(h->d_agent_tables, tab.data(), sizeof(u32) * tab.size(), cudaMemcpyHostToDevice));
    c.tool_name_off = h->d_agent_tables; c.tool_name_len = h->d_agent_tables + ntools;
    c.tool_lit_off = h->d_agent_tables + 2 * ntools; c.tool_lit_len = h->d_agent_tables + 3 * ntools;
    c.tool_topic_id = h->d_agent_tables + 4 * ntools;
    CUDA_TRY(h, cudaMemcpy(h->d_lit, pool.data(), pool.size(), cudaMemcpyHostToDevice));
    CUDA_TRY(h, cudaMemcpy(h->d_agent_cfg, &c, sizeof c, cudaMemcpyHostToDevice));
    h->h_agent_cfg = c; h->agent_set = true;
    return 0;
}

extern "C" int ck_set_agent_tool_topic_ids(ck_handle* h, int32_t self_topic_id, const uint32_t* ids, uint32_t ntools) {
    cudaSetDevice(h->device);
    if (!h->agent_set || ntools != h->h_agent_cfg.ntools) return fail(h, "ck_set_agent_tool_topic_ids: agent node not set / size mismatch");
    CUDA_TRY(h, cudaStreamSynchronize(h->stream));
    if (ntools) CUDA_TRY(h, cudaMemcpy(h->d_agent_tables + 4 * (size_t)ntools, ids, sizeof(u32) * ntools, cudaMemcpyHostToDevice));
    h->h_agent_cfg.self_topic_id = self_topic_id;
    CUDA_TRY(h, cudaMemcpy(h->d_agent_cfg, &h->h_agent_cfg, sizeof h->h_agent_cfg, cudaMemcpyHostToDevice));
    return 0;
}

extern "C" int ck_tailcall_plan(ck_handle* h, uint64_t unix_ms, uint64_t seed) {
    cudaSetDevice(h->device);
    if (!h->agent_set) return fail(h, "ck_tailcall_plan: call ck_set_agent_node first");
    if (h->h_agent_cfg.self_topic_id < 0) return fail(h, "ck_tailcall_plan: the agent's own topic is not registered");
    u32 n = h->n;
    if (n > h->max_payloads) return fail(h, "ck_tailcall_plan: more payloads than max_payloads");
    {
        KTimer t(h, CK_K_FANOUT);
        if (n) CKL(h) ck_tailcall_plan_kernel<<<(n + 127) / 128, 128, 0, h->stream>>>(view_of(h), n, h->d_cols, n, h->d_agent_cfg, h->d_lit,
            unix_ms, seed, h->d_aux, h->d_glue, h->d_descs, h->d_pay_len, h->d_pubs);
        CUDA_TRY(h, cudaGetLastError());
    }
    if (scan_emit(h, n, h->d_aux)) return 1;
    {
        KTimer t(h, CK_K_ROUTE);
        u32 npubs = 2 * n;
        if (npubs) CKL(h) ck_route_kernel<<<(npubs + 255) / 256, 256, 0, h->stream>>>(view_of(h), h->d_cols, n, h->d_pubs, npubs,
            h->tab, h->num_partitions, h->d_topic_hist, h->hist_cap);
        CUDA_TRY(h, cudaGetLastError());
        h->n_pubs = npubs;
    }
    return 0;
}

extern "C" int ck_fanout_plan(ck_handle* h, uint64_t unix_ms, uint64_t seed, uint32_t max_fanout, uint32_t sequential) {
    cudaSetDevice(h->device);
    if (!h->agent_set) return fail(h, "ck_fanout_plan: call ck_set_agent_node first");
    u32 n = h->n;
    {
        KTimer t(h, CK_K_FANOUT);
        static bool f2_attr = false;
        if (!f2_attr) {
            CUDA_TRY(h, cudaFuncSetAttribute(ck_fanout2_count_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)CK_F2_SMEM));
            CUDA_TRY(h, cudaFuncSetAttribute(ck_fanout2_plan_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)CK_F2_SMEM));
            f2_attr = true;
        }
        if (n) CKL(h) ck_fanout2_count_kernel<<<(n + CK_F2_WARPS - 1) / CK_F2_WARPS, 32 * CK_F2_WARPS, CK_F2_SMEM, h->stream>>>(view_of(h), n, h->d_cols, n, h->d_agent_cfg,
                                                                                                             max_fanout, sequential, h->d_counts);
        CUDA_TRY(h, cudaGetLastError());
    }
    if (run_scan(h, h->d_counts, n, h->d_slot_base, 0)) return 1;
    *h->h_grand = 0;
    if (n) CUDA_TRY(h, cudaMemcpyAsync(h->h_grand, h->d_grand, sizeof(unsigned long long), cudaMemcpyDeviceToHost, h->stream));
    CUDA_TRY(h, cudaStreamSynchronize(h->stream));
    unsigned long long slots = *h->h_grand;
    if (slots > h->max_payloads) return fail(h, "ck_fanout_plan: more payloads than max_payloads");
    {
        KTimer t(h, CK_K_FANOUT);
        if (n) CKL(h) ck_fanout2_plan_kernel<<<(n + CK_F2_WARPS - 1) / CK_F2_WARPS, 32 * CK_F2_WARPS, CK_F2_SMEM, h->stream>>>(view_of(h), n, h->d_cols, n, h->d_agent_cfg, h->d_lit,
            h->d_agent_tables + 5 * (size_t)h->h_agent_cfg.ntools, h->d_slot_base, unix_ms, seed, h->d_aux, h->d_glue, h->d_descs, h->d_pay_len, h->d_pubs);
        CUDA_TRY(h, cudaGetLastError());
    }
    if (scan_emit(h, (u32)slots, h->d_aux)) return 1;
    {
        KTimer t(h, CK_K_ROUTE);
        u32 npubs = 2 * (u32)slots;
        if (npubs) CKL(h) ck_route_kernel<<<(npubs + 255) / 256, 256, 0, h->stream>>>(view_of(h), h->d_cols, n, h->d_pubs, npubs,
            h->tab, h->num_partitions, h->d_topic_hist, h->hist_cap);
        CUDA_TRY(h, cudaGetLastError());
        h->n_pubs = npubs;
    }
    return 0;
}

// ---- grouping the publish table by topic (csrc/ck_group.cuh) ---------------------------------------------------------------
extern "C" int ck_group_publishes(ck_handle* h) {
    cudaSetDevice(h->device);
    if (group_alloc(h)) return 1;
    h->grouped = true;
    ck_key_pub kf; kf.pubs = h->d_pubs; kf.rank = h->comm_rank; kf.world = h->comm_ready ? h->comm_world : 1;
    return group_sort(h, kf, h->n_pubs, CK_K_ROUTE);
}

// engine options.  CK_OPT_BUCKET (1): bucket every submitted batch by record length before the thread-per-record walk —
// for topics that carry records of mixed sizes / shapes (a warp takes as long as its longest record, and lanes on
// different schema branches run one after the other); homogeneous batches do not need it (it costs six small launches).
extern "C" int ck_set_option(ck_handle* h, uint32_t option, uint64_t value) {
    if (option == 1) { h->opt_bucket = value != 0; return 0; }
    return fail(h, "ck_set_option: unknown option");
}

// order[n_publishes]: publish indices grouped by key (0 = unregistered topic, 1 + id = registered topic id, 4095 = unused
// slot), send order kept inside a group; key_counts[4096].  wait = 0: copies queued only (page-locked destinations).
extern "C" int ck_fetch_groups(ck_handle* h, uint32_t* host_order, uint32_t* host_key_counts, int wait) {
    cudaSetDevice(h->device);
    if (!h->grouped) return fail(h, "ck_fetch_groups: call ck_group_publishes first");
    if (h->n_pubs) CUDA_TRY(h, cudaMemcpyAsync(host_order, h->d_g_o2, sizeof(u32) * (size_t)h->n_pubs, cudaMemcpyDeviceToHost, h->stream));
    CUDA_TRY(h, cudaMemcpyAsync(host_key_counts, h->d_g_keys, sizeof(u32) * CK_G_KEYS, cudaMemcpyDeviceToHost, h->stream));
    if (wait) CUDA_TRY(h, cudaStreamSynchronize(h->stream));
    return 0;
}

// ---- Kafka RecordBatch v2 framing (csrc/ck_kafka.cuh) -------------------------------------------------------------------
static int rb_alloc(ck_handle* h) {
    if (h->d_rb_batch_off) return 0;
    size_t mr = (size_t)h->max_records + 1;
    CUDA_TRY(h, cudaMalloc((void**)&h->d_rb_batch_off, sizeof(long long) * mr));
    CUDA_TRY(h, cudaMalloc((void**)&h->d_rb_rec_base, sizeof(u32) * mr));
    CUDA_TRY(h, cudaMalloc((void**)&h->d_rb_batch_bad, sizeof(u32) * mr));
    CUDA_TRY(h, cudaMalloc((void**)&h->d_rb_rec_pos, sizeof(long long) * mr));
    CUDA_TRY(h, cudaMalloc((void**)&h->d_rb_rec_batch, sizeof(u32) * mr));
    CUDA_TRY(h, cudaMalloc((void**)&h->d_rb_val_len, sizeof(u32) * mr));
    CUDA_TRY(h, cudaMalloc((void**)&h->d_rb_key_off, sizeof(long long) * mr));
    CUDA_TRY(h, cudaMalloc((void**)&h->d_rb_key_len, sizeof(int) * mr));
    CUDA_TRY(h, cudaMalloc((void**)&h->d_rb_corr_off, sizeof(long long) * mr));
    CUDA_TRY(h, cudaMalloc((void**)&h->d_rb_corr_len, sizeof(int) * mr));
    CUDA_TRY(h, cudaMalloc((void**)&h->d_rb_rec_bad, sizeof(u32) * mr));
    return 0;
}
static int rb_alloc_codec(ck_handle* h) {
    if (h->d_rb_slot) return 0;
    size_t mr = (size_t)h->max_records + 1;
    CUDA_TRY(h, cudaMalloc((void**)&h->d_rb_slot, sizeof(long long) * (mr + 1)));
    CUDA_TRY(h, cudaMalloc((void**)&h->d_rb_sec_off, sizeof(long long) * mr));
    CUDA_TRY(h, cudaMalloc((void**)&h->d_rb_dlen, sizeof(u32) * mr));
    CUDA_TRY(h, cudaMalloc((void**)&h->d_rb_sec_len, sizeof(u32) * mr));
    return 0;
}
static inline uint32_t host_be32(const uint8_t* p) { return ((uint32_t)p[0] << 24) | ((uint32_t)p[1] << 16) | ((uint32_t)p[2] << 8) | p[3]; }

// A fetch response's record set (concatenated RecordBatch v2 frames, as it came off the socket) goes to HBM in one copy;
// CRC32C check, record split and varint field decode run on the device and the walker reads every value where it lies.
// The host only chains through the frame headers (12 + batchLength bytes each) to index the frames.
// Frames compressed with gzip (codec 1) or LZ4 (codec 3) are decompressed on the device into 16-byte aligned slots of
// the input buffer right after the submitted bytes; their records are read there.  Such a fetch costs one more host
// synchronisation (the decompressed total, to check it against max_in_bytes); a fetch without them takes the same path
// as before.  Other codecs (snappy, zstd) leave their frames bad with reason CK_RB_BAD_CODEC.
extern "C" int ck_submit_recordbatch(ck_handle* h, const uint8_t* host_buf, uint64_t nbytes, uint32_t* n_records) {
    cudaSetDevice(h->device);
    if (nbytes > h->max_in) return fail(h, "ck_submit_recordbatch: buffer larger than max_in_bytes");
    if (rb_alloc(h)) return 1;
    std::vector<long long> boff; std::vector<u32> rbase;
    uint64_t pos = 0; uint64_t total = 0;
    bool compressed = false;
    while (pos + 12 <= nbytes) {
        uint32_t blen = host_be32(host_buf + pos + 8);
        uint64_t end = pos + 12 + (uint64_t)blen;
        if ((int32_t)blen < (int32_t)(CK_RB_HEADER - 12) || end > nbytes) break;         // truncated trailing frame: legal in a fetch response
        uint32_t cnt = host_be32(host_buf + pos + 57);
        if (total + cnt > h->max_records) return fail(h, "ck_submit_recordbatch: more records than max_records");
        uint32_t codec = host_buf[pos + 22] & 7u;
        compressed |= codec == CK_RB_GZIP || codec == CK_RB_LZ4;
        boff.push_back((long long)pos); rbase.push_back((u32)total);
        total += cnt; pos = end;
    }
    boff.push_back((long long)pos); rbase.push_back((u32)total);
    u32 nb = (u32)boff.size() - 1, n = (u32)total;
    if (n_records) *n_records = n;
    if (compressed && rb_alloc_codec(h)) return 1;
    h->rb_dbase = 0; h->rb_dlen = 0;
    CUDA_TRY(h, cudaMemcpyAsync(h->d_in, host_buf, pos, cudaMemcpyHostToDevice, h->stream));
    CUDA_TRY(h, cudaMemsetAsync(h->d_in + pos, 0, 16, h->stream));
    CUDA_TRY(h, cudaMemcpyAsync(h->d_rb_batch_off, boff.data(), sizeof(long long) * (nb + 1), cudaMemcpyHostToDevice, h->stream));
    CUDA_TRY(h, cudaMemcpyAsync(h->d_rb_rec_base, rbase.data(), sizeof(u32) * (nb + 1), cudaMemcpyHostToDevice, h->stream));
    CUDA_TRY(h, cudaStreamSynchronize(h->stream));           // the two index vectors are pageable stack objects
    h->rb_n = n;
    if (nb && !compressed) {
        KTimer t(h, CK_K_WALK);
        CKL(h) ck_rb_crc_kernel<<<(nb + 7) / 8, 256, 0, h->stream>>>(h->d_in, h->d_rb_batch_off, nb, h->d_rb_batch_bad);
        CKL(h) ck_rb_split_kernel<<<(nb + 127) / 128, 128, 0, h->stream>>>(h->d_in, h->d_rb_batch_off, h->d_rb_rec_base, nb, nullptr, nullptr,
                                                                        h->d_rb_batch_bad, h->d_rb_rec_pos, h->d_rb_rec_batch);
        if (n) CKL(h) ck_rb_fields_kernel<<<(n + 127) / 128, 128, 0, h->stream>>>(h->d_in, (long long)pos, h->d_rb_rec_pos, h->d_rb_rec_batch, h->d_rb_batch_bad, n,
            h->d_in_off, h->d_rb_val_len, h->d_rb_key_off, h->d_rb_key_len, h->d_rb_corr_off, h->d_rb_corr_len, h->d_rb_rec_bad);
        CUDA_TRY(h, cudaGetLastError());
    } else if (nb) {
        // CRC, size pass, scan of the slot sizes, capacity check (the one extra synchronisation), decompress, split
        {
            KTimer t(h, CK_K_WALK);
            CKL(h) ck_rb_crc_kernel<<<(nb + 7) / 8, 256, 0, h->stream>>>(h->d_in, h->d_rb_batch_off, nb, h->d_rb_batch_bad);
            CUDA_TRY(h, cudaGetLastError());
        }
        {
            KTimer t(h, CK_K_CODEC);
            CKL(h) ck_rb_csize_kernel<<<(nb + 127) / 128, 128, 0, h->stream>>>(h->d_in, h->d_rb_batch_off, nb, h->d_rb_batch_bad, h->d_rb_dlen);
            CUDA_TRY(h, cudaGetLastError());
        }
        if (run_scan(h, h->d_rb_dlen, nb, h->d_rb_slot, 15)) return 1;
        unsigned long long dtotal = 0;
        CUDA_TRY(h, cudaMemcpyAsync(h->h_grand, h->d_grand, sizeof(unsigned long long), cudaMemcpyDeviceToHost, h->stream));
        CUDA_TRY(h, cudaStreamSynchronize(h->stream));
        dtotal = *h->h_grand;
        uint64_t dbase = (pos + 15) & ~15ull;
        if (dbase + dtotal > h->max_in) {
            char b[256];
            snprintf(b, sizeof b, "ck_submit_recordbatch: %llu submitted + %llu decompressed bytes (with padding) exceed max_in_bytes = %llu",
                     (unsigned long long)pos, dtotal, (unsigned long long)h->max_in);
            h->rb_n = 0; h->n = 0;
            return fail(h, b);
        }
        {
            KTimer t(h, CK_K_CODEC);
            CKL(h) ck_rb_decompress_kernel<<<(nb + 127) / 128, 128, 0, h->stream>>>(h->d_in, h->d_rb_batch_off, nb, (long long)dbase, h->d_rb_slot,
                                                                                 h->d_rb_dlen, h->d_rb_batch_bad, h->d_rb_sec_off, h->d_rb_sec_len);
            CUDA_TRY(h, cudaGetLastError());
        }
        CUDA_TRY(h, cudaMemsetAsync(h->d_in + dbase + dtotal, 0, 16, h->stream));
        h->rb_dbase = dbase; h->rb_dlen = dtotal;
        {
            KTimer t(h, CK_K_WALK);
            CKL(h) ck_rb_split_kernel<<<(nb + 127) / 128, 128, 0, h->stream>>>(h->d_in, h->d_rb_batch_off, h->d_rb_rec_base, nb, h->d_rb_sec_off,
                                                                            h->d_rb_sec_len, h->d_rb_batch_bad, h->d_rb_rec_pos, h->d_rb_rec_batch);
            if (n) CKL(h) ck_rb_fields_kernel<<<(n + 127) / 128, 128, 0, h->stream>>>(h->d_in, (long long)(dbase + dtotal), h->d_rb_rec_pos, h->d_rb_rec_batch,
                h->d_rb_batch_bad, n, h->d_in_off, h->d_rb_val_len, h->d_rb_key_off, h->d_rb_key_len, h->d_rb_corr_off, h->d_rb_corr_len, h->d_rb_rec_bad);
            CUDA_TRY(h, cudaGetLastError());
        }
    }
    h->cur_in = h->d_in; h->cur_in_off = h->d_in_off; h->cur_len = h->d_rb_val_len; h->n = n; h->n_payloads = 0; h->n_pubs = 0;
    if (launch_decode(h)) return 1;
    if (n) { CKL(h) ck_rb_mark_bad_kernel<<<(n + 255) / 256, 256, 0, h->stream>>>(h->d_rb_rec_bad, n, h->d_cols, n); CUDA_TRY(h, cudaGetLastError()); }
    return 0;
}

// the decompressed records sections of the last ck_submit_recordbatch: host_dst[0 .. *len) = input bytes [*base, *base + *len)
// (the offsets ck_fetch_rb_index reports for records of compressed frames lie there); *len = 0 when no frame was compressed
extern "C" int ck_fetch_rb_decompressed(ck_handle* h, uint8_t* host_dst, uint64_t cap, uint64_t* base, uint64_t* len) {
    cudaSetDevice(h->device);
    if (base) *base = h->rb_dbase;
    if (len) *len = h->rb_dlen;
    if (!h->rb_dlen || !host_dst) return 0;
    if (h->rb_dlen > cap) return fail(h, "ck_fetch_rb_decompressed: host buffer too small");
    CUDA_TRY(h, cudaMemcpyAsync(host_dst, h->d_in + h->rb_dbase, h->rb_dlen, cudaMemcpyDeviceToHost, h->stream));
    CUDA_TRY(h, cudaStreamSynchronize(h->stream));
    return 0;
}

// per record of the last ck_submit_recordbatch: where value / key / correlation_id header lie in the submitted buffer
// (key_len / corr_len = -1: absent), and whether its frame failed the CRC / framing check
extern "C" int ck_fetch_rb_index(ck_handle* h, int64_t* val_off, uint32_t* val_len, int64_t* key_off, int32_t* key_len,
                                 int64_t* corr_off, int32_t* corr_len, uint32_t* bad) {
    cudaSetDevice(h->device);
    u32 n = h->rb_n;
    if (!n) return 0;
    if (val_off) CUDA_TRY(h, cudaMemcpyAsync(val_off, h->d_in_off, sizeof(long long) * n, cudaMemcpyDeviceToHost, h->stream));
    if (val_len) CUDA_TRY(h, cudaMemcpyAsync(val_len, h->d_rb_val_len, sizeof(u32) * n, cudaMemcpyDeviceToHost, h->stream));
    if (key_off) CUDA_TRY(h, cudaMemcpyAsync(key_off, h->d_rb_key_off, sizeof(long long) * n, cudaMemcpyDeviceToHost, h->stream));
    if (key_len) CUDA_TRY(h, cudaMemcpyAsync(key_len, h->d_rb_key_len, sizeof(int) * n, cudaMemcpyDeviceToHost, h->stream));
    if (corr_off) CUDA_TRY(h, cudaMemcpyAsync(corr_off, h->d_rb_corr_off, sizeof(long long) * n, cudaMemcpyDeviceToHost, h->stream));
    if (corr_len) CUDA_TRY(h, cudaMemcpyAsync(corr_len, h->d_rb_corr_len, sizeof(int) * n, cudaMemcpyDeviceToHost, h->stream));
    if (bad) CUDA_TRY(h, cudaMemcpyAsync(bad, h->d_rb_rec_bad, sizeof(u32) * n, cudaMemcpyDeviceToHost, h->stream));
    CUDA_TRY(h, cudaStreamSynchronize(h->stream));
    return 0;
}

// produce side: the publishes host_idx[0..n) of the current plan (one topic-partition, in send order) become ONE
// RecordBatch v2 frame — varint record headers, key = correlation id when keyed, calfkit's two headers, CRC32C — built
// on the device from the payloads where they lie in the output buffer, then copied to host_frame.
extern "C" int ck_encode_recordbatch(ck_handle* h, const uint32_t* host_idx, uint32_t n, int64_t base_offset, int64_t timestamp_ms,
                                     uint8_t* host_frame, uint64_t cap, uint64_t* frame_len) {
    cudaSetDevice(h->device);
    if (!n || n > h->n_pubs) return fail(h, "ck_encode_recordbatch: index list empty or longer than the publish table");
    if (!h->d_rb_idx) {
        CUDA_TRY(h, cudaMalloc((void**)&h->d_rb_idx, sizeof(u32) * (size_t)h->max_pubs));
        CUDA_TRY(h, cudaMalloc((void**)&h->d_rb_sizes, sizeof(u32) * (size_t)h->max_pubs));
        CUDA_TRY(h, cudaMalloc((void**)&h->d_rb_rec_off, sizeof(long long) * ((size_t)h->max_pubs + 1)));
        CUDA_TRY(h, cudaMalloc((void**)&h->d_rb_frame_len, sizeof(long long)));
        h->rb_frame_cap = h->max_out + 256ull * h->max_payloads + 4096;
        CUDA_TRY(h, cudaMalloc((void**)&h->d_rb_frame, h->rb_frame_cap + CK_PAD));
        CUDA_TRY(h, cudaMalloc((void**)&h->d_rb_partial, sizeof(u32) * (h->rb_frame_cap / CK_RB_CRC_CHUNK + 2)));
    }
    CUDA_TRY(h, cudaMemcpyAsync(h->d_rb_idx, host_idx, sizeof(u32) * n, cudaMemcpyHostToDevice, h->stream));
    {
        KTimer t(h, CK_K_EMIT);
        CKL(h) ck_rb_size_kernel<<<(n + 255) / 256, 256, 0, h->stream>>>(h->d_pubs, h->d_rb_idx, n, h->d_pay_len, h->d_cols, h->n, h->d_rb_sizes);
        CUDA_TRY(h, cudaGetLastError());
    }
    if (run_scan(h, h->d_rb_sizes, n, h->d_rb_rec_off, 0)) return 1;
    // the frame's size is known on the device only; bound it on the host to size the launches and the copy
    uint64_t out_total = 0;
    { unsigned long long g = 0; CUDA_TRY(h, cudaMemcpyAsync(&g, h->d_grand, sizeof g, cudaMemcpyDeviceToHost, h->stream)); CUDA_TRY(h, cudaStreamSynchronize(h->stream)); out_total = g; }
    uint64_t total = CK_RB_HEADER + out_total;
    if (total > h->rb_frame_cap) return fail(h, "ck_encode_recordbatch: frame larger than the frame buffer");
    if (total > cap) return fail(h, "ck_encode_recordbatch: host buffer too small");
    {
        KTimer t(h, CK_K_EMIT);
        CKL(h) ck_rb_write_kernel<<<(n + 7) / 8, 256, 0, h->stream>>>(view_of(h), h->d_pubs, h->d_rb_idx, n, h->d_pay_len, h->d_out_off, h->d_out, h->d_cols, h->n,
                                                                h->d_rb_rec_off, h->d_rb_frame);
        CKL(h) ck_rb_header_kernel<<<1, 32, 0, h->stream>>>(h->d_rb_frame, h->d_rb_rec_off, n, base_offset, timestamp_ms, h->d_rb_frame_len);
        u32 nchunks = (u32)((total - CK_RB_CRC_FROM + CK_RB_CRC_CHUNK - 1) / CK_RB_CRC_CHUNK);
        CKL(h) ck_rb_crc_chunks_kernel<<<(nchunks + 7) / 8, 256, 0, h->stream>>>(h->d_rb_frame, h->d_rb_frame_len, h->d_rb_partial);
        CKL(h) ck_rb_crc_fold_kernel<<<1, 32, 0, h->stream>>>(h->d_rb_frame, h->d_rb_frame_len, h->d_rb_partial);
        CUDA_TRY(h, cudaGetLastError());
    }
    CUDA_TRY(h, cudaMemcpyAsync(host_frame, h->d_rb_frame, total, cudaMemcpyDeviceToHost, h->stream));
    CUDA_TRY(h, cudaStreamSynchronize(h->stream));
    if (frame_len) *frame_len = total;
    return 0;
}

// Runs of frames (ck_encode_recordbatches): scratch sized from max_out / max_payloads for every publish a plan can hold
// (up to two per payload).  plain: the records
// sections back to back; slots: one per 64 KB chunk, at its plaintext offset + 64 * chunk
// index (a compressed chunk never exceeds its input by 64 bytes); out: the frames.  The compression pool is a fixed
// number of threads (128 per SM), each with a hash table and DEFLATE scratch of its own.
static int rbs_alloc(ck_handle* h) {
    if (h->d_rbs_idx) return 0;
    size_t mp = (size_t)h->max_pubs + 1;
    h->rbs_plain_cap = 2 * h->max_out + 256ull * h->max_pubs + 4096;
    h->rbs_chunk_cap = h->rbs_plain_cap / CK_RBS_CHUNK + mp;
    h->rbs_out_cap = h->rbs_plain_cap + 128ull * mp + 16ull * h->rbs_chunk_cap;
    int sms = 0;
    CUDA_TRY(h, cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, h->device));
    h->rbs_pool = (u32)sms * 128u;
    size_t big = mp > h->rbs_chunk_cap + 1 ? mp : h->rbs_chunk_cap + 1;
    CUDA_TRY(h, cudaMalloc((void**)&h->d_rbs_idx, sizeof(u32) * mp));
    CUDA_TRY(h, cudaMalloc((void**)&h->d_rbs_goff, sizeof(u32) * mp));
    CUDA_TRY(h, cudaMalloc((void**)&h->d_rbs_base, sizeof(long long) * mp));
    CUDA_TRY(h, cudaMalloc((void**)&h->d_rbs_delta, sizeof(u32) * mp));
    CUDA_TRY(h, cudaMalloc((void**)&h->d_rbs_size, sizeof(u32) * mp));
    CUDA_TRY(h, cudaMalloc((void**)&h->d_rbs_open, sizeof(u32) * mp));
    CUDA_TRY(h, cudaMalloc((void**)&h->d_rbs_fid, sizeof(u32) * mp));
    CUDA_TRY(h, cudaMalloc((void**)&h->d_rbs_ffirst, sizeof(u32) * (mp + 1)));
    CUDA_TRY(h, cudaMalloc((void**)&h->d_rbs_nch, sizeof(u32) * mp));
    CUDA_TRY(h, cudaMalloc((void**)&h->d_rbs_fsize, sizeof(u32) * mp));
    CUDA_TRY(h, cudaMalloc((void**)&h->d_rbs_fgroup, sizeof(u32) * mp));
    CUDA_TRY(h, cudaMalloc((void**)&h->d_rbs_recoff, sizeof(long long) * (mp + 1)));
    CUDA_TRY(h, cudaMalloc((void**)&h->d_rbs_openx, sizeof(long long) * (mp + 1)));
    CUDA_TRY(h, cudaMalloc((void**)&h->d_rbs_foff, sizeof(long long) * (mp + 1)));
    CUDA_TRY(h, cudaMalloc((void**)&h->d_rbs_cbase, sizeof(long long) * (mp + 1)));
    CUDA_TRY(h, cudaMalloc((void**)&h->d_rbs_csz, sizeof(u32) * h->rbs_chunk_cap));
    CUDA_TRY(h, cudaMalloc((void**)&h->d_rbs_ccrc, sizeof(u32) * h->rbs_chunk_cap));
    CUDA_TRY(h, cudaMalloc((void**)&h->d_rbs_coff, sizeof(long long) * (h->rbs_chunk_cap + 1)));
    CUDA_TRY(h, cudaMalloc((void**)&h->d_rbs_tile, sizeof(unsigned long long) * (big / CK_SCAN_TILE + 2)));
    CUDA_TRY(h, cudaMalloc((void**)&h->d_rbs_grand, sizeof(unsigned long long) * 4));
    CUDA_TRY(h, cudaMalloc((void**)&h->d_rbs_plain, h->rbs_plain_cap + CK_PAD));
    CUDA_TRY(h, cudaMalloc((void**)&h->d_rbs_slots, h->rbs_plain_cap + 64ull * h->rbs_chunk_cap + CK_PAD));
    CUDA_TRY(h, cudaMalloc((void**)&h->d_rbs_out, h->rbs_out_cap + CK_PAD));
    CUDA_TRY(h, cudaMalloc((void**)&h->d_rbs_tabs, sizeof(u32) * ((size_t)h->rbs_pool << CK_DFL_TAB_BITS)));
    CUDA_TRY(h, cudaMalloc((void**)&h->d_rbs_dtabs, sizeof(ck_dfl_tables) * (size_t)h->rbs_pool));
    CUDA_TRY(h, cudaMallocHost((void**)&h->h_rbs, sizeof(unsigned long long) * 4));
    return 0;
}

// produce side, every (topic, partition) of a step in one call: groups of publishes -> runs of RecordBatch v2 frames split
// to max_batch_bytes, records sections compressed with gzip or LZ4 on the device.  Two host synchronisations: after the
// split (frame count, plaintext total) and, for compressed frames, after the scan of the compressed sizes.
extern "C" int ck_encode_recordbatches(ck_handle* h, const uint32_t* host_idx, uint32_t n, const uint32_t* host_group_off,
                                       uint32_t n_groups, const int64_t* host_base_offsets, int64_t timestamp_ms, uint32_t codec,
                                       uint32_t max_batch_bytes, uint32_t* n_frames, uint64_t* total_bytes) {
    cudaSetDevice(h->device);
    h->rbs_nf = 0; h->rbs_total = 0;
    if (codec != 0 && codec != CK_RB_GZIP && codec != CK_RB_LZ4) return fail(h, "ck_encode_recordbatches: codec must be 0 (none), 1 (gzip) or 3 (LZ4)");
    if (max_batch_bytes < CK_RB_HEADER + 1) return fail(h, "ck_encode_recordbatches: max_batch_bytes must be at least 62");
    if (n > h->max_pubs) return fail(h, "ck_encode_recordbatches: more indices than max_payloads * 2");
    if (!n_groups || host_group_off[0] != 0 || host_group_off[n_groups] != n) return fail(h, "ck_encode_recordbatches: group offsets must run from 0 to n");
    if (n_groups > h->max_pubs) return fail(h, "ck_encode_recordbatches: more groups than max_payloads * 2");
    for (u32 g = 0; g < n_groups; g++) if (host_group_off[g + 1] < host_group_off[g]) return fail(h, "ck_encode_recordbatches: group offsets must not decrease");
    for (u32 k = 0; k < n; k++) if (host_idx[k] >= h->n_pubs) return fail(h, "ck_encode_recordbatches: index outside the publish table");
    if (rbs_alloc(h)) return 1;
    if (!n) { if (n_frames) *n_frames = 0; if (total_bytes) *total_bytes = 0; return 0; }
    CUDA_TRY(h, cudaMemcpyAsync(h->d_rbs_idx, host_idx, sizeof(u32) * n, cudaMemcpyHostToDevice, h->stream));
    CUDA_TRY(h, cudaMemcpyAsync(h->d_rbs_goff, host_group_off, sizeof(u32) * (n_groups + 1), cudaMemcpyHostToDevice, h->stream));
    if (host_base_offsets) CUDA_TRY(h, cudaMemcpyAsync(h->d_rbs_base, host_base_offsets, sizeof(long long) * n_groups, cudaMemcpyHostToDevice, h->stream));
    unsigned long long* gr = h->d_rbs_grand;                  // 0 plaintext bytes, 1 frames, 2 chunks, 3 output bytes
    {
        KTimer t(h, CK_K_EMIT);
        CKL(h) ck_rbs_split_kernel<<<(n_groups + 7) / 8, 256, 0, h->stream>>>(h->d_pubs, h->d_rbs_idx, h->d_rbs_goff, n_groups, h->d_pay_len,
                                                                            h->d_cols, h->n, max_batch_bytes, h->d_rbs_delta, h->d_rbs_size, h->d_rbs_open);
        CUDA_TRY(h, cudaGetLastError());
    }
    if (run_scan(h, h->d_rbs_size, n, h->d_rbs_recoff, 0, h->d_rbs_tile, gr + 0)) return 1;
    if (run_scan(h, h->d_rbs_open, n, h->d_rbs_openx, 0, h->d_rbs_tile, gr + 1)) return 1;
    CUDA_TRY(h, cudaMemcpyAsync(h->h_rbs, gr, sizeof(unsigned long long) * 2, cudaMemcpyDeviceToHost, h->stream));
    CUDA_TRY(h, cudaStreamSynchronize(h->stream));
    uint64_t plain = h->h_rbs[0]; u32 nf = (u32)h->h_rbs[1];
    uint64_t cmax = plain / CK_RBS_CHUNK + nf;                // each frame adds at most one partial chunk
    char msg[256];
    if (plain > h->rbs_plain_cap || (!codec && plain + (uint64_t)CK_RB_HEADER * nf > h->rbs_out_cap) || cmax > h->rbs_chunk_cap) {
        snprintf(msg, sizeof msg, "ck_encode_recordbatches: %llu bytes of records in %u frames exceed the scratch (%llu bytes of records, %llu bytes of frames)",
                 (unsigned long long)plain, nf, (unsigned long long)h->rbs_plain_cap, (unsigned long long)h->rbs_out_cap);
        return fail(h, msg);
    }
    {
        KTimer t(h, CK_K_EMIT);
        CKL(h) ck_rbs_index_kernel<<<(n + 255) / 256, 256, 0, h->stream>>>(h->d_rbs_open, h->d_rbs_openx, n, nf, h->d_rbs_fid, h->d_rbs_ffirst);
        CKL(h) ck_rb_write_kernel<<<(n + 7) / 8, 256, 0, h->stream>>>(view_of(h), h->d_pubs, h->d_rbs_idx, n, h->d_pay_len, h->d_out_off, h->d_out,
                                                                h->d_cols, h->n, h->d_rbs_recoff, codec ? h->d_rbs_plain : h->d_rbs_out,
                                                                h->d_rbs_delta, h->d_rbs_fid, codec ? 0u : CK_RB_HEADER);
        CKL(h) ck_rbs_layout_kernel<<<(nf + 256) / 256, 256, 0, h->stream>>>(h->d_rbs_ffirst, h->d_rbs_recoff, nf, codec, h->d_rbs_nch, h->d_rbs_foff);
        CUDA_TRY(h, cudaGetLastError());
    }
    uint64_t total = plain + (uint64_t)CK_RB_HEADER * nf;
    if (codec) {
        if (run_scan(h, h->d_rbs_nch, nf, h->d_rbs_cbase, 0, h->d_rbs_tile, gr + 2)) return 1;
        {
            KTimer t(h, CK_K_CODEC);
            CKL(h) ck_rbs_compress_kernel<<<h->rbs_pool / 128, 128, 0, h->stream>>>(h->d_rbs_plain, h->d_rbs_recoff, h->d_rbs_ffirst, h->d_rbs_cbase, nf,
                gr + 2, (u32)cmax, codec, h->d_rbs_slots, h->d_rbs_csz, h->d_rbs_ccrc, h->d_rbs_tabs, h->d_rbs_dtabs);
            CUDA_TRY(h, cudaGetLastError());
        }
        if (run_scan(h, h->d_rbs_csz, (u32)cmax, h->d_rbs_coff, 0, h->d_rbs_tile, gr + 3)) return 1;
        {
            KTimer t(h, CK_K_EMIT);
            CKL(h) ck_rbs_fsize_kernel<<<(nf + 255) / 256, 256, 0, h->stream>>>(h->d_rbs_cbase, h->d_rbs_coff, nf, codec, h->d_rbs_fsize);
            CUDA_TRY(h, cudaGetLastError());
        }
        if (run_scan(h, h->d_rbs_fsize, nf, h->d_rbs_foff, 0, h->d_rbs_tile, gr + 3)) return 1;
        CUDA_TRY(h, cudaMemcpyAsync(h->h_rbs + 3, gr + 3, sizeof(unsigned long long), cudaMemcpyDeviceToHost, h->stream));
        CUDA_TRY(h, cudaStreamSynchronize(h->stream));
        total = h->h_rbs[3];
        if (total > h->rbs_out_cap) {
            snprintf(msg, sizeof msg, "ck_encode_recordbatches: %llu bytes of frames exceed the frame buffer (%llu bytes)",
                     (unsigned long long)total, (unsigned long long)h->rbs_out_cap);
            return fail(h, msg);
        }
    }
    {
        KTimer t(h, CK_K_EMIT);
        if (codec) CKL(h) ck_rbs_copy_kernel<<<(u32)((cmax + 7) / 8), 256, 0, h->stream>>>(h->d_rbs_slots, h->d_rbs_recoff, h->d_rbs_ffirst, h->d_rbs_cbase,
                                                                                        h->d_rbs_coff, nf, gr + 2, codec, h->d_rbs_foff, h->d_rbs_out);
        CKL(h) ck_rbs_header_kernel<<<(nf + 127) / 128, 128, 0, h->stream>>>(h->d_rbs_out, h->d_rbs_foff, h->d_rbs_ffirst, h->d_rbs_recoff, nf, h->d_rbs_goff,
                                                                           n_groups, host_base_offsets ? h->d_rbs_base : nullptr, timestamp_ms, codec,
                                                                           h->d_rbs_cbase, h->d_rbs_ccrc, h->d_rbs_fgroup);
        CKL(h) ck_rbs_crc_kernel<<<(nf + 7) / 8, 256, 0, h->stream>>>(h->d_rbs_out, h->d_rbs_foff, nf);
        CUDA_TRY(h, cudaGetLastError());
    }
    h->rbs_nf = nf; h->rbs_total = total;
    if (n_frames) *n_frames = nf;
    if (total_bytes) *total_bytes = total;
    return 0;
}

// the result of the last ck_encode_recordbatches: host_out[0 .. total_bytes) = the frames back to back,
// host_frame_off[n_frames + 1], host_frame_group[n_frames]
extern "C" int ck_fetch_recordbatches(ck_handle* h, uint8_t* host_out, uint64_t cap, uint64_t* host_frame_off, uint32_t* host_frame_group) {
    cudaSetDevice(h->device);
    if (h->rbs_total > cap) return fail(h, "ck_fetch_recordbatches: host buffer too small");
    if (!h->rbs_nf) { if (host_frame_off) host_frame_off[0] = 0; return 0; }
    CUDA_TRY(h, cudaMemcpyAsync(host_out, h->d_rbs_out, h->rbs_total, cudaMemcpyDeviceToHost, h->stream));
    if (host_frame_off) CUDA_TRY(h, cudaMemcpyAsync(host_frame_off, h->d_rbs_foff, sizeof(long long) * (h->rbs_nf + 1), cudaMemcpyDeviceToHost, h->stream));
    if (host_frame_group) CUDA_TRY(h, cudaMemcpyAsync(host_frame_group, h->d_rbs_fgroup, sizeof(u32) * h->rbs_nf, cudaMemcpyDeviceToHost, h->stream));
    CUDA_TRY(h, cudaStreamSynchronize(h->stream));
    return 0;
}

// ---- aggregation gate (csrc/ck_gate.cuh) ------------------------------------------------------------------------------
extern "C" int ck_gate_create(ck_handle* h, uint32_t max_entries, uint32_t max_slots, uint64_t arena_bytes) {
    cudaSetDevice(h->device);
    if (h->gate_set) return fail(h, "ck_gate_create: already created");
    if (arena_bytes >= (1ull << 32)) return fail(h, "ck_gate_create: arena must be smaller than 4 GiB (32-bit segment offsets)");
    ck_gate g{};
    u32 cap = 64; while (cap < 4 * (uint64_t)max_entries) cap <<= 1;
    g.cap = cap; g.max_entries = max_entries; g.max_slots = max_slots; g.arena_cap = arena_bytes;
    CUDA_TRY(h, cudaMalloc((void**)&g.keys, sizeof(unsigned long long) * cap));
    CUDA_TRY(h, cudaMalloc((void**)&g.vals, sizeof(u32) * cap));
    CUDA_TRY(h, cudaMalloc((void**)&g.entries, sizeof(ck_gate_entry) * (size_t)max_entries));
    CUDA_TRY(h, cudaMalloc((void**)&g.slots, sizeof(ck_gate_slot) * (size_t)max_slots));
    CUDA_TRY(h, cudaMalloc((void**)&g.arena, arena_bytes + CK_PAD));
    CUDA_TRY(h, cudaMalloc((void**)&g.ctr, sizeof(unsigned long long) * 8));
    CUDA_TRY(h, cudaMalloc((void**)&h->d_rec_entry, sizeof(u32) * (size_t)h->max_records));
    CUDA_TRY(h, cudaMemsetAsync(g.keys, 0, sizeof(unsigned long long) * cap, h->stream));
    CUDA_TRY(h, cudaMemsetAsync(g.ctr, 0, sizeof(unsigned long long) * 8, h->stream));
    CUDA_TRY(h, cudaStreamSynchronize(h->stream));
    h->gate = g; h->gate_set = true;
    return 0;
}

extern "C" int ck_gate_reset(ck_handle* h) {
    cudaSetDevice(h->device);
    if (!h->gate_set) return fail(h, "ck_gate_reset: call ck_gate_create first");
    CUDA_TRY(h, cudaMemsetAsync(h->gate.keys, 0, sizeof(unsigned long long) * h->gate.cap, h->stream));
    CUDA_TRY(h, cudaMemsetAsync(h->gate.ctr, 0, sizeof(unsigned long long) * 8, h->stream));
    return 0;
}

extern "C" int ck_gate_stats(ck_handle* h, uint64_t* out5) {
    cudaSetDevice(h->device);
    if (!h->gate_set) return fail(h, "ck_gate_stats: call ck_gate_create first");
    CUDA_TRY(h, cudaMemcpyAsync(out5, h->gate.ctr, sizeof(unsigned long long) * 5, cudaMemcpyDeviceToHost, h->stream));
    CUDA_TRY(h, cudaStreamSynchronize(h->stream));
    return 0;
}

// after ck_fanout_plan on a batch of post-LLM envelopes: every record that went out as list[Call] becomes a pending entry
extern "C" int ck_gate_register(ck_handle* h, uint32_t min_pending) {
    cudaSetDevice(h->device);
    if (!h->gate_set) return fail(h, "ck_gate_register: call ck_gate_create first");
    u32 n = h->n;
    if (!n) return 0;
    KTimer t(h, CK_K_FANOUT);
    CKL(h) ck_gate_register_kernel<<<(n + 127) / 128, 128, 0, h->stream>>>(view_of(h), n, h->d_cols, n, h->gate, min_pending, h->d_rec_entry);
    CKL(h) ck_gate_copy_base_kernel<<<(n + 7) / 8, 256, 0, h->stream>>>(view_of(h), n, h->gate, h->d_rec_entry);
    CUDA_TRY(h, cudaGetLastError());
    return 0;
}

// a batch of records arriving at the agent's topic: probe -> resolve -> merge -> encode.  Per record (column ACTION):
// CK_ACT_SILENT (collected, set still incomplete: only the handler-return publish), CK_ACT_GATE_COMPLETE (payload i = the
// envelope carrying base_state + collected results), CK_ACT_GATE_PASS (no pending fan-out: continue with the inbound state).
extern "C" int ck_gate_arrive(ck_handle* h, uint64_t stamp_base) {
    cudaSetDevice(h->device);
    if (!h->gate_set) return fail(h, "ck_gate_arrive: call ck_gate_create first");
    if (!h->tool_set) return fail(h, "ck_gate_arrive: call ck_set_tool_node (publish topic) first");
    u32 n = h->n;
    {
        KTimer t(h, CK_K_PLAN);
        if (n) {
            CKL(h) ck_gate_probe_kernel<<<(n + 127) / 128, 128, 0, h->stream>>>(view_of(h), n, h->d_cols, n, h->gate, stamp_base, h->d_rec_entry);
            CKL(h) ck_gate_resolve_kernel<<<(n + 127) / 128, 128, 0, h->stream>>>(view_of(h), n, h->d_cols, n, h->gate, stamp_base, h->d_rec_entry,
                h->h_tool_cfg.publish_topic_id, h->d_glue, h->d_descs, h->d_pay_len, h->d_pubs);
            CKL(h) ck_gate_merge_kernel<<<(n + 3) / 4, 128, 0, h->stream>>>(view_of(h), n, h->d_cols, n, h->gate, h->d_rec_entry, h->d_glue, h->d_descs, h->d_pay_len);
        }
        CUDA_TRY(h, cudaGetLastError());
    }
    if (scan_emit(h, n, h->gate.arena)) return 1;
    h->n_pubs = 2 * n;
    return 0;
}

// ---- cross-partition forward over peer memory (csrc/ck_xsend.cuh) --------------------------------------------------------
static int x_alloc(ck_handle* h) {
    if (h->d_x_hist) return 0;
    u32 nb_max = (h->max_pubs + CK_X_BLOCK - 1) / CK_X_BLOCK;
    size_t nh = (size_t)CK_X_MAXWORLD * nb_max;
    CUDA_TRY(h, cudaMalloc((void**)&h->d_x_hist, sizeof(u32) * nh));
    CUDA_TRY(h, cudaMalloc((void**)&h->d_x_base, sizeof(long long) * (nh + 1)));
    CUDA_TRY(h, cudaMalloc((void**)&h->d_x_nbytes, sizeof(unsigned long long) * CK_X_MAXWORLD));
    CUDA_TRY(h, cudaMalloc((void**)&h->d_x_src_off, sizeof(long long) * ((size_t)h->max_pubs + 1)));
    CUDA_TRY(h, cudaMalloc((void**)&h->d_x_len, sizeof(long long) * ((size_t)h->max_pubs + 1)));
    CUDA_TRY(h, cudaMalloc((void**)&h->d_x_dst_off, sizeof(long long) * ((size_t)h->max_pubs + 1)));
    CUDA_TRY(h, cudaMalloc((void**)&h->d_x_len32, sizeof(u32) * ((size_t)h->max_pubs + 1)));
    CUDA_TRY(h, cudaMalloc((void**)&h->d_x_pub, sizeof(u32) * ((size_t)h->max_pubs + 1)));
    size_t nt = (nh > h->max_pubs ? nh : h->max_pubs) / CK_SCAN_TILE + 2;
    CUDA_TRY(h, cudaMalloc((void**)&h->d_x_tile, sizeof(unsigned long long) * nt));
    CUDA_TRY(h, cudaMalloc((void**)&h->d_x_grand, sizeof(unsigned long long)));
    CUDA_TRY(h, cudaMalloc((void**)&h->d_x_grand2, sizeof(unsigned long long)));
    CUDA_TRY(h, cudaMallocHost((void**)&h->h_x, sizeof(long long) * (2 * CK_X_MAXWORLD + 2)));
    return 0;
}

// receive buffer of this rank: `world` regions (one per source rank), each max_fwd meta entries + data_cap payload bytes.
// ipc_handle_out (64 bytes): give it to every peer (any side channel: the Python binding all-gathers it).
extern "C" int ck_comm_create(ck_handle* h, uint32_t rank, uint32_t world, uint32_t max_fwd, uint64_t data_cap, uint8_t* ipc_handle_out) {
    cudaSetDevice(h->device);
    if (world < 1 || world > CK_X_MAXWORLD || rank >= world) return fail(h, "ck_comm_create: world must be 1..16 and rank < world");
    if (h->d_recv) return fail(h, "ck_comm_create: already created");
    static_assert(sizeof(cudaIpcMemHandle_t) == 64, "ipc handle size");
    h->comm_rank = rank; h->comm_world = world; h->max_fwd = max_fwd;
    h->region_data_cap = (data_cap + 15) & ~15ull;
    h->region_stride = (CK_X_HDR + (unsigned long long)max_fwd * sizeof(ck_xmeta) + h->region_data_cap + 255) & ~255ull;
    CUDA_TRY(h, cudaMalloc((void**)&h->d_recv, h->region_stride * world + CK_X_FLAGS_BYTES + CK_PAD));
    CUDA_TRY(h, cudaMemset(h->d_recv, 0, h->region_stride * world + CK_X_FLAGS_BYTES));
    CUDA_TRY(h, cudaMalloc((void**)&h->d_x_overflow, sizeof(u32) * (CK_X_MAXWORLD + 1)));
    CUDA_TRY(h, cudaMemset(h->d_x_overflow, 0, sizeof(u32) * (CK_X_MAXWORLD + 1)));     // [world]: barrier timeout flag
    cudaIpcMemHandle_t ih;
    CUDA_TRY(h, cudaIpcGetMemHandle(&ih, h->d_recv));
    memcpy(ipc_handle_out, &ih, 64);
    // the exchange is a dozen small dependent kernels: on a highest-priority stream their blocks are scheduled as soon as
    // any SM slot frees up instead of queueing behind the other lane's million-record kernels
    int lo = 0, hi = 0;
    CUDA_TRY(h, cudaDeviceGetStreamPriorityRange(&lo, &hi));
    CUDA_TRY(h, cudaStreamCreateWithPriority(&h->xstream, cudaStreamNonBlocking, hi));
    CUDA_TRY(h, cudaEventCreateWithFlags(&h->x_ev0, cudaEventDisableTiming));
    CUDA_TRY(h, cudaEventCreateWithFlags(&h->x_ev1, cudaEventDisableTiming));
    return 0;
}

// handles[world][64]: every rank's ck_comm_create output, in rank order (this rank's own entry is ignored)
extern "C" int ck_comm_connect(ck_handle* h, const uint8_t* handles) {
    cudaSetDevice(h->device);
    if (!h->d_recv) return fail(h, "ck_comm_connect: call ck_comm_create first");
    for (u32 d = 0; d < h->comm_world; d++) {
        if (d == h->comm_rank) { h->peers.recv[d] = h->d_recv; continue; }
        cudaIpcMemHandle_t ih; memcpy(&ih, handles + 64 * (size_t)d, 64);
        void* p = nullptr;
        CUDA_TRY(h, cudaIpcOpenMemHandle(&p, ih, cudaIpcMemLazyEnablePeerAccess));
        h->peer_opened[d] = p; h->peers.recv[d] = (u8*)p;
    }
    h->comm_ready = true;
    return 0;
}

// plan + pack + transfer of the keyed publishes of the current plan whose partition another rank owns: queued on the
// handle's stream, no host synchronisation.  The caller brackets it with two barriers (peers consumed the previous
// contents / every peer's stores have landed).
static int exchange_send_on_stream(ck_handle* h, uint64_t step);
extern "C" int ck_exchange_send(ck_handle* h, uint64_t step) {
    cudaSetDevice(h->device);
    if (!h->comm_ready) return fail(h, "ck_exchange_send: call ck_comm_create / ck_comm_connect first");
    if (x_alloc(h)) return 1;
    // fork: everything below runs on the high-priority side stream, after what is queued on the handle's stream so far
    CUDA_TRY(h, cudaEventRecord(h->x_ev0, h->stream));
    CUDA_TRY(h, cudaStreamWaitEvent(h->xstream, h->x_ev0, 0));
    cudaStream_t main_stream = h->stream;
    h->stream = h->xstream;
    int rc = exchange_send_on_stream(h, step);
    h->stream = main_stream;
    if (rc) return rc;
    CUDA_TRY(h, cudaEventRecord(h->x_ev1, h->xstream));                  // join
    CUDA_TRY(h, cudaStreamWaitEvent(h->stream, h->x_ev1, 0));
    return 0;
}

static int exchange_send_on_stream(ck_handle* h, uint64_t step) {
    u32 rank = h->comm_rank, world = h->comm_world, npubs = h->n_pubs;
    u32 nb = (npubs + CK_X_BLOCK - 1) / CK_X_BLOCK;
    if (!nb) nb = 1;
    h->x_nb = nb;
    u32 nh = world * nb;
    {
        KTimer t(h, CK_K_ROUTE);
        CUDA_TRY(h, cudaMemsetAsync(h->d_x_nbytes, 0, sizeof(unsigned long long) * CK_X_MAXWORLD, h->stream));
        CKL(h) ck_xplan_count_kernel<<<nb, CK_X_BLOCK, 0, h->stream>>>(h->d_pubs, npubs, h->d_pay_len, rank, world, h->d_x_hist, h->d_x_nbytes);
        CUDA_TRY(h, cudaGetLastError());
    }
    if (run_scan(h, h->d_x_hist, nh, h->d_x_base, 0, h->d_x_tile, h->d_x_grand)) return 1;       // d_x_grand = payloads selected
    {
        KTimer t(h, CK_K_ROUTE);
        CUDA_TRY(h, cudaMemsetAsync(h->d_x_len32, 0, sizeof(u32) * ((size_t)npubs + 1), h->stream));
        CKL(h) ck_xplan_scatter_kernel<<<nb, CK_X_BLOCK, 0, h->stream>>>(h->d_pubs, npubs, h->d_pay_len, h->d_out_off, rank, world, h->d_x_base,
                                                                  h->d_x_src_off, h->d_x_len, h->d_x_len32, h->d_x_pub);
        CUDA_TRY(h, cudaGetLastError());
    }
    // byte offsets of the (16-byte padded) payloads in destination order; scanned over all publish slots so that the
    // launch does not need the selected count on the host (unselected tail entries are zero)
    if (run_scan(h, h->d_x_len32, npubs ? npubs : 1, h->d_x_dst_off, 15, h->d_x_tile, h->d_x_grand2)) return 1;
    unsigned long long flags_off = h->region_stride * world;
    {
        KTimer t(h, CK_K_EMIT);
        // barrier 1: every peer has consumed what it received last time (its own stream order puts that before this point)
        CKL(h) ck_xbarrier_kernel<<<1, 32, 0, h->stream>>>(h->peers, rank, world, flags_off, 0, step, h->d_x_overflow + CK_X_MAXWORLD);
        if (npubs) CKL(h) ck_xsend_kernel<<<148 * 4, 256, 0, h->stream>>>(h->d_pubs, h->d_x_pub, h->d_x_src_off, h->d_x_len32, h->d_x_dst_off, h->d_x_base, nb,
            h->d_x_grand, h->d_out, h->peers, rank, world, h->region_stride, h->max_fwd, h->region_data_cap, h->d_x_overflow);
        CKL(h) ck_xhdr_kernel<<<1, 32, 0, h->stream>>>(h->d_x_dst_off, h->d_x_base, nb, h->d_x_grand, h->peers, rank, world, h->region_stride, step, h->d_x_overflow);
        // barrier 2: everybody's stores (to everybody) have landed
        CKL(h) ck_xbarrier_kernel<<<1, 32, 0, h->stream>>>(h->peers, rank, world, flags_off, 1, step, h->d_x_overflow + CK_X_MAXWORLD);
        CUDA_TRY(h, cudaGetLastError());
    }
    return 0;
}

// what this rank received (after the caller's closing barrier): per source rank the header {step, count, overflow, bytes};
// ck_recv_buffer gives the device address and layout for in-place use, ck_fetch_received copies region `src` to the host
extern "C" int ck_recv_info(ck_handle* h, void** dev_recv, uint64_t* region_stride, uint32_t* max_fwd, uint64_t* data_cap) {
    if (!h->d_recv) return fail(h, "ck_recv_info: call ck_comm_create first");
    if (dev_recv) *dev_recv = h->d_recv;
    if (region_stride) *region_stride = h->region_stride;
    if (max_fwd) *max_fwd = h->max_fwd;
    if (data_cap) *data_cap = h->region_data_cap;
    return 0;
}
extern "C" int ck_fetch_received(ck_handle* h, uint32_t src, uint64_t* hdr4 /* step, count, overflow, nbytes */, uint8_t* host_meta, uint8_t* host_data, uint64_t data_cap) {
    cudaSetDevice(h->device);
    if (!h->d_recv || src >= h->comm_world) return fail(h, "ck_fetch_received: no such region");
    const u8* region = h->d_recv + (size_t)src * h->region_stride;
    ck_xregion_hdr hd{};
    CUDA_TRY(h, cudaMemcpyAsync(&hd, region, sizeof hd, cudaMemcpyDeviceToHost, h->stream));
    CUDA_TRY(h, cudaStreamSynchronize(h->stream));
    hdr4[0] = hd.step; hdr4[1] = hd.count; hdr4[2] = hd.overflow; hdr4[3] = hd.nbytes;
    { u32 to = 0; CUDA_TRY(h, cudaMemcpy(&to, h->d_x_overflow + CK_X_MAXWORLD, sizeof to, cudaMemcpyDeviceToHost)); if (to) return fail(h, "exchange barrier timed out: a peer did not arrive"); }
    if (hd.nbytes > data_cap) return fail(h, "ck_fetch_received: host buffer too small");
    if (host_meta && hd.count) CUDA_TRY(h, cudaMemcpyAsync(host_meta, region + CK_X_HDR, sizeof(ck_xmeta) * (size_t)hd.count, cudaMemcpyDeviceToHost, h->stream));
    if (host_data && hd.nbytes) CUDA_TRY(h, cudaMemcpyAsync(host_data, region + CK_X_HDR + (size_t)h->max_fwd * sizeof(ck_xmeta), hd.nbytes, cudaMemcpyDeviceToHost, h->stream));
    CUDA_TRY(h, cudaStreamSynchronize(h->stream));
    return 0;
}

// the pipelined form: ck_peek_received reads every region header with one small copy (one synchronisation of the engine's
// stream, which the caller has normally just done anyway), ck_fetch_received_async queues the copies of one region into
// page-locked memory and returns; they are complete after the next ck_sync
extern "C" int ck_peek_received(ck_handle* h, uint64_t* hdr4 /* [world][4]: step, count, overflow, nbytes */) {
    cudaSetDevice(h->device);
    if (!h->d_recv) return fail(h, "ck_peek_received: call ck_comm_create first");
    ck_xregion_hdr hd[CK_X_MAXWORLD];
    CUDA_TRY(h, cudaMemcpy2DAsync(hd, sizeof(ck_xregion_hdr), h->d_recv, h->region_stride, sizeof(ck_xregion_hdr), h->comm_world,
                                  cudaMemcpyDeviceToHost, h->stream));
    u32 to = 0;
    CUDA_TRY(h, cudaMemcpyAsync(&to, h->d_x_overflow + CK_X_MAXWORLD, sizeof to, cudaMemcpyDeviceToHost, h->stream));
    CUDA_TRY(h, cudaStreamSynchronize(h->stream));
    if (to) return fail(h, "exchange barrier timed out: a peer did not arrive");
    for (u32 r = 0; r < h->comm_world; r++) {
        hdr4[4 * r] = hd[r].step; hdr4[4 * r + 1] = hd[r].count; hdr4[4 * r + 2] = hd[r].overflow; hdr4[4 * r + 3] = hd[r].nbytes;
    }
    return 0;
}
extern "C" int ck_fetch_received_async(ck_handle* h, uint32_t src, uint64_t count, uint64_t nbytes, uint8_t* host_meta, uint8_t* host_data) {
    cudaSetDevice(h->device);
    if (!h->d_recv || src >= h->comm_world) return fail(h, "ck_fetch_received_async: no such region");
    if (count > h->max_fwd || nbytes > h->region_data_cap) return fail(h, "ck_fetch_received_async: count / nbytes beyond the region");
    const u8* region = h->d_recv + (size_t)src * h->region_stride;
    if (host_meta && count) CUDA_TRY(h, cudaMemcpyAsync(host_meta, region + CK_X_HDR, sizeof(ck_xmeta) * (size_t)count, cudaMemcpyDeviceToHost, h->stream));
    if (host_data && nbytes) CUDA_TRY(h, cudaMemcpyAsync(host_data, region + CK_X_HDR + (size_t)h->max_fwd * sizeof(ck_xmeta), nbytes, cudaMemcpyDeviceToHost, h->stream));
    return 0;
}

// multi-GPU exchange planning: see ck_xplan_*_kernel.  One host synchronisation (the all-to-all needs the split
// sizes on the host); the scatter and the offset scan are queued behind it.
extern "C" int ck_exchange_plan(ck_handle* h, uint32_t rank, uint32_t world, const int64_t** dev_src_off, const int64_t** dev_len,
                                const int64_t** dev_dst_off, const uint32_t** dev_pub, int64_t* host_counts, int64_t* host_nbytes,
                                uint32_t* n_sel) {
    cudaSetDevice(h->device);
    if (world < 1 || world > CK_X_MAXWORLD || rank >= world) return fail(h, "ck_exchange_plan: world must be 1..16 and rank < world");
    if (x_alloc(h)) return 1;
    u32 npubs = h->n_pubs;
    u32 nb = (npubs + CK_X_BLOCK - 1) / CK_X_BLOCK;
    for (u32 d = 0; d < world; d++) { host_counts[d] = 0; host_nbytes[d] = 0; }
    *n_sel = 0;
    if (dev_src_off) *dev_src_off = (const int64_t*)h->d_x_src_off;
    if (dev_len) *dev_len = (const int64_t*)h->d_x_len;
    if (dev_dst_off) *dev_dst_off = (const int64_t*)h->d_x_dst_off;
    if (dev_pub) *dev_pub = h->d_x_pub;
    if (!nb) return 0;
    u32 nh = world * nb;
    {
        KTimer t(h, CK_K_ROUTE);
        CUDA_TRY(h, cudaMemsetAsync(h->d_x_nbytes, 0, sizeof(unsigned long long) * CK_X_MAXWORLD, h->stream));
        CKL(h) ck_xplan_count_kernel<<<nb, CK_X_BLOCK, 0, h->stream>>>(h->d_pubs, npubs, h->d_pay_len, rank, world, h->d_x_hist, h->d_x_nbytes);
        CUDA_TRY(h, cudaGetLastError());
    }
    if (run_scan(h, h->d_x_hist, nh, h->d_x_base, 0, h->d_x_tile, h->d_x_grand)) return 1;
    // first slot of every destination (= base[d * nb]), the total, and the bytes per destination
    CUDA_TRY(h, cudaMemcpy2DAsync(h->h_x, sizeof(long long), h->d_x_base, sizeof(long long) * nb, sizeof(long long), world,
                                  cudaMemcpyDeviceToHost, h->stream));
    CUDA_TRY(h, cudaMemcpyAsync(h->h_x + CK_X_MAXWORLD, h->d_x_nbytes, sizeof(long long) * world, cudaMemcpyDeviceToHost, h->stream));
    CUDA_TRY(h, cudaMemcpyAsync(h->h_x + 2 * CK_X_MAXWORLD, h->d_x_grand, sizeof(long long), cudaMemcpyDeviceToHost, h->stream));
    CUDA_TRY(h, cudaStreamSynchronize(h->stream));
    long long total = h->h_x[2 * CK_X_MAXWORLD];
    for (u32 d = 0; d < world; d++) {
        long long next = d + 1 < world ? h->h_x[d + 1] : total;
        host_counts[d] = next - h->h_x[d];
        host_nbytes[d] = h->h_x[CK_X_MAXWORLD + d];
    }
    *n_sel = (u32)total;
    {
        KTimer t(h, CK_K_ROUTE);
        CKL(h) ck_xplan_scatter_kernel<<<nb, CK_X_BLOCK, 0, h->stream>>>(h->d_pubs, npubs, h->d_pay_len, h->d_out_off, rank, world, h->d_x_base,
                                                                  h->d_x_src_off, h->d_x_len, h->d_x_len32, h->d_x_pub);
        CUDA_TRY(h, cudaGetLastError());
    }
    if (total && run_scan(h, h->d_x_len32, (u32)total, h->d_x_dst_off, 0, h->d_x_tile, h->d_x_grand)) return 1;
    return 0;
}

extern "C" int ck_gather_spans(ck_handle* h, const uint8_t* dev_src, const int64_t* dev_src_off, const int64_t* dev_src_len,
                               uint32_t n, uint8_t* dev_dst, const int64_t* dev_dst_off) {
    cudaSetDevice(h->device);
    KTimer t(h, CK_K_EMIT);
    if (n) CKL(h) ck_gather_spans_kernel<<<(n + 7) / 8, 256, 0, h->stream>>>(dev_src, (const long long*)dev_src_off, (const long long*)dev_src_len, n,
                                                                     dev_dst, (const long long*)dev_dst_off);
    CUDA_TRY(h, cudaGetLastError());
    return 0;
}

extern "C" uint64_t ck_launch_count(ck_handle* h) { return h->n_launch; }

extern "C" int ck_sync(ck_handle* h) {
    cudaSetDevice(h->device);
    CUDA_TRY(h, cudaStreamSynchronize(h->stream));
    return 0;
}

extern "C" int ck_out_size(ck_handle* h, uint64_t* out_bytes, uint32_t* n_payloads, uint32_t* n_publishes) {
    cudaSetDevice(h->device);
    *h->h_grand = 0;
    if (h->n_payloads) {
        CUDA_TRY(h, cudaMemcpyAsync(h->h_grand, h->d_grand, sizeof(unsigned long long), cudaMemcpyDeviceToHost, h->stream));
    }
    CUDA_TRY(h, cudaStreamSynchronize(h->stream));
    if (out_bytes) *out_bytes = *h->h_grand;
    if (n_payloads) *n_payloads = h->n_payloads;
    if (n_publishes) *n_publishes = h->n_pubs;
    return 0;
}

extern "C" int ck_fetch_columns(ck_handle* h, uint32_t* host_cols) {
    cudaSetDevice(h->device);
    CUDA_TRY(h, cudaMemcpyAsync(host_cols, h->d_cols, sizeof(u32) * (size_t)CK_NUM_COLS * h->n, cudaMemcpyDeviceToHost, h->stream));
    CUDA_TRY(h, cudaStreamSynchronize(h->stream));
    return 0;
}

// selected column rows only (a worker needs status / action / the key span, not all 55 columns of a million records)
static int fetch_cols_impl(ck_handle* h, const uint32_t* which, uint32_t k, uint32_t* host_rows, bool wait);
extern "C" int ck_fetch_cols(ck_handle* h, const uint32_t* which, uint32_t k, uint32_t* host_rows) { return fetch_cols_impl(h, which, k, host_rows, true); }
extern "C" int ck_fetch_cols_async(ck_handle* h, const uint32_t* which, uint32_t k, uint32_t* host_rows) { return fetch_cols_impl(h, which, k, host_rows, false); }
static int fetch_cols_impl(ck_handle* h, const uint32_t* which, uint32_t k, uint32_t* host_rows, bool wait) {
    cudaSetDevice(h->device);
    for (uint32_t j = 0; j < k; j++) {
        if (which[j] >= CK_NUM_COLS) return fail(h, "ck_fetch_cols: no such column");
        if (h->n) CUDA_TRY(h, cudaMemcpyAsync(host_rows + (size_t)j * h->n, h->d_cols + (size_t)which[j] * h->n, sizeof(u32) * (size_t)h->n,
                                             cudaMemcpyDeviceToHost, h->stream));
    }
    if (wait) CUDA_TRY(h, cudaStreamSynchronize(h->stream));
    return 0;
}

// how many records of the current batch went through the canonicaliser pass, and the overlay bytes it produced (waits)
extern "C" int ck_canon_stats(ck_handle* h, uint32_t* n_listed, uint64_t* overlay_bytes) {
    cudaSetDevice(h->device);
    ck_canon_ctl c{};
    if (h->n) CUDA_TRY(h, cudaMemcpyAsync(&c, h->d_canon_ctl, sizeof c, cudaMemcpyDeviceToHost, h->stream));
    CUDA_TRY(h, cudaStreamSynchronize(h->stream));
    if (n_listed) *n_listed = c.count;
    if (overlay_bytes) *overlay_bytes = c.cursor;
    return 0;
}

// page-locked host memory for the batch arenas (calfkit/engine/lane.py): what cudaMemcpyAsync needs to overlap the
// two PCIe directions with the kernels
extern "C" int ck_host_alloc(uint64_t bytes, void** out) {
    *out = nullptr;
    cudaError_t e = cudaHostAlloc(out, bytes ? bytes : 1, cudaHostAllocPortable);
    if (e != cudaSuccess) { g_create_error = std::string("ck_host_alloc: ") + cudaGetErrorString(e); return 1; }
    return 0;
}
extern "C" void ck_host_free(void* p) { if (p) cudaFreeHost(p); }

static int fetch_output_impl(ck_handle* h, uint8_t* host_out, uint64_t cap, int64_t* host_out_off, uint32_t* host_out_len,
                             ck_publish* host_pubs, bool wait) {
    cudaSetDevice(h->device);
    uint64_t total = 0;
    if (ck_out_size(h, &total, nullptr, nullptr)) return 1;
    if (total > cap) return fail(h, "ck_fetch_output: host buffer too small");
    if (total > h->max_out) return fail(h, "ck_fetch_output: device output buffer overflowed (raise max_out_bytes)");
    if (host_out && total) CUDA_TRY(h, cudaMemcpyAsync(host_out, h->d_out, total, cudaMemcpyDeviceToHost, h->stream));
    if (host_out_off && h->n_payloads) CUDA_TRY(h, cudaMemcpyAsync(host_out_off, h->d_out_off, sizeof(long long) * ((size_t)h->n_payloads + 1), cudaMemcpyDeviceToHost, h->stream));
    if (host_out_len && h->n_payloads) CUDA_TRY(h, cudaMemcpyAsync(host_out_len, h->d_pay_len, sizeof(u32) * (size_t)h->n_payloads, cudaMemcpyDeviceToHost, h->stream));
    if (host_pubs && h->n_pubs) CUDA_TRY(h, cudaMemcpyAsync(host_pubs, h->d_pubs, sizeof(ck_pub) * (size_t)h->n_pubs, cudaMemcpyDeviceToHost, h->stream));
    if (wait) CUDA_TRY(h, cudaStreamSynchronize(h->stream));
    return 0;
}
extern "C" int ck_fetch_output(ck_handle* h, uint8_t* host_out, uint64_t cap, int64_t* host_out_off, uint32_t* host_out_len,
                               ck_publish* host_pubs) {
    return fetch_output_impl(h, host_out, cap, host_out_off, host_out_len, host_pubs, true);
}
// same copies, queued only (the destination must be page-locked for them to be asynchronous): the caller overlaps its
// own work and calls ck_sync before reading
extern "C" int ck_fetch_output_async(ck_handle* h, uint8_t* host_out, uint64_t cap, int64_t* host_out_off, uint32_t* host_out_len,
                                     ck_publish* host_pubs) {
    return fetch_output_impl(h, host_out, cap, host_out_off, host_out_len, host_pubs, false);
}

extern "C" int ck_fetch_overlay(ck_handle* h, uint8_t* host_ovl, uint64_t cap, int64_t* host_off, uint32_t* host_len, uint64_t* used) {
    cudaSetDevice(h->device);
    if (!h->n) { if (used) *used = 0; return 0; }
    long long total = 0;
    CUDA_TRY(h, cudaMemcpyAsync(&total, &h->d_canon_ctl->cursor, sizeof(long long), cudaMemcpyDeviceToHost, h->stream));
    CUDA_TRY(h, cudaMemcpyAsync(host_off, h->d_ovl_off, sizeof(long long) * (size_t)h->n, cudaMemcpyDeviceToHost, h->stream));
    CUDA_TRY(h, cudaMemcpyAsync(host_len, h->d_ovl_len, sizeof(u32) * (size_t)h->n, cudaMemcpyDeviceToHost, h->stream));
    CUDA_TRY(h, cudaStreamSynchronize(h->stream));
    if ((uint64_t)total > h->max_ovl) total = (long long)h->max_ovl;
    if ((uint64_t)total > cap) return fail(h, "ck_fetch_overlay: host buffer too small");
    if (total) CUDA_TRY(h, cudaMemcpyAsync(host_ovl, h->d_ovl, (size_t)total, cudaMemcpyDeviceToHost, h->stream));
    CUDA_TRY(h, cudaStreamSynchronize(h->stream));
    if (used) *used = (uint64_t)total;
    return 0;
}

extern "C" int ck_fetch_topic_hist(ck_handle* h, uint32_t* host_hist, uint32_t n) {
    cudaSetDevice(h->device);
    if (n > h->hist_cap) n = h->hist_cap;
    CUDA_TRY(h, cudaMemcpyAsync(host_hist, h->d_topic_hist, sizeof(u32) * n, cudaMemcpyDeviceToHost, h->stream));
    CUDA_TRY(h, cudaStreamSynchronize(h->stream));
    return 0;
}

extern "C" void* ck_stream(ck_handle* h) { return (void*)h->stream; }

extern "C" int ck_device_buffers2(ck_handle* h, void** pubs, void** pay_len, void** descs) {
    if (pubs) *pubs = h->d_pubs;
    if (pay_len) *pay_len = h->d_pay_len;
    if (descs) *descs = h->d_descs;
    return 0;
}

extern "C" int ck_device_buffers(ck_handle* h, void** in, void** in_off, void** out, void** out_off, void** cols) {
    if (in) *in = h->d_in;
    if (in_off) *in_off = h->d_in_off;
    if (out) *out = h->d_out;
    if (out_off) *out_off = h->d_out_off;
    if (cols) *cols = h->d_cols;
    return 0;
}

extern "C" int ck_profile(ck_handle* h, int enable) { cudaSetDevice(h->device); profile_collect(h); h->profile = enable != 0; return 0; }

extern "C" int ck_profile_read(ck_handle* h, float* ms, uint32_t* launches, int reset) {
    cudaSetDevice(h->device);
    profile_collect(h);
    for (int k = 0; k < CK_NUM_KERNELS; k++) { ms[k] = h->k_ms[k]; launches[k] = h->k_n[k]; if (reset) { h->k_ms[k] = 0; h->k_n[k] = 0; } }
    return 0;
}
