/* calfkit_b200.h — C-ABI of libcalfkit_b200.so (sm_100a).
 *
 * The reference (calf-ai/calfkit-sdk v0.2.5) has no FFI for this path: its per-record hot loop is
 *   FastStream decoder -> Envelope validation      calfkit/nodes/base.py:151, calfkit/models/envelope.py:9-17
 *   BaseNodeDef.handler / prepare_context           calfkit/nodes/base.py:64-68,149-164
 *   ToolNodeDef.run                                  calfkit/nodes/tool.py:37-86
 *   BaseNodeDef._publish_action -> broker.publish    calfkit/nodes/base.py:70-147
 *   handler return -> publisher(publish_topic)       calfkit/worker/worker.py:52-53
 * The entry points below are what a ctypes binding underneath calfkit.worker.Worker would bind to
 * replace that loop batch-wise (binding shown in INTEGRATION.md).  Plain C: int status (0 = ok),
 * caller-owned buffers, no exceptions, no torch types.  A bad record never fails a batch: per-record
 * status codes live in the column table (ck_common.h).
 *
 * Threading: one handle = one CUDA stream; calls on one handle must be serialised by the caller,
 * different handles are independent (use two for double buffering).  Calls that launch work return
 * once it is enqueued; ck_sync / ck_fetch_* wait for it.
 */
#ifndef CALFKIT_B200_H
#define CALFKIT_B200_H

#include <stdint.h>
#include "../calfkit-sdk_b200/csrc/ck_common.h"

#ifdef __cplusplus
extern "C" {
#endif

typedef struct ck_handle ck_handle;

typedef struct {           /* one publish; mirrors struct ck_pub in csrc/ck_kernels.cuh */
    uint32_t payload;      /* index into the payload offsets, 0xffffffff = slot unused */
    int32_t  topic_id;     /* registered topic id, or -1: read the name at (record, topic_off, topic_len) */
    uint32_t topic_off, topic_len;
    uint32_t record;       /* input record this publish derives from */
    uint32_t has_key;      /* 1: key = correlation id bytes (nodes/base.py:86,103,117,134) */
    int32_t  partition;    /* murmur2(key) % num_partitions, -1 when unkeyed */
    uint32_t pad;          /* FNV-1a of the topic name (set when the name was looked up): groups unregistered topics */
} ck_publish;

/* lifecycle ------------------------------------------------------------------------------------ */
int  ck_create(int device, uint64_t max_in_bytes, uint64_t max_out_bytes, uint32_t max_records,
               uint32_t max_payloads /* >= max_records; fan-out needs records * (fanout + 1) */,
               uint64_t max_aux_bytes, ck_handle** out);
void ck_destroy(ck_handle* h);
const char* ck_last_error(ck_handle* h);          /* h may be NULL: error of the last failed ck_create */
int  ck_version(void);

/* routing table: replaces the implicit "one FastStream subscriber per node.subscribe_topics"
 * binding of Worker.register_handlers (calfkit/worker/worker.py:33-55).  names = concatenated UTF-8
 * topic strings, offsets[n+1]; ids = caller-chosen non-negative ids. Re-registering replaces. */
int  ck_register_topics(ck_handle* h, const uint8_t* names, const uint32_t* offsets, uint32_t n,
                        const int32_t* ids, uint32_t num_partitions);

/* configure the handle for one @agent_tool node (calfkit/nodes/tool.py:24-35,89-95).
 * publish_topic_id: registered id of node.publish_topic or -1.
 * Result template (optional, nparts > 0): the tool's return value is the JSON string made of
 * literal pieces (kind 0, already JSON-escaped) and raw string arguments (kind 1, blob = key name);
 * nparts == 0: results are supplied by the host through ck_tool_plan(aux). */
int  ck_set_tool_node(ck_handle* h, int32_t publish_topic_id, uint32_t nparts, const uint32_t* kinds,
                      const uint8_t* blob, const uint32_t* part_offsets);

/* decode: copy a batch of records (concatenated bytes + n+1 offsets, pinned or pageable host
 * memory) to HBM and run validate+extract: records in the canonical spelling (what the reference's
 * model_dump_json() emits) are recognised in place; any other valid spelling is re-emitted canonically
 * on the device first (ck_fetch_overlay returns those bytes); invalid ones get a per-record status.
 * ck_submit_device: the batch is already resident (device pointers stay owned by the caller and must
 * outlive the following plan/emit calls; at least 64 readable bytes must follow the last record:
 * the kernels read whole aligned vectors). */
int  ck_submit(ck_handle* h, const uint8_t* host_in, const int64_t* host_off, uint32_t n);
int  ck_submit_device(ck_handle* h, const uint8_t* dev_in, const int64_t* dev_off, uint32_t n);

/* engine options.  option 1 (bucket): value != 0 -> every submitted batch is bucketed by record length (stable radix sort of
 * the record indices on the device) before the thread-per-record walk, so that the lanes of a warp walk records of one size
 * class; for topics with mixed sizes / shapes (reference analogue: none — the reference handles one record at a time) */
int  ck_set_option(ck_handle* h, uint32_t option, uint64_t value);

/* group the publish table of the current plan by destination topic on the device (stable two-pass radix sort over 12-bit
 * keys: 0 = topic without a registered id, 1 + id = registered topic, 4095 = unused slot) — the per-topic split a producer
 * needs (reference: one broker.publish per topic, nodes/base.py:82-87) without any host-side scan of the table.
 * ck_fetch_groups: order[n_publishes] = publish indices grouped by key (send order kept inside a group) and
 * key_counts[4096]; wait = 0 queues the copies only (page-locked destinations, ck_sync before reading). */
int  ck_group_publishes(ck_handle* h);
int  ck_fetch_groups(ck_handle* h, uint32_t* host_order, uint32_t* host_key_counts, int wait);

/* Kafka RecordBatch v2 framing on the device (reference: aiokafka under broker.subscriber / broker.publish,
 * calfkit/worker/worker.py:45-53, calfkit/nodes/base.py:82-87).  ck_submit_recordbatch takes a fetch response's record set
 * (concatenated v2 frames) as it came off the socket: one H2D copy, then CRC32C verification, record split and zig-zag
 * varint field decode on the device; the walker reads each value where it lies.  Frames compressed with gzip (codec 1) or
 * LZ4 (codec 3) are decompressed on the device into 16-byte aligned slots of the input buffer right after the submitted
 * bytes (one extra host synchronisation, paid only by fetches that hold such frames; submitted + decompressed bytes must fit
 * max_in_bytes).  Records of a frame that fails the CRC / framing / decompression check, or whose codec is not decoded on
 * the device (snappy, zstd), get status 6 (bad frame); a truncated trailing frame is ignored.  *n_records = records decoded.
 * ck_fetch_rb_index: per record, where value / key / the `correlation_id` header lie (-1 = absent), as offsets into the
 * submitted buffer followed by the decompressed sections; bad = 0, 1 (CRC / framing / decompression) or 2 (codec).
 * ck_fetch_rb_decompressed: host_dst[0 .. *len) = the decompressed sections, which start at offset *base of that space.
 * ck_encode_recordbatch: the publishes host_idx[0..n) of the current plan (one topic-partition, in send order) -> one
 * uncompressed v2 frame (offsetDelta = position in the list, key = correlation id when keyed, headers content-type and
 * correlation_id, CRC32C), built on the device and copied to host_frame. */
int  ck_submit_recordbatch(ck_handle* h, const uint8_t* host_buf, uint64_t nbytes, uint32_t* n_records);
int  ck_fetch_rb_index(ck_handle* h, int64_t* val_off, uint32_t* val_len, int64_t* key_off, int32_t* key_len,
                       int64_t* corr_off, int32_t* corr_len, uint32_t* bad);
int  ck_fetch_rb_decompressed(ck_handle* h, uint8_t* host_dst, uint64_t cap, uint64_t* base, uint64_t* len);
int  ck_encode_recordbatch(ck_handle* h, const uint32_t* host_idx, uint32_t n, int64_t base_offset, int64_t timestamp_ms,
                           uint8_t* host_frame, uint64_t cap, uint64_t* frame_len);
/* ck_encode_recordbatches: publishes host_idx[0..n) of the current plan (indices of live publishes), in groups: group g =
 * host_idx[group_off[g] .. group_off[g+1]), one topic-partition each, in send order.  Every group becomes a run of v2
 * frames, as a producer that closes a batch at max_batch_bytes writes them: a frame takes the group's next records while
 * 61 + (their encoded sizes) <= max_batch_bytes, and always at least one; frames never span groups; offsetDelta is the
 * position inside the frame.  codec: 0 none, 1 gzip, 3 LZ4 (anything else is an error); base_offsets: NULL = 0 for every
 * group; frame k of group g gets baseOffset = base_offsets[g] + (records of g in earlier frames).  Compressed sections are
 * made on the device in 64 KB chunks:
 *   LZ4   one LZ4 frame, descriptor 60 40 82 (independent 64 KB blocks, no checksums, no content size); a chunk that does
 *         not get smaller is stored raw.  Section <= 11 + P + 4 * ceil(P / 65536) bytes for P bytes of records.
 *   gzip  one member, header 1f 8b 08 00 00000000 00 ff; every chunk one non-final dynamic-Huffman block + an empty stored
 *         block (or stored blocks when smaller), matches up to 32 KB back into the previous chunk; final block 03 00,
 *         CRC-32, ISIZE.  Section <= 20 + P + 10 * ceil(P / 65536) bytes.
 * The output depends on the arguments only.  *n_frames / *total_bytes describe the result, which stays on the device
 * until ck_fetch_recordbatches; a request larger than the scratch (sized from max_out_bytes / max_payloads) fails.
 * ck_fetch_recordbatches: host_out[0 .. total_bytes) = the frames back to back, frame_off[n_frames + 1],
 * frame_group[n_frames]. */
int  ck_encode_recordbatches(ck_handle* h, const uint32_t* host_idx, uint32_t n, const uint32_t* host_group_off,
                             uint32_t n_groups, const int64_t* host_base_offsets, int64_t timestamp_ms, uint32_t codec,
                             uint32_t max_batch_bytes, uint32_t* n_frames, uint64_t* total_bytes);
int  ck_fetch_recordbatches(ck_handle* h, uint8_t* host_out, uint64_t cap, uint64_t* host_frame_off, uint32_t* host_frame_group);

/* tool node, host tools only: gather every record's tool-call `args` JSON into the output buffer
 * (payload i = args of record i, empty when the record does not reach the tool). */
int  ck_tool_args(ck_handle* h);
/* tool node: run + publish plan + encode + route.  host_aux/host_aux_off: JSON return values per
 * record (offsets[n+1]) for host tools, NULL for a device template. */
int  ck_tool_plan(ck_handle* h, const uint8_t* host_aux, const int64_t* host_aux_off);
/* ReturnCall of the state as it is on the wire (e.g. an Agent's final output after the host LLM step):
 * pop the current frame, publish to its callback topic and to the node's publish_topic. */
int  ck_return_plan(ck_handle* h);
/* client reply path (calfkit/client/deserialize.py:55-89): payload i = the output value of reply envelope i as JSON —
 * mode 0: first DataPart.data of final_output_parts, else first TextPart.text (auto); 1: TextPart.text only
 * (output_type=str); 2: DataPart.data only (typed output; the caller validates the value).  A reply without the
 * wanted part (the reference raises DeserializationError) gets CK_ACT_RAISES and an empty payload.  No publishes. */
int  ck_reply_plan(ck_handle* h, uint32_t mode);
/* same as ck_tool_plan, aux blob already in HBM */
int  ck_tool_plan_device(ck_handle* h, const uint8_t* dev_aux, const int64_t* dev_aux_off);

/* agent fan-out (calfkit/nodes/agent.py:177-211 + nodes/base.py:73-88): one Call envelope per
 * pending tool call of every record.  tool_names/topic strings: registry tool_name -> subscribe
 * topic[0]; agent_name/callback: the agent's name and subscribe_topics[0]; frame ids are uuid7s
 * built from (unix_ms, seed, output index). */
int  ck_set_agent_node(ck_handle* h, int32_t publish_topic_id, const uint8_t* agent_name, uint32_t agent_name_len,
                       const uint8_t* callback_topic, uint32_t callback_len,
                       const uint8_t* tool_names, const uint32_t* tool_name_off,
                       const uint8_t* tool_topics, const uint32_t* tool_topic_off, uint32_t ntools);
int  ck_set_agent_tool_topic_ids(ck_handle* h, int32_t self_topic_id /* id of the agent's subscribe_topics[0], -1 = unregistered */,
                                 const uint32_t* ids /* 0xffffffff = unregistered */, uint32_t ntools);
/* sequential != 0: Agent(sequential_only_mode=True) — only the first pending call goes out, as a single
 * Call (agent.py:94-108,179-192). */
int  ck_fanout_plan(ck_handle* h, uint64_t unix_ms, uint64_t seed, uint32_t max_fanout, uint32_t sequential);
/* TailCall to the agent's own topic (all requested tools invalid -> retry, agent.py:171-175;
 * nodes/base.py:120-136): the current frame is replaced by a fresh one inheriting its callback_topic. */
int  ck_tailcall_plan(ck_handle* h, uint64_t unix_ms, uint64_t seed);
/* aggregation gate on the device (calfkit/nodes/agent.py:57-68 _parallel_state_aggregation, models/state.py:127-141
 * PendingToolBatch): an HBM-resident table keyed by correlation id holding, per pending fan-out, the state the agent fanned
 * out from and the expected tool_call_ids with the results collected so far.
 *   ck_gate_create    sizes the table (entries = concurrent fan-outs, slots = sum of their expected ids, arena < 4 GiB)
 *   ck_gate_register  after ck_fanout_plan on a batch of post-LLM envelopes: every record that went out as list[Call]
 *                     (ACTION == CK_ACT_FANOUT) becomes a pending entry (a new one replaces an old one for the same id)
 *   ck_gate_arrive    on a submitted batch of records arriving at the agent's topic; stamp_base = records this node
 *                     consumed before this batch (arrival order across and inside batches).  Column ACTION afterwards:
 *                     CK_ACT_SILENT (collected, still incomplete; only the handler-return publish to publish_topic),
 *                     9 = complete (payload i = inbound envelope carrying base_state + the collected results in order
 *                     of collection; the entry is deleted), 10 = no pending fan-out (continue with the inbound state)
 *   ck_gate_stats     out5 = {entries used, slots used, arena bytes used, live entries, capacity failures}
 *   ck_gate_reset     forget everything (e.g. when live == 0 and the arena is mostly used) */
int  ck_gate_create(ck_handle* h, uint32_t max_entries, uint32_t max_slots, uint64_t arena_bytes);
int  ck_gate_register(ck_handle* h, uint32_t min_pending /* 2 = the reference's rule; 1 also registers single Calls */);
int  ck_gate_arrive(ck_handle* h, uint64_t stamp_base);
int  ck_gate_stats(ck_handle* h, uint64_t* out5);
int  ck_gate_reset(ck_handle* h);
/* cross-partition forward over NVLink peer memory (records shard by Kafka partition across the GPUs of a box; reference
 * analogue: producing to a topic-partition another worker process consumes, nodes/base.py:82-87 key=correlation_id).
 *   ck_comm_create    this rank's receive buffer: one region per source rank (max_fwd payloads, data_cap bytes each);
 *                     ipc_handle_out[64] is handed to every peer (any side channel); max_fwd and data_cap MUST be the same
 *                     on every rank (a rank addresses its region inside a peer's buffer with its own geometry)
 *   ck_comm_connect   handles[world][64] in rank order: maps the peers' receive buffers (CUDA IPC, same box)
 *   ck_exchange_send  plan + pack + transfer in one pass on the handle's stream, no host synchronisation: the keyed
 *                     publishes of the current plan whose partition % world != rank are written straight into the owner's
 *                     region for this rank (payload bytes 16-byte aligned + {len, topic_id, partition, source publish}),
 *                     then the region header {step, count, overflow, bytes}.  The caller brackets it with two barriers:
 *                     before (every peer has consumed what it received last time) and after (all stores have landed).
 *   ck_recv_info / ck_fetch_received: where the regions are / one region copied to the host */
int  ck_comm_create(ck_handle* h, uint32_t rank, uint32_t world, uint32_t max_fwd, uint64_t data_cap, uint8_t* ipc_handle_out);
int  ck_comm_connect(ck_handle* h, const uint8_t* handles);
int  ck_exchange_send(ck_handle* h, uint64_t step);
int  ck_recv_info(ck_handle* h, void** dev_recv, uint64_t* region_stride, uint32_t* max_fwd, uint64_t* data_cap);
int  ck_fetch_received(ck_handle* h, uint32_t src, uint64_t* hdr4, uint8_t* host_meta, uint8_t* host_data, uint64_t data_cap);
/* pipelined form: ck_peek_received reads all region headers ([world][4] = step, count, overflow, nbytes) with one stream
 * synchronisation; ck_fetch_received_async queues the copies of region `src` into page-locked memory and returns (complete
 * after the next ck_sync).  A region stays valid until this engine's next ck_exchange_send. */
int  ck_peek_received(ck_handle* h, uint64_t* hdr4);
int  ck_fetch_received_async(ck_handle* h, uint32_t src, uint64_t count, uint64_t nbytes, uint8_t* host_meta, uint8_t* host_data);
/* multi-GPU exchange planning (records shard by Kafka partition across the GPUs of a box; reference analogue:
 * producing to a topic-partition another worker process consumes, nodes/base.py:82-87 key=correlation_id).  Selects the
 * keyed publishes whose partition % world != rank, ordered by destination rank (stable), into library-owned device
 * arrays: payload span in the output buffer (src_off, len), offset in the packed send buffer (dst_off, exclusive
 * scan of len) and the index of the publish (pub).  host_counts / host_nbytes [world]: payloads and bytes per
 * destination (the all-to-all split sizes).  Waits for the stream once. */
int  ck_exchange_plan(ck_handle* h, uint32_t rank, uint32_t world, const int64_t** dev_src_off, const int64_t** dev_len,
                      const int64_t** dev_dst_off, const uint32_t** dev_pub, int64_t* host_counts, int64_t* host_nbytes,
                      uint32_t* n_sel);
/* copy n spans src[src_off[i] .. +src_len[i]) -> dst[dst_off[i] ..) on the handle's stream (device pointers);
 * used to pack cross-partition payloads before the NCCL all-to-all */
int  ck_gather_spans(ck_handle* h, const uint8_t* dev_src, const int64_t* dev_src_off, const int64_t* dev_src_len,
                     uint32_t n, uint8_t* dev_dst, const int64_t* dev_dst_off);

/* results ---------------------------------------------------------------------------------------- */
int  ck_sync(ck_handle* h);
uint64_t ck_launch_count(ck_handle* h);   /* kernels launched by this handle so far */
int  ck_out_size(ck_handle* h, uint64_t* out_bytes, uint32_t* n_payloads, uint32_t* n_publishes);  /* waits */
int  ck_fetch_columns(ck_handle* h, uint32_t* host_cols /* CK_NUM_COLS * n, column-major */);
/* records of the current batch that were not in the canonical spelling (re-emitted into the overlay, or rejected), and the
 * overlay bytes in use; 0 / 0 means every column span refers to the submitted bytes */
int  ck_canon_stats(ck_handle* h, uint32_t* n_listed, uint64_t* overlay_bytes);
/* k selected rows of the column table: host_rows[j * n + i] = column which[j] of record i */
int  ck_fetch_cols(ck_handle* h, const uint32_t* which, uint32_t k, uint32_t* host_rows);
/* page-locked host memory for batch arenas: the landing zone of polled record batches (reference seam: the consume loop
 * FastStream runs under calfkit/worker/worker.py:45-51) and of the produced payloads; copies to and from it overlap with
 * the kernels and with each other.  ck_last_error(NULL) after a failure. */
int  ck_host_alloc(uint64_t bytes, void** out);
void ck_host_free(void* p);
/* payload i = host_out[host_out_off[i] .. + host_out_len[i]); starts are 16-byte aligned, so
 * host_out_off[i+1] - host_out_off[i] is the length rounded up to 16 and *out_bytes of ck_out_size is
 * the padded total */
int  ck_fetch_output(ck_handle* h, uint8_t* host_out, uint64_t cap, int64_t* host_out_off /* n_payloads+1 */,
                     uint32_t* host_out_len /* n_payloads */, ck_publish* host_pubs /* n_publishes */);
/* the same copies queued only (page-locked destinations): overlap host work, then ck_sync before reading */
int  ck_fetch_output_async(ck_handle* h, uint8_t* host_out, uint64_t cap, int64_t* host_out_off, uint32_t* host_out_len,
                           ck_publish* host_pubs);
int  ck_fetch_cols_async(ck_handle* h, const uint32_t* which, uint32_t k, uint32_t* host_rows);
/* canonical re-emissions of the records that were submitted in a non-canonical spelling: record i has one iff
 * host_off[i] >= 0 (then host_ovl[host_off[i] .. + host_len[i]) are its canonical bytes; column spans of that
 * record refer to them) */
int  ck_fetch_overlay(ck_handle* h, uint8_t* host_ovl, uint64_t cap, int64_t* host_off, uint32_t* host_len, uint64_t* used);
int  ck_fetch_topic_hist(ck_handle* h, uint32_t* host_hist, uint32_t n);

/* introspection for benchmarks / tests ------------------------------------------------------------ */
void* ck_stream(ck_handle* h);                     /* cudaStream_t of the handle */
int  ck_device_buffers(ck_handle* h, void** in, void** in_off, void** out, void** out_off, void** cols);
int  ck_device_buffers2(ck_handle* h, void** pubs, void** pay_len, void** descs);
int  ck_profile(ck_handle* h, int enable);         /* record (asynchronous) CUDA events around every kernel */
int  ck_profile_read(ck_handle* h, float* ms /* CK_NUM_KERNELS */, uint32_t* launches /* CK_NUM_KERNELS */, int reset);

enum { CK_K_WALK = 0, CK_K_PLAN, CK_K_SCAN, CK_K_EMIT, CK_K_ROUTE, CK_K_FANOUT, CK_K_CANON, CK_K_WALK_LONG, CK_K_WALK_ELEMS, CK_K_CODEC, CK_NUM_KERNELS };

#ifdef __cplusplus
}
#endif
#endif
