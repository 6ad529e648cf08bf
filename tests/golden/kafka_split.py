"""TEST INFRASTRUCTURE ONLY — CPU restatement of how a Kafka producer splits one topic-partition's records into batches
(aiokafka closes a batch at max_batch_size bytes), on top of the framing restatement in oracle/kafka_batch.py.  The device
counterpart is ck_encode_recordbatches (csrc/ck_kafka.cuh, ck_rbs_split_kernel)."""
from __future__ import annotations

from oracle import kafka_batch as kb


def split_batches(records: list[kb.KRecord], max_batch_size: int) -> list[list[kb.KRecord]]:
    """a producer's batches of one topic-partition: a frame takes the next records while its kb.encode_batch length (61 +
    the records, each encoded with its offsetDelta inside the frame) stays <= max_batch_size, and always at least one"""
    out: list[list[kb.KRecord]] = []
    cur: list[kb.KRecord] = []
    size = kb.HEADER_LEN
    for r in records:
        n = len(kb.encode_record(r, len(cur), 0))
        if cur and size + n > max_batch_size:
            out.append(cur)
            cur, size = [], kb.HEADER_LEN
            n = len(kb.encode_record(r, 0, 0))
        cur.append(r)
        size += n
    if cur:
        out.append(cur)
    return out
