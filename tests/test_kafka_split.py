"""The producer's batch split restated in tests/golden/kafka_split.py (split_batches): every frame kb.encode_batch writes
for a chunk stays within the limit unless it holds a single record, no frame could have taken its successor's first
record, and the chunks are the records in order."""
import os
import random
import sys

import pytest

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden"))


@pytest.mark.parametrize("limit", [62, 200, 1000, 16384, 1 << 20])
def test_split_batches_is_greedy_with_exact_sizes(limit):
    import kafka_split as ks
    from oracle import kafka_batch as kb
    rng = random.Random(limit)
    recs = [kb.calfkit_record(bytes(rng.randrange(32, 127) for _ in range(rng.choice([0, 5, 60, 300, 3000, 20000]))),
                              f"{i:032x}", keyed=i % 3 != 0) for i in range(700)]
    chunks = ks.split_batches(recs, limit)
    assert [r for c in chunks for r in c] == recs and all(chunks)
    for i, c in enumerate(chunks):
        n = len(kb.encode_batch(c))
        assert n <= limit or len(c) == 1
        if i + 1 < len(chunks):
            assert len(kb.encode_batch(c + chunks[i + 1][:1])) > limit      # maximal: the next record would not fit
    assert ks.split_batches([], limit) == []
