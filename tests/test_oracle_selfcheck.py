"""CPU: the oracle's pieces agree with each other and with the product's host code
(run builder / block decoder), and crc64 is pinned to the reference's own crc.cpp."""
import json
import os

import numpy as np

from incubator_pegasus_b200 import synth

CRC64_GOLDEN = os.path.join(os.path.dirname(__file__), "golden", "crc64_reference.json")


def test_crc64_pinned_to_reference_build(oracle, pgs):
    # the answers of the reference's own crc.cpp, stored by tests/golden/make_crc64_golden.py
    with open(CRC64_GOLDEN) as f:
        rows = json.load(f)["rows"]
    assert len(rows) == 22
    L = oracle.lib()
    for r in rows:
        b, init, want = bytes.fromhex(r["data"]), int(r["init"], 16), int(r["crc64"], 16)
        assert L.orc_crc64(b, len(b), init) == want
        assert pgs.lib().pgs_crc64(b, len(b), init) == want
    assert L.orc_crc64(b"hashkey", 7, 0) == 0x1299D9B06672773A  # SURVEY §8c known answers
    assert L.orc_crc64(b"hello, crc64", 12, 0) == 0xAE149F2F8267B7B0


def test_block_codec_cross_check(oracle, pgs):
    runs = synth.compaction_runs(k=2, n_per_run=3000)
    for r in runs:
        br = pgs.build_run(r)                                 # product builder
        assert np.all(br.blk_off % 16 == 0)
        assert pgs.decode_blocks(br).same_as(r)               # product decoder
        assert oracle.Run.from_blocks(br).records().same_as(r)  # oracle decoder
        ob = oracle.BlockRunCPU.from_run(oracle.Run.from_records(r))  # oracle builder
        assert ob.decode().records().same_as(r)


def test_block_level_compaction_equals_semantic(oracle):
    runs = synth.compaction_runs(k=4, n_per_run=5000)
    o = [oracle.Run.from_records(r) for r in runs]
    fp = oracle.filter_params(default_ttl=500)
    for bottommost in (True, False):
        want, st = oracle.compact(o, bottommost, fp, synth.NOW)
        for threads in (1, 3):
            got, st2, _ = oracle.compact_blocks([oracle.BlockRunCPU.from_run(x) for x in o], bottommost, fp, synth.NOW,
                                                threads)
            assert got.decode().records().same_as(want.records())
            assert st2.out_records == st.out_records and st2.dropped_expired == st.dropped_expired
