"""Copies records of the reference's captured Lab3 stream into tests/golden/ as the Avro codec's known-answer
fixtures, so the tests need no copy of the reference.  These are DATA records captured from Kafka (base64
Confluent-framed Avro, assets/lab3/data/ride_requests.jsonl), not source code.

    ride_requests_head.jsonl      200 records: lines 1-120, 5001-5040 and 19961-20000
    ride_requests_sample.jsonl.xz every 8th line of the whole capture, plus the lines holding its earliest and latest
                                  request_ts, in capture order (the capture itself is 6.8 MB)

    python tests/golden/make_wire_fixture.py <reference checkout>/assets/lab3/data/ride_requests.jsonl
"""
import base64
import json
import lzma
import os
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))

from qsa_b200.wire import avro, schemas  # noqa: E402

SAMPLE_STRIDE = 8

if __name__ == "__main__":
    if len(sys.argv) != 2:
        raise SystemExit(__doc__)
    with open(sys.argv[1]) as f:
        lines = f.readlines()
    picked = lines[:120] + lines[5000:5040] + lines[19960:20000]
    with open(os.path.join(HERE, "ride_requests_head.jsonl"), "w") as out:
        out.writelines(picked)
    print("wrote", len(picked), "records")
    cs = avro.CompiledSchema(schemas.RIDE_REQUESTS_VALUE)
    ts = [cs.decode(base64.b64decode(json.loads(line)["value"]), 5)["request_ts"] for line in lines]
    keep = set(range(0, len(lines), SAMPLE_STRIDE)) | {ts.index(min(ts)), ts.index(max(ts))}
    sample = [lines[i] for i in sorted(keep)]
    with lzma.open(os.path.join(HERE, "ride_requests_sample.jsonl.xz"), "wt", preset=9 | lzma.PRESET_EXTREME) as out:
        out.writelines(sample)
    print("wrote", len(sample), "of", len(lines), "records")
