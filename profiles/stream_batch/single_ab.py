"""One 256 MiB gzip -6 text file through inflate_stream_device, with the package of the source tree given (a build of the parent
commit or of this change): input and output resident, one warm-up call, then the best of 5 calls (host clock around a call that
ends in a synchronise). The output is checked against the input. Prints one JSON line; single_ab.jsonl holds two such pairs, the
parent and this change alternating in one run on one card.
    python profiles/stream_batch/single_ab.py <tree> <label>"""
import json
import os
import subprocess
import sys
import time

import numpy as np

tree = os.path.abspath(sys.argv[1])
sys.path.insert(0, tree)
import zwz_b200 as z  # noqa: E402
from tools import corpus  # noqa: E402

path = "/tmp/single_ab_256M_gzip6.gz"
size = 256 << 20
raw = corpus.gen_text(size, 596, 1).tobytes()
if not os.path.exists(path):
    c = subprocess.run(["gzip", "-6", "-c"], input=raw, capture_output=True, check=True).stdout
    with open(path + ".tmp", "wb") as f:
        f.write(c)
    os.replace(path + ".tmp", path)
with open(path, "rb") as f:
    comp = f.read()
ctx = z.Context(0)
d = ctx.malloc_device(len(comp))
o = ctx.malloc_device(size + 64)
ctx.h2d(d, np.frombuffer(comp, dtype=np.uint8))
ts = []
for _ in range(6):
    t0 = time.perf_counter()
    r = ctx.inflate_stream_device(d, len(comp), o, size + 64)
    ts.append(time.perf_counter() - t0)
    assert r == (size, z.STREAM_END), r
back = np.empty(size, dtype=np.uint8)
ctx.d2h(back, o)
assert back.tobytes() == raw
print(json.dumps({"tree": sys.argv[2], "comp_bytes": len(comp), "best_s": min(ts[1:]), "gbps": size / min(ts[1:]) / 1e9, "times": ts}))
