"""Writes ``launch_trace.json.gz``, the golden launch trace of every case of
tests/test_gpu_launch_trace.py.  Needs a CUDA device:

    python tests/golden/make_launch_trace.py [output path]
"""

import gzip
import json
import os
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path[:0] = [os.path.dirname(os.path.dirname(HERE)), os.path.dirname(HERE)]

import test_gpu_launch_trace as T  # noqa: E402


def main():
    out = sys.argv[1] if len(sys.argv) > 1 else T.GOLDEN
    traces = {name: T.trace(name) for name in sorted(T.CASES)}
    text = "{\n" + ",\n".join(f"{json.dumps(k)}: {json.dumps(v, separators=(',', ':'))}"
                               for k, v in traces.items()) + "\n}\n"
    with open(out, "wb") as f:
        f.write(gzip.compress(text.encode(), 9, mtime=0))
    print(f"{len(traces)} cases -> {out} ({os.path.getsize(out)} bytes)")


if __name__ == "__main__":
    main()
