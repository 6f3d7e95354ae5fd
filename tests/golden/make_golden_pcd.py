"""Generates tests/golden/demo_000000_head.pcd: the first 4096 points of MULLS's demo_data/pcd/000000.pcd, byte for byte,
under the original header with WIDTH and POINTS set to 4096 (the whole scan is 124 668 points, 4 MB).

    python tests/golden/make_golden_pcd.py <MULLS checkout>/demo_data/pcd/000000.pcd

Prints the SHA-256 of the (4096, 12) float32 rows mulls_b200.io.read_pcd makes of the ORIGINAL file's first 4096 points:
tests/test_io.py pins the fixture's reading to it.
"""
import hashlib
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
from mulls_b200 import io  # noqa: E402

N = 4096
OUT = os.path.join(os.path.dirname(os.path.abspath(__file__)), "demo_000000_head.pcd")


def main(src):
    with open(src, "rb") as f:
        header = []
        while True:
            line = f.readline()
            key = line.split(b" ", 1)[0].upper()
            if key in (b"WIDTH", b"POINTS"):
                line = key + b" %d\n" % N
            header.append(line)
            if key == b"DATA":
                break
        assert header[-1].split()[1] == b"binary", header[-1]
        nf = len(next(h for h in header if h.startswith(b"FIELDS")).split()) - 1
        body = f.read(N * 4 * nf)
    with open(OUT, "wb") as f:
        f.write(b"".join(header) + body)
    rows = io.read_pcd(src)[:N]
    print(OUT, os.path.getsize(OUT), "bytes; sha256 of the original's first rows:",
          hashlib.sha256(rows.tobytes()).hexdigest())


if __name__ == "__main__":
    main(sys.argv[1])
