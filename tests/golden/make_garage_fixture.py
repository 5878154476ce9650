"""Convert the reference's GICP test clouds (multithreaded_gicp/test/*_82_garage.pcd,
binary PCD, fields x y z intensity float32) into tests/golden/garage.npz.

    python tests/golden/make_garage_fixture.py <LOCUS checkout>

Needs a checkout of the original LOCUS project; the .npz is committed so that the
tests do not.
"""
import os
import sys

import numpy as np


def read_pcd(path):
    b = open(path, "rb").read()
    marker = b"DATA binary\n"
    i = b.index(marker) + len(marker)
    hdr = b[:i].decode()
    n = int([l for l in hdr.splitlines() if l.startswith("POINTS")][0].split()[1])
    assert "FIELDS x y z intensity" in hdr and "SIZE 4 4 4 4" in hdr
    return np.frombuffer(b[i:i + n * 16], dtype=np.float32).reshape(n, 4).copy()


if __name__ == "__main__":
    if len(sys.argv) != 2:
        sys.exit(__doc__)
    ref = os.path.join(sys.argv[1], "multithreaded_gicp", "test")
    q = read_pcd(os.path.join(ref, "query_82_garage.pcd"))
    r = read_pcd(os.path.join(ref, "reference_82_garage.pcd"))
    assert q.shape == (811, 4) and r.shape == (8112, 4)
    out = os.path.join(os.path.dirname(os.path.abspath(__file__)), "garage.npz")
    np.savez_compressed(out, query=q, reference=r)
    print("wrote", out, q.shape, r.shape)
