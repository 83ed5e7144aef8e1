"""Shrink a Keras ``WHENet.h5`` into the committed reader fixture under tests/golden/.

The original file is 18 MB, almost all of it raw float32 tensor data.  This writes

* ``whenet_h5_skeleton.h5.gz`` - the same file byte for byte (superblock, object headers, B-trees,
  heaps, attributes, data addresses) except that every dataset keeps only its first and last
  ``KEEP`` values and the rest of its data is zeroed; gzip makes the zeros vanish.
* ``whenet_h5_digests.json``   - the SHA-256 of every tensor's full little-endian float32 bytes as
  read from the original file, so the converted ``.npz`` can still be checked bit for bit.

    python tools/make_h5_fixture.py path/to/WHENet.h5
"""
import gzip
import hashlib
import json
import os
import struct
import sys

import numpy as np

ROOT = os.path.join(os.path.dirname(os.path.abspath(__file__)), "..")
sys.path.insert(0, os.path.join(ROOT, "headposeestimation-whenet_b200"))
import h5lite  # noqa: E402

GOLD = os.path.join(ROOT, "tests", "golden")
KEEP = 64


def main(src):
    names, weights, meta = h5lite.read_keras_weights(src)
    f = h5lite.H5File(src)
    buf = bytearray(f.buf)
    found = {}
    for lname in names:
        gaddr = dict(f.children(f.root_addr))[lname]
        found.update(f.visit(gaddr))
    for wn, arr in weights.items():
        lay = f.obj(found[wn]).first(0x08)
        daddr, dsize = struct.unpack_from("<QQ", lay, 2)
        assert dsize == arr.nbytes, wn
        keep = KEEP * arr.itemsize
        if dsize > 2 * keep:
            buf[daddr + keep:daddr + dsize - keep] = bytes(dsize - 2 * keep)
    with gzip.GzipFile(os.path.join(GOLD, "whenet_h5_skeleton.h5.gz"), "wb", compresslevel=9, mtime=0) as g:
        g.write(bytes(buf))
    digests = {"keep": KEEP, "layer_names": names, "meta": meta,
               "sha256": {k: hashlib.sha256(np.ascontiguousarray(v, dtype="<f4").tobytes()).hexdigest()
                          for k, v in weights.items()}}
    with open(os.path.join(GOLD, "whenet_h5_digests.json"), "w") as fo:
        json.dump(digests, fo, indent=0)
    print("%d tensors, skeleton %d bytes" % (len(weights), os.path.getsize(os.path.join(GOLD, "whenet_h5_skeleton.h5.gz"))))


if __name__ == "__main__":
    main(sys.argv[1])
