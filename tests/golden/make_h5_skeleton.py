#!/usr/bin/env python
"""
The reference's genomad/data/nn_classifier.h5 (24.6 MB) without its dataset payloads: every byte that is not the contiguous data
of one of the 32 weight datasets (HDF5 superblock, object headers, B-trees, heaps, attributes -- 34,924 bytes), with each payload's
name, offset and size.  The payloads are the arrays of genomad_b200/data/nn_classifier.npz, which also records the file's sha256, so
``rebuild`` reproduces the reference file exactly (tests/test_host_cpu.py::test_h5lite_reads_reference_file_if_present checks the
sha256 and reads the rebuilt file).

    python tests/golden/make_h5_skeleton.py REFERENCE/genomad/data/nn_classifier.h5    # -> tests/golden/nn_classifier_h5_skeleton.npz
"""
import hashlib
import sys
from pathlib import Path

import numpy as np

HERE = Path(__file__).resolve().parent
ROOT = HERE.parents[1]
OUT = HERE / "nn_classifier_h5_skeleton.npz"


def rebuild(skeleton_npz, weights_npz) -> bytes:
    s, z = np.load(skeleton_npz), np.load(weights_npz)
    rest = s["rest"].tobytes()
    buf, pos, r = bytearray(), 0, 0
    for name, off, n in zip(s["names"], s["offsets"].tolist(), s["nbytes"].tolist()):
        buf += rest[r:r + off - pos]
        r += off - pos
        payload = np.ascontiguousarray(z[name], z[name].dtype.newbyteorder("<")).tobytes()
        assert len(payload) == n, name
        buf += payload
        pos = off + n
    buf += rest[r:]
    assert len(buf) == int(s["file_size"])
    return bytes(buf)


def main():
    sys.path.insert(0, str(ROOT))
    from genomad_b200 import h5lite
    src = Path(sys.argv[1])
    raw = src.read_bytes()
    f = h5lite.H5File(src)
    regions = sorted((f.offsets[k], f.datasets[k].nbytes, k) for k in f.datasets)
    rest, pos = bytearray(), 0
    for off, n, _ in regions:
        assert off >= pos
        rest += raw[pos:off]
        pos = off + n
    rest += raw[pos:]
    np.savez_compressed(OUT, names=np.array([k for _, _, k in regions]), offsets=np.array([o for o, _, _ in regions], np.int64),
                        nbytes=np.array([n for _, n, _ in regions], np.int64), file_size=np.int64(len(raw)),
                        rest=np.frombuffer(bytes(rest), np.uint8))
    weights = ROOT / "genomad_b200" / "data" / "nn_classifier.npz"
    assert rebuild(OUT, weights) == raw
    assert hashlib.sha256(raw).hexdigest() == str(np.load(weights)["__sha256__"])
    print(f"wrote {OUT} ({len(rest)} bytes outside the payloads)")


if __name__ == "__main__":
    main()
