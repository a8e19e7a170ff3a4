"""Write tests/golden/hdf5_sample.h5, the fixture of dlrm_jl_b200.hdf5_min's test.

    python tests/golden/make_hdf5_sample.py

The file has the container shape of the reference's PyTorch golden files (the subset hdf5_min
reads), laid out as the HDF5 file format specification (version 0 superblock) describes it:
superblock v0, a root group with a local heap and a version 1 B-tree over two symbol-table
nodes, one version 1 object header per dataset (dataspace v1, datatype v1, contiguous layout
v3), little-endian data.  The datasets are tests/helpers.py:hdf5_sample_arrays.
"""
import os
import struct
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(HERE, "..", ".."))
from tests.helpers import hdf5_sample_arrays  # noqa: E402

UNDEF = 0xFFFFFFFFFFFFFFFF
LEAF_K, INTERNAL_K = 4, 16          # group leaf / internal node K of the superblock


def _pad8(b: bytes) -> bytes:
    return b + b"\0" * (-len(b) % 8)


def _object_header(messages) -> bytes:
    body = b"".join(struct.pack("<HHB3x", mtype, len(_pad8(data)), 0) + _pad8(data) for mtype, data in messages)
    return struct.pack("<BBHII4x", 1, 0, len(messages), 1, len(body)) + body


def _datatype(a: np.ndarray) -> bytes:
    if a.dtype == np.float32:        # IEEE little-endian, implied mantissa msb, sign bit 31
        return struct.pack("<B3BI", 0x11, 0x20, 31, 0, 4) + struct.pack("<HHBBBBI", 0, 32, 23, 8, 0, 23, 127)
    if a.dtype == np.int64:          # two's complement little-endian
        return struct.pack("<B3BI", 0x10, 0x08, 0, 0, 8) + struct.pack("<HH", 0, 64)
    raise ValueError(a.dtype)


def write_hdf5(path: str, arrays: dict) -> None:
    names = sorted(arrays)
    heap_data = b"\0" * 8                # offset 0: the empty name of the root group
    name_off = {}
    for n in names:
        name_off[n] = len(heap_data)
        heap_data += _pad8(n.encode() + b"\0")
    half = (len(names) + 1) // 2
    leaves = [names[:half], names[half:]]
    assert all(0 < len(leaf) <= 2 * LEAF_K for leaf in leaves)

    # fixed-size structures first, then the datasets' headers and data, addresses known in order
    root_oh = 96
    heap = root_oh + len(_object_header([(0x11, bytes(16))]))
    heap_seg = heap + 32
    btree = heap_seg + len(heap_data)
    btree_size = 24 + (2 * INTERNAL_K + 1) * 8 + 2 * INTERNAL_K * 8
    snods = [btree + btree_size + i * (8 + 2 * LEAF_K * 40) for i in range(len(leaves))]
    pos = snods[-1] + 8 + 2 * LEAF_K * 40
    headers, data_at = {}, {}
    for n in names:
        a = np.asarray(arrays[n])
        dataspace = struct.pack("<BBB5x", 1, a.ndim, 0) + b"".join(struct.pack("<Q", d) for d in a.shape)
        size = len(_object_header([(0x01, dataspace), (0x03, _datatype(a)), (0x08, bytes(18))]))
        data_at[n] = pos + size
        layout = struct.pack("<BBQQ", 3, 1, data_at[n], a.nbytes)
        headers[n] = (pos, _object_header([(0x01, dataspace), (0x03, _datatype(a)), (0x08, layout)]))
        pos = data_at[n] + a.nbytes
    eof = pos

    out = bytearray(eof)

    def put(addr: int, b: bytes) -> None:
        out[addr:addr + len(b)] = b

    put(0, b"\x89HDF\r\n\x1a\n" + struct.pack("<BBBBBBBBHHI", 0, 0, 0, 0, 0, 8, 8, 0, LEAF_K, INTERNAL_K, 0))
    put(24, struct.pack("<QQQQ", 0, UNDEF, eof, UNDEF))
    put(56, struct.pack("<QQI4xQQ", 0, root_oh, 1, btree, heap))          # root symbol-table entry
    put(root_oh, _object_header([(0x11, struct.pack("<QQ", btree, heap))]))
    put(heap, b"HEAP" + struct.pack("<B3xQQQ", 0, len(heap_data), UNDEF, heap_seg))
    put(heap_seg, heap_data)
    node = b"TREE" + struct.pack("<BBHQQ", 0, 0, len(leaves), UNDEF, UNDEF) + struct.pack("<Q", 0)
    for addr, leaf in zip(snods, leaves):
        node += struct.pack("<QQ", addr, name_off[leaf[-1]])             # child, then the largest name in it
    put(btree, node)
    for addr, leaf in zip(snods, leaves):
        put(addr, b"SNOD" + struct.pack("<BBH", 1, 0, len(leaf))
            + b"".join(struct.pack("<QQI4x16x", name_off[n], headers[n][0], 0) for n in leaf))
    for n in names:
        put(*headers[n])
        put(data_at[n], np.asarray(arrays[n]).astype(arrays[n].dtype.newbyteorder("<")).tobytes())
    with open(path, "wb") as fh:
        fh.write(bytes(out))


if __name__ == "__main__":
    dst = os.path.join(HERE, "hdf5_sample.h5")
    write_hdf5(dst, hdf5_sample_arrays())
    print(f"{dst}: {os.path.getsize(dst)} bytes")
