"""Generates tests/golden/example.index, the .index file of the example database:

    python tests/golden/make_index_golden.py

The reference's ``Database.create_index`` (src/database.py:227-243) puts every fingerprint of the database, in vid
order, into ``faiss.IndexFlatL2(480)`` and calls ``faiss.write_index``.  This script writes the same file field by field
from the faiss 1.7.4 layout of an IndexFlat (impl/index_write.cpp): fourcc "IxF2", d (int32), ntotal (int64), two
int64 dummies (1 << 20), is_trained (1 byte), metric_type (int32, METRIC_L2 = 1, so no metric_arg), the element count
of the code vector as uint64 in units of 4 bytes, then the rows as float32.  It needs neither faiss nor a GPU."""
import os
import struct

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))


def main():
    rows = np.load(os.path.join(HERE, 'example-dct.npz'))['dct']     # vid order of the example database
    n, d = rows.shape
    head = b'IxF2' + struct.pack('<iqqqBi', d, n, 1 << 20, 1 << 20, 1, 1) + struct.pack('<Q', n * d)
    with open(os.path.join(HERE, 'example.index'), 'wb') as f:
        f.write(head + rows.astype('<f4').tobytes())
    print('example.index', n, 'x', d)


if __name__ == '__main__':
    main()
