"""The reference's database build and search flow on the faiss shim, pinned to the reference's own outputs.

With ``install_faiss_shim()`` the reference's ``import faiss`` binds to dctdomain_b200.index, so its
``Database.create_index`` (src/database.py:227-243) and ``query_db.search_db`` (src/query_db.py:62-91) run on the GPU
index without edits.  The reference's modules are not part of this repository: these tests make the faiss calls of
those two functions (SURVEY.md §3.4) on a database with the reference's SQLite schema (tests/minidb.py) and compare with
the reference's shipped ``test/test/example-search.txt`` and ``example-dct.npz`` (the ``save_fprints`` output of the
example database), and with ``example.index``, the faiss IndexFlatL2 file of that database
(tests/golden/make_index_golden.py)."""
import logging
import os
import sys
from io import BytesIO

import numpy as np
import pytest

from conftest import GOLDEN as G
from minidb import MiniDB

pytestmark = pytest.mark.gpu


@pytest.fixture()
def faiss():
    import dctdomain_b200
    saved = sys.modules.get('faiss')
    try:
        yield dctdomain_b200.install_faiss_shim()
    finally:
        sys.modules.pop('faiss', None)
        if saved is not None:
            sys.modules['faiss'] = saved


def _build_db(tmp_path, name='example'):
    """The example database (fingerprints in the vid order of the original) with the reference's schema; ``path`` is
    the database path without its extension, as the reference's ``Database`` keeps it."""
    z = np.load(os.path.join(G, 'example-dct.npz'))
    db = MiniDB(str(tmp_path / f'{name}.db'), z)
    db.path = str(tmp_path / name)
    return db, z


def _golden_index():
    return open(os.path.join(G, 'example.index'), 'rb').read()


def test_reference_database_and_search_db_on_the_shim(faiss, tmp_path, caplog):
    from dctdomain_b200 import query_db as dq
    db, z = _build_db(tmp_path)
    # Database.create_index: every blob in vid order -> IndexFlatL2(480).add -> write_index
    rows = db.cur.execute(""" SELECT fingerprint FROM fingerprints """).fetchall()
    fps = np.array([np.load(BytesIO(r[0]), allow_pickle=True) for r in rows], dtype=np.int8)
    index = faiss.IndexFlatL2(fps.shape[1])
    index.add(fps)
    faiss.write_index(index, f'{db.path}.index')
    db.close()
    assert open(f'{db.path}.index', 'rb').read() == _golden_index()
    # search_db: read_index, the metric flipped after the load, one index.search per query protein (pid ascending)
    index = faiss.read_index(f'{db.path}.index')
    index.metric_type = faiss.METRIC_L1
    path = f'{db.path}.db'
    query_db, fp_db = MiniDB(path), MiniDB(path)
    with caplog.at_level(logging.INFO):
        for (pid,) in query_db.cur.execute(""" SELECT pid FROM sequences """).fetchall():
            qfps = query_db.load_fprints(pid=pid)
            dm, im = index.search(np.array([fp[1] for fp in qfps]), 50)
            dq.get_top_hits(dm, im, 50, fp_db, query_db, [fp[0] for fp in qfps], 'l1')
    query_db.close()
    fp_db.close()
    lines = [r.getMessage() for r in caplog.records if r.getMessage().startswith('Query:')]
    assert lines == open(os.path.join(G, 'example-search.txt')).read().splitlines()


def test_vectorised_create_index_and_save_fprints_equal_the_reference(faiss, tmp_path):
    """dctdomain_b200.database.create_index / save_fprints on the example database: byte-identical .index, the arrays
    and dtypes of the reference's example-dct.npz."""
    from dctdomain_b200 import database as ddb
    db, z = _build_db(tmp_path)
    ddb.create_index(db)
    assert open(f'{db.path}.index', 'rb').read() == _golden_index()
    ddb.save_fprints(db, str(tmp_path / 'ours.npz'))
    b = np.load(tmp_path / 'ours.npz')
    assert sorted(z.files) == sorted(b.files)
    for key in z.files:
        assert z[key].dtype == b[key].dtype and np.array_equal(z[key], b[key]), key
    db.close()
