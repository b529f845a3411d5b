"""TSV container I/O (SURVEY.md section 8f-3): generativeimage2text_b200/tsv_io.py -- format checks everywhere, and
byte-for-byte against what the reference's tsv_io.py wrote for the same rows."""
import base64
import json
import os

import numpy as np
import pytest

from generativeimage2text_b200 import tsv_io
from helpers import load_golden


def _rows(n, seed=0):
    g = np.random.Generator(np.random.PCG64(seed))
    rows = []
    for i in range(n):
        blob = base64.b64encode(g.integers(0, 256, size=int(g.integers(1, 4000)), dtype=np.uint8).tobytes())
        rows.append(('img_%05d' % i, blob, json.dumps([{'caption': 'c %d' % i}])))
    return rows


def _files(path):
    base = os.path.splitext(path)[0]
    return [path, base + '.lineidx', base + '.lineidx.8b']


def test_writer_format_and_random_access(tmp_path):
    p = str(tmp_path / 'a' / 'data.tsv')
    rows = _rows(37)
    tsv_io.tsv_writer(iter(rows), p)
    raw = open(p, 'rb').read()
    lines = raw.split(b'\n')
    assert lines[-1] == b'' and len(lines) == 38
    off8 = np.fromfile(_files(p)[2], dtype='<i8')
    offtxt = [int(x) for x in open(_files(p)[1]).read().split()]
    starts = np.cumsum([0] + [len(l) + 1 for l in lines[:-1]])[:-1]
    assert off8.tolist() == offtxt == starts.tolist()
    t = tsv_io.TSVFile(p)
    assert len(t) == 37
    for i in (0, 36, 5, 20, 5, -1):
        k, b, c = t[i]
        assert (k, b.encode(), c) == rows[i]
        assert t.get_key(i) == rows[i][0]
    assert t.seek_first_columns() == [r[0] for r in rows]
    assert [r[0] for r in t] == [r[0] for r in rows]
    assert [r[0] for r in tsv_io.tsv_reader(p)] == [r[0] for r in rows]
    assert t.get_row_len(3) == len(lines[3]) + 1
    with pytest.raises(IndexError):
        t[37]


def test_empty_and_generate_lineidx(tmp_path):
    p = str(tmp_path / 'e.tsv')
    tsv_io.tsv_writer(iter([]), p)
    assert len(tsv_io.TSVFile(p)) == 0 and list(tsv_io.TSVFile(p)) == []
    q = str(tmp_path / 'g.tsv')
    rows = _rows(11, 3)
    tsv_io.tsv_writer(iter(rows), q)
    want = open(_files(q)[2], 'rb').read()
    os.remove(_files(q)[1])
    os.remove(_files(q)[2])
    with pytest.raises(FileNotFoundError):
        len(tsv_io.TSVFile(q))
    assert tsv_io.generate_lineidx(q) == 11
    assert open(_files(q)[2], 'rb').read() == want
    # last row without a trailing newline
    with open(q, 'ab') as fp:
        fp.write(b'tail\tx')
    assert tsv_io.generate_lineidx(q) == 12
    assert tsv_io.TSVFile(q)[11] == ['tail', 'x']


def test_concat_parts(tmp_path):
    parts, allrows = [], []
    for r in range(3):
        p = str(tmp_path / ('out.tsv.%d.3.tsv' % r))
        rows = _rows(5 + 4 * r, 10 + r)
        tsv_io.tsv_writer(iter(rows), p)
        parts.append(p)
        allrows += rows
    out = str(tmp_path / 'out.tsv')
    tsv_io.concat_tsv_files(parts, out)
    t = tsv_io.TSVFile(out)
    assert len(t) == len(allrows)
    for i in range(len(allrows)):
        assert t[i][0] == allrows[i][0] and t[i][1].encode() == allrows[i][1]


def test_byte_identical_to_reference_tsv_io(tmp_path):
    """Writer, reader and concat against what the reference's tsv_io.py produced for the same rows (stored by
    oracle/make_reference_units.py)."""
    g = load_golden('reference_tsv_io')
    rows = _rows(*g['meta']['rows'])
    a = str(tmp_path / 'ours.tsv')
    tsv_io.tsv_writer(iter(rows), a)
    for fa, ext in zip(_files(a), ('tsv', 'lineidx', 'lineidx_8b')):
        assert open(fa, 'rb').read() == g['written_' + ext].tobytes(), fa
    b = str(tmp_path / 'ref.tsv')
    for fb, ext in zip(_files(b), ('tsv', 'lineidx', 'lineidx_8b')):
        with open(fb, 'wb') as fp:
            fp.write(g['written_' + ext].tobytes())
    ours_on_ref = tsv_io.TSVFile(b)
    assert len(ours_on_ref) == len(rows)
    for i, ref_read in g['meta']['reads'].items():
        assert ours_on_ref[int(i)] == ref_read['row']
        assert ours_on_ref.get_key(int(i)) == ref_read['key']
    # merged parts: same .tsv and .lineidx.8b as the reference's concat
    split = g['meta']['split']
    p1, p2 = str(tmp_path / 'p.0.2.tsv'), str(tmp_path / 'p.1.2.tsv')
    tsv_io.tsv_writer(iter(rows[:split]), p1)
    tsv_io.tsv_writer(iter(rows[split:]), p2)
    o1 = str(tmp_path / 'm_ours.tsv')
    tsv_io.concat_tsv_files([p1, p2], o1)
    assert open(o1, 'rb').read() == g['merged_tsv'].tobytes()
    assert open(_files(o1)[2], 'rb').read() == g['merged_lineidx_8b'].tobytes()
