"""results.h5 without h5py: the minimal earliest-format HDF5 writer / reader (pydnmfk_b200/h5min.py) behind
data_io.write_results / read_results (reference data_io.py:199-209, read back at pyDNMFk.py:278)."""
import os
import struct

import numpy as np
import pytest

from pydnmfk_b200 import h5min
from pydnmfk_b200 import data_io

NAMES = ('clusterSilhouetteCoefficients', 'avgSilhouetteCoefficients', 'L_err', 'L_errDist', 'avgErr', 'ErrTol', 'AIC')


def _results(k=4, seed=0):
    r = np.random.default_rng(seed)
    return {'clusterSilhouetteCoefficients': r.random(k), 'avgSilhouetteCoefficients': np.float64(r.random()),
            'L_err': np.float32(r.random()), 'L_errDist': r.random(20).astype(np.float32), 'avgErr': r.random(),
            'ErrTol': np.float32(0.125), 'AIC': np.array(r.random((2, 3)))}


def test_round_trip_keeps_names_shapes_dtypes_values(tmp_path):
    d = _results()
    p = str(tmp_path / 'results.h5')
    h5min.write(p, d)
    back = h5min.read(p)
    assert sorted(back) == sorted(NAMES)
    for name, val in d.items():
        val = np.asarray(val)
        assert back[name].shape == val.shape and back[name].dtype == val.dtype, name
        assert np.array_equal(back[name], val), name


def test_integer_empty_and_many_datasets(tmp_path):
    d = {'d%03d' % i: np.arange(i, dtype=np.int32 if i % 2 else np.int64).reshape(-1) for i in range(40)}
    d['u8'] = np.arange(7, dtype=np.uint8)
    d['big'] = np.random.default_rng(1).random((257, 33))
    p = str(tmp_path / 'many.h5')
    h5min.write(p, d)
    back = h5min.read(p)
    assert sorted(back) == sorted(d)
    for name, val in d.items():
        assert back[name].dtype == val.dtype and np.array_equal(back[name], val), name
    with pytest.raises(TypeError):
        h5min.write(p, {'s': np.array(['a', 'b'])})


def test_fixed_structures_of_the_format(tmp_path):
    """The fields libhdf5 checks before anything else, at the offsets the file-format specification gives them."""
    p = str(tmp_path / 'results.h5')
    h5min.write(p, _results())
    b = open(p, 'rb').read()
    assert b[:8] == b'\x89HDF\r\n\x1a\n'
    assert b[8] == 0 and b[13] == 8 and b[14] == 8                      # superblock v0, 8-byte offsets and lengths
    leaf_k, internal_k = struct.unpack_from('<HH', b, 16)
    assert (leaf_k, internal_k) == (4, 16)
    base, free, eof, driver = struct.unpack_from('<QQQQ', b, 24)
    assert base == 0 and free == h5min.UNDEF and driver == h5min.UNDEF and eof == len(b)
    name_off, root, cache, _ = struct.unpack_from('<QQII', b, 56)
    btree, heap = struct.unpack_from('<QQ', b, 80)
    assert name_off == 0 and cache == 1 and root % 8 == 0 and btree % 8 == 0 and heap % 8 == 0
    assert b[root] == 1 and struct.unpack_from('<H', b, root + 2)[0] == 1  # v1 object header with one message ...
    mtype, msize = struct.unpack_from('<HH', b, root + 16)
    assert mtype == 0x11 and msize == 16                                # ... the symbol-table message
    assert struct.unpack_from('<QQ', b, root + 24) == (btree, heap)
    assert b[btree:btree + 4] == b'TREE' and b[btree + 4] == 0 and b[btree + 5] == 0
    used, left, right = struct.unpack_from('<HQQ', b, btree + 6)
    assert used == 1 and left == h5min.UNDEF and right == h5min.UNDEF
    assert b[heap:heap + 4] == b'HEAP'
    hsize, hfree, hdata = struct.unpack_from('<QQQ', b, heap + 8)
    assert hsize % 8 == 0 and hdata % 8 == 0
    nxt, fsize = struct.unpack_from('<QQ', b, hdata + hfree)
    assert nxt == 1 and hfree + fsize == hsize                          # one free block, up to the end of the segment
    key0, snod, key1 = struct.unpack_from('<QQQ', b, btree + 24)
    assert key0 == 0 and b[snod:snod + 4] == b'SNOD' and b[snod + 4] == 1
    nsym = struct.unpack_from('<H', b, snod + 6)[0]
    assert nsym == len(NAMES)
    names = []
    for i in range(nsym):
        off, ohdr, ctype, _ = struct.unpack_from('<QQII', b, snod + 8 + 40 * i)
        end = b.index(b'\x00', hdata + off)
        names.append(b[hdata + off:end].decode())
        assert ctype == 0 and ohdr % 8 == 0 and b[ohdr] == 1
        nmsg, _refs, size = struct.unpack_from('<HII', b, ohdr + 2)
        pos, types = ohdr + 16, []
        for _ in range(nmsg):
            t, s = struct.unpack_from('<HH', b, pos)
            assert s % 8 == 0
            types.append(t)
            pos += 8 + s
        assert pos == ohdr + 16 + size and types == [0x1, 0x3, 0x5, 0x8]
    assert names == sorted(NAMES) and names[-1] == b[hdata + key1:b.index(b'\x00', hdata + key1)].decode()
    # the float32 datatype message of L_errDist: class 1 version 1, little endian, msb-implied mantissa, sign bit 31
    off, ohdr = struct.unpack_from('<QQ', b, snod + 8 + 40 * names.index('L_errDist'))
    pos = ohdr + 16
    pos += 8 + struct.unpack_from('<H', b, pos + 2)[0]
    dt = b[pos + 8:pos + 8 + 20]
    assert dt[:4] == bytes([0x11, 0x20, 31, 0]) and struct.unpack_from('<I', dt, 4)[0] == 4
    assert struct.unpack_from('<HHBBBBI', dt, 8) == (0, 32, 23, 8, 0, 23, 127)


def _h5py_style_file(arr):
    """A file laid out the way libhdf5's default (earliest) writer does it -- built here by hand, not by h5min.write: data
    address before the headers, object header with a modification-time and a NIL message and a continuation block."""
    def msg(t, data, flags=0):
        data = data + b'\x00' * (-len(data) % 8)
        return struct.pack('<HHB3s', t, len(data), flags, b'\x00' * 3) + data
    name = b'AIC\x00'
    heap = b'\x00' * 8 + name + b'\x00' * 4 + struct.pack('<QQ', 1, 72) + b'\x00' * 56
    raw = arr.astype('<f8').tobytes()
    out = bytearray(2048 + len(raw))
    A_ROOT, A_TREE, A_HEAP, A_HDATA, A_SNOD, A_OBJ, A_CONT, A_DATA = 96, 136, 680, 712, 800, 1128, 1400, 2048
    out[0:8] = b'\x89HDF\r\n\x1a\n'
    out[8:24] = struct.pack('<BBBBBBBBHHI', 0, 0, 0, 0, 0, 8, 8, 0, 4, 16, 0)
    out[24:56] = struct.pack('<QQQQ', 0, h5min.UNDEF, len(out), h5min.UNDEF)
    out[56:96] = struct.pack('<QQIIQQ', 0, A_ROOT, 1, 0, A_TREE, A_HEAP)
    body = msg(0x11, struct.pack('<QQ', A_TREE, A_HEAP))
    out[A_ROOT:A_ROOT + 16 + len(body)] = struct.pack('<BBHII4s', 1, 0, 1, 1, len(body), b'\x00' * 4) + body
    out[A_TREE:A_TREE + 48] = b'TREE' + struct.pack('<BBHQQ', 0, 0, 1, h5min.UNDEF, h5min.UNDEF) + struct.pack('<QQQ', 0, A_SNOD, 8)
    out[A_HEAP:A_HEAP + 32] = b'HEAP' + struct.pack('<B3sQQQ', 0, b'\x00' * 3, len(heap), 16, A_HDATA)
    out[A_HDATA:A_HDATA + len(heap)] = heap
    out[A_SNOD:A_SNOD + 48] = b'SNOD' + struct.pack('<BBH', 1, 0, 1) + struct.pack('<QQII16s', 8, A_OBJ, 0, 0, b'\x00' * 16)
    space = struct.pack('<BBBBI', 1, arr.ndim, 1, 0, 0) + b''.join(struct.pack('<Q', d) for d in arr.shape) * 2   # + max dims
    dtype = struct.pack('<BBBBI', 0x11, 0x20, 63, 0, 8) + struct.pack('<HHBBBBI', 0, 64, 52, 11, 0, 52, 1023)
    cont = msg(0x08, struct.pack('<BBQQ', 3, 1, A_DATA, len(raw))) + msg(0x12, struct.pack('<B3sI', 1, b'\x00' * 3, 1700000000))
    body = (msg(0x01, space) + msg(0x03, dtype, 1) + msg(0x05, struct.pack('<BBBBI', 2, 2, 2, 1, 0))
            + msg(0x00, b'\x00' * 24) + msg(0x10, struct.pack('<QQ', A_CONT, len(cont))))
    out[A_OBJ:A_OBJ + 16 + len(body)] = struct.pack('<BBHII4s', 1, 0, 7, 1, len(body), b'\x00' * 4) + body
    out[A_CONT:A_CONT + len(cont)] = cont
    out[A_DATA:A_DATA + len(raw)] = raw
    return bytes(out)


def test_reader_parses_a_library_style_layout(tmp_path):
    arr = np.random.default_rng(3).random((5, 7))
    p = tmp_path / 'lib.h5'
    p.write_bytes(_h5py_style_file(arr))
    back = h5min.read(str(p))
    assert list(back) == ['AIC'] and back['AIC'].dtype == np.float64 and np.array_equal(back['AIC'], arr)


def _libhdf5_sample():
    """A file written by libhdf5 itself, copied from scipy's test data (scipy/io/matlab/tests/data, BSD-3-Clause):
    MATLAB v7.3 = HDF5 behind a 512-byte user block, earliest format: v0 superblock, symbol-table root group, v1
    object headers."""
    return os.path.join(os.path.dirname(os.path.abspath(__file__)), 'golden', 'testhdf5_7.4_GLNX86.mat')


def test_reader_against_a_file_written_by_libhdf5():
    back = h5min.read(_libhdf5_sample())
    assert list(back) == ['testdouble'] and back['testdouble'].shape == (9, 1)
    assert np.allclose(back['testdouble'][:, 0], np.arange(9) * np.pi / 4, rtol=0, atol=1e-15)


def test_writer_messages_equal_the_ones_libhdf5_wrote(tmp_path):
    """Datatype and dataspace messages, B-tree node prefix, heap free block: byte for byte what libhdf5 put into its file."""
    ref = open(_libhdf5_sample(), 'rb').read()[512:]
    arr = np.arange(9, dtype=np.float64).reshape(9, 1) * np.pi / 4
    p = str(tmp_path / 'mine.h5')
    h5min.write(p, {'testdouble': arr})
    mine = open(p, 'rb').read()

    def messages(b):
        root = struct.unpack_from('<Q', b, 64)[0]
        btree, heap = struct.unpack_from('<QQ', b, root + 24)
        snod = struct.unpack_from('<Q', b, btree + 32)[0]
        ohdr = struct.unpack_from('<Q', b, snod + 16)[0]
        nmsg = struct.unpack_from('<H', b, ohdr + 2)[0]
        pos, out = ohdr + 16, {}
        for _ in range(nmsg):
            t, s, f = struct.unpack_from('<HHB', b, pos)
            out.setdefault(t, (b[pos + 8:pos + 8 + s], f))
            pos += 8 + s
        hsize, hfree, hdata = struct.unpack_from('<QQQ', b, heap + 8)
        return out, b[btree:btree + 32], struct.unpack_from('<QQ', b, hdata + hfree) + (hsize - hfree,), b[hdata:hdata + 24]
    m_ref, bt_ref, free_ref, names_ref = messages(ref)
    m_mine, bt_mine, free_mine, names_mine = messages(mine)
    assert m_mine[0x3] == m_ref[0x3]                      # datatype: IEEE float64, little endian (+ the 'constant' flag)
    assert m_mine[0x1][0] == m_ref[0x1][0]                # dataspace v1, rank 2, dims 9 x 1
    assert bt_mine == bt_ref                              # TREE, group node, level 0, one entry, no siblings, key[0] = 0
    assert names_mine == names_ref                        # heap: empty root name, then 'testdouble' padded to 8
    assert free_mine[0] == free_ref[0] == 1 and free_mine[1] == free_mine[2] and free_ref[1] == free_ref[2]
    assert np.array_equal(h5min.read(p)['testdouble'], h5min.read(_libhdf5_sample())['testdouble'])


def test_reader_handles_a_user_block(tmp_path):
    """Superblock at 512 behind a user block, base address 512 (what MATLAB does): every address is relative to it."""
    d = _results(seed=9)
    p = str(tmp_path / 'plain.h5')
    h5min.write(p, d)
    b = bytearray(open(p, 'rb').read())
    b[24:32] = struct.pack('<Q', 512)                    # base address
    q = tmp_path / 'userblock.h5'
    q.write_bytes(b'MATLAB 7.3-like user block'.ljust(512, b' ') + bytes(b))
    back = h5min.read(str(q))
    for name, val in d.items():
        assert np.array_equal(back[name], np.asarray(val)), name
    with pytest.raises(ValueError):
        h5min.read(__file__)


def test_data_io_results_file(tmp_path, monkeypatch):
    """write_results / read_results: results.h5 exists with or without h5py; the npz twin only without it."""
    d = _results(seed=5)
    data_io.write_results(str(tmp_path) + '/', d)
    assert (tmp_path / 'results.h5').exists()
    back = data_io.read_results(str(tmp_path) + '/')
    for name, val in d.items():
        assert np.allclose(back[name], np.asarray(val)), name
    if data_io._h5py() is None:
        assert (tmp_path / 'results.npz').exists()
        # a results.h5 the minimal reader cannot parse falls back to the npz twin
        (tmp_path / 'results.h5').write_bytes(b'\x89HDF\r\n\x1a\n' + b'\x02' + b'\x00' * 100)
        back = data_io.read_results(str(tmp_path) + '/')
        assert np.allclose(back['AIC'], d['AIC'])
