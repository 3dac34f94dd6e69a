"""The line-aligned block reader every file-level entry reads sync text with (poolgen_b200/sync_io.py: _line_blocks)."""
import numpy as np
import pytest

import poolgen_b200 as pb
from poolgen_b200 import sync_io


def _lines(crlf=False):
    body = []
    for i in range(23):
        if i % 7 == 3:
            body.append(b"#a comment line")
        elif i % 9 == 5:
            body.append(b"")
        else:
            body.append(b"chr%d\t%d\tN\t" % (i % 3, 100 + i) + b"\t".join([b"1:0:%d:0:0:0" % i] * (1 + i % 4)))
    return [ln + (b"\r\n" if crlf else b"\n") for ln in body]


def _file(tmp_path, lines, last_newline=True):
    data = b"".join(lines)
    if not last_newline:
        data = data.rstrip(b"\n")
    p = tmp_path / "t.sync"
    p.write_bytes(data)
    return str(p), data


def _blocks(fname, start, end, block_bytes, depth=1):
    bufs = [np.empty(block_bytes, np.uint8) for _ in range(depth)]
    held = []  # the caller may still read the last depth - 1 blocks when the next one arrives
    out = []
    for at, view in sync_io._line_blocks(fname, start, end, block_bytes, bufs):
        for a, v, copy in held:
            assert v.tobytes() == copy, a
        out.append((at, view.tobytes()))
        held = (held + [(at, view, out[-1][1])])[-(depth - 1):] if depth > 1 else []
    return out


def _check(blocks, data, start, end, block_bytes):
    """the blocks tile [start, end), end in a newline except the last, fit the block and are each as long as the
    greedy rule makes them: the next block's first line would not have fit"""
    assert b"".join(b for _, b in blocks) == data[start:end]
    at = start
    for i, (a, b) in enumerate(blocks):
        assert a == at and 0 < len(b) <= block_bytes
        at += len(b)
        if i + 1 < len(blocks):
            assert b.endswith(b"\n")
            nxt = blocks[i + 1][1]
            first = nxt[:nxt.find(b"\n") + 1] if b"\n" in nxt else nxt
            assert len(b) + len(first) > block_bytes


@pytest.mark.parametrize("crlf", [False, True])
@pytest.mark.parametrize("last_newline", [True, False])
def test_every_block_size(tmp_path, crlf, last_newline):
    lines = _lines(crlf)
    fname, data = _file(tmp_path, lines, last_newline)
    longest = max(len(ln) for ln in lines)
    for bb in range(longest, len(data) + 2):
        blocks = _blocks(fname, 0, len(data), bb)
        _check(blocks, data, 0, len(data), bb)
        if last_newline:
            assert blocks[-1][1].endswith(b"\n")
    # three buffers in turn (the scan's ring): the same blocks, and a block stays intact while two newer are read
    for bb in (longest, longest + 17, 3 * longest):
        assert _blocks(fname, 0, len(data), bb, depth=3) == _blocks(fname, 0, len(data), bb)


def test_line_at_the_block_size(tmp_path):
    lines = _lines()
    fname, data = _file(tmp_path, lines)
    longest = max(len(ln) for ln in lines)
    _check(_blocks(fname, 0, len(data), longest), data, 0, len(data), longest)
    with pytest.raises(pb.PgError, match="longer than the block size"):
        _blocks(fname, 0, len(data), longest - 1)
    # one line of exactly the block size, then the same line one byte longer
    one = tmp_path / "one.sync"
    one.write_bytes(b"c\t1\tN\t1:0:0:0:0:0\n")
    n = one.stat().st_size
    assert _blocks(str(one), 0, n, n) == [(0, one.read_bytes())]
    one.write_bytes(b"c\t1\tN\t1:0:0:0:0:0\nc\t12\tN\t1:0:0:0:0:0\n")
    with pytest.raises(pb.PgError, match="longer than the block size"):
        _blocks(str(one), 0, one.stat().st_size, n)


def test_last_line_without_newline(tmp_path):
    """a last line without a newline joins the block before it where it fits, and is never refused when it fits
    the block on its own"""
    p = tmp_path / "u.sync"
    p.write_bytes(b"x" * 20)
    assert _blocks(str(p), 0, 20, 64) == [(0, b"x" * 20)]
    assert _blocks(str(p), 0, 20, 20) == [(0, b"x" * 20)]
    with pytest.raises(pb.PgError, match="longer than the block size"):
        _blocks(str(p), 0, 20, 19)
    data = b"a" * 20 + b"\n" + b"b" * 20
    p.write_bytes(data)
    for bb in (30, 40):
        assert _blocks(str(p), 0, len(data), bb) == [(0, data[:21]), (21, data[21:])]
    assert _blocks(str(p), 0, len(data), 41) == [(0, data)]


@pytest.mark.parametrize("last_newline", [True, False])
def test_file_split_ranges(tmp_path, last_newline):
    lines = _lines() * 4
    fname, data = _file(tmp_path, lines, last_newline)
    longest = max(len(ln) for ln in lines)
    for n_threads in (1, 2, 3, 5):
        splits = pb.find_file_splits(fname, n_threads)
        for bb in (longest, 2 * longest + 3, len(data)):
            whole = []
            for s, e in zip(splits[:-1], splits[1:]):
                blocks = _blocks(fname, s, e, bb)
                _check(blocks, data, s, e, bb)
                whole += blocks
            assert b"".join(b for _, b in whole) == data
