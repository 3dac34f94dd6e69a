"""A kinship handle stays usable after one of its scratch allocations is refused."""
import numpy as np
import pytest

import poolgen_b200 as pb

pytestmark = pytest.mark.gpu


def _load(kin, text, fs, max_loci):
    nl, off, pos, loc, alle = kin.append_sync_text(text, fs, max_loci)
    return nl, pos, loc, alle, kin.get_columns(0, kin.columns)


def test_kinship_reload_after_refused_allocation(ctx):
    """append_sync_text with max_loci = 2^40 asks for terabytes of loader scratch: the allocation is refused and the
    call raises.  After reset() the handle loads the same text again, and what it holds equals a fresh handle's load."""
    n, A, L = 16, 4, 800
    out = np.empty(L * (16 + n * 24), dtype=np.uint8)
    text = out[:pb.synth_sync_text_host(0x5EC0, 0, L, n, A, out)].tobytes()
    fs = pb.FilterStats(pool_sizes=np.full(n, 1.0 / n))

    fresh = pb.Kinship(ctx, n, 6 * L)
    expect = _load(fresh, text, fs, L)
    fresh.close()
    assert expect[0] == L and expect[4].shape[0] > 0

    kin = pb.Kinship(ctx, n, 6 * L)
    _load(kin, text, fs, L)
    with pytest.raises(pb.PgError):
        kin.append_sync_text(text, fs, 1 << 40)
    kin.reset()
    got = _load(kin, text, fs, L)
    kin.close()

    assert got[0] == expect[0]
    for g, e in zip(got[1:], expect[1:]):
        assert np.array_equal(g, e, equal_nan=True)
