"""Host model of the 16-bit quotient-tag visited table (search_common.cuh Tag16Map / tag16_of; the
shared-memory visited set of search_kernel_v3 and the level-1 table of search_kernel_v2): the id ->
(bucket, tag) map must be a bijection on [0, 2^K) with 14-bit tags, and the multiply-shift
division the device uses must be exact."""
import numpy as np
import pytest


def tag_map(K, nbk):
    s = 0
    while (1 << s) < nbk:
        s += 1
    assert K + s <= 32
    magic = ((1 << (K + s)) + nbk - 1) // nbk
    assert magic < (1 << 32)
    return (1 << K) - 1, magic, K + s


@pytest.mark.parametrize("K,nbk", [(20, 283), (20, 64), (20, 577), (17, 16), (22, 300), (22, 1024), (12, 16)])
def test_bucket_tag_is_a_bijection_with_14_bit_tags(K, nbk):
    assert (1 << K) <= nbk << 14, "host picks n_buckets >= 2^K / 2^14"
    kmask, magic, shift = tag_map(K, nbk)
    ids = np.arange(1 << K, dtype=np.uint64)
    h = (ids * np.uint64(0x9E3779B1)) & np.uint64(kmask)          # odd multiplier mod 2^K: a bijection
    assert len(np.unique(h)) == 1 << K
    tag = (h * np.uint64(magic)) >> np.uint64(shift)              # device: 64-bit multiply-shift
    assert np.array_equal(tag, h // np.uint64(nbk)), "multiply-shift division must be exact for h < 2^K"
    bucket = h - tag * np.uint64(nbk)
    assert bucket.max() < nbk and tag.max() < (1 << 14)
    key = bucket * np.uint64(1 << 14) + tag
    assert len(np.unique(key)) == 1 << K, "(bucket, tag) must identify the id"
    # displaced copies carry d = 1, 2 in the top two bits and never look empty
    assert ((2 << 14) | int(tag.max())) < 0xFFFF


def test_halfword_zero_trick_is_exact():
    """bucket16_insert scans a bucket with (v - 0x00010001) & ~v & 0x80008000: non-zero exactly
    when one of the two 16-bit halves of v is zero; with the low half checked first the position of
    an empty (0xFFFF) entry is exact too."""
    rng = np.random.default_rng(0)
    special = np.array([0, 1, 0xFFFF, 0x8000, 0x7FFF, 0xBFFF, 0x0100, 0x00FF], np.uint64)
    lo = np.concatenate([special.repeat(len(special)), rng.integers(0, 1 << 16, 200000).astype(np.uint64)])
    hi = np.concatenate([np.tile(special, len(special)), rng.integers(0, 1 << 16, 200000).astype(np.uint64)])
    # force plenty of zero halves
    lo[::7] = 0
    hi[::11] = 0
    v = (hi << np.uint64(16)) | lo
    m32 = np.uint64(0xFFFFFFFF)
    flag = ((v - np.uint64(0x00010001)) & m32) & (~v & m32) & np.uint64(0x80008000)
    assert np.array_equal(flag != 0, (lo == 0) | (hi == 0))
    # empty-slot position: s = ~v has 0xFFFF where v has a zero half
    s = ~v & m32
    has_empty = flag != 0
    half = np.where((s & np.uint64(0xFFFF)) == np.uint64(0xFFFF), 0, 1)
    truth = np.where(lo == 0, 0, 1)
    assert np.array_equal(half[has_empty], truth[has_empty])


class Tag16Table:
    """Sequential model of bucket16_insert (search_common.cuh): 16 entries of 16 bits per bucket,
    entry = (displacement << 14) | tag, 0xFFFF empty, at most two buckets of displacement."""

    def __init__(self, K, nbk):
        self.kmask, self.magic, self.shift = tag_map(K, nbk)
        self.nbk = nbk
        self.t = np.full((nbk, 16), 0xFFFF, np.uint16)

    def insert(self, id_):
        """-> (newly_inserted, overflow)"""
        h = (id_ * 0x9E3779B1) & 0xFFFFFFFF & self.kmask
        tag = (h * self.magic) >> self.shift
        b = h - tag * self.nbk
        for d in range(3):
            want = (d << 14) | tag
            row = self.t[b]
            if (row == want).any():
                return False, False
            empty = np.flatnonzero(row == 0xFFFF)
            if len(empty):
                row[empty[0]] = want
                return True, False
            b = 0 if b + 1 == self.nbk else b + 1
        return False, True


@pytest.mark.parametrize("K,nbk,n_ids,seed", [(20, 283, 3400, 0), (20, 283, 3900, 1), (17, 64, 800, 2), (12, 16, 200, 3), (20, 64, 880, 4)])
def test_tag16_table_is_an_exact_set(K, nbk, n_ids, seed):
    """Up to the 87.5 % load limit the kernel enforces (14 of 16 entries per bucket on average) the
    table behaves exactly like a set; an overflow may only be reported, never a wrong answer."""
    rng = np.random.default_rng(seed)
    assert n_ids <= nbk * 14
    universe = rng.choice(1 << K, n_ids, replace=False)
    stream = np.concatenate([universe, rng.choice(universe, 3 * n_ids)])   # every id again, several times
    rng.shuffle(stream)
    table, seen, overflows = Tag16Table(K, nbk), set(), 0
    for id_ in stream.tolist():
        fresh, ovf = table.insert(id_)
        if ovf:
            overflows += 1          # the kernel re-runs the query with the 32-bit table
            continue
        assert fresh == (id_ not in seen), id_
        seen.add(id_)
    assert overflows <= 0.02 * len(stream)
