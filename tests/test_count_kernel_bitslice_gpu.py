"""
The packed count kernel (log_discrete_packed_kernel) counts its rows' codes with a carry-save adder tree over
each lane's words and one warp reduction per row.  Its counts and the count tuples it feeds the tally must be
the uint8 kernel's (log_discrete_stream_kernel) exactly: at every horizon around the word, vector and
per-lane-slot boundaries, past one full round of vectors per lane (H > 10240 two-bit codes), at rows whose
counts pass 2^16, with garbage in the pad bits and pad bytes, at N not a multiple of 32 rows, and on rows off
16-byte alignment (the byte path).
"""
import numpy as np
import pytest
import torch

from oracle import lev_oracle as lo

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def eng():
    from rlmd_b200 import engine
    return engine


def _codes(rs, n, h, k):
    p = rs.dirichlet(np.ones(k))       # uneven code frequencies: every count differs
    return rs.choice(k, size=(n, h), p=p).astype(np.uint8)


def _garbage_pad(eng, packed):
    """The same codes with every pad bit of the last code byte and every pad byte of a row set."""
    per = 8 // packed.bits
    h = packed.horizon
    nb = (h + per - 1) // per
    d = packed.data.cpu().numpy().copy()
    if h % per:
        d[:, nb - 1] |= np.uint8((0xFF << (packed.bits * (h % per))) & 0xFF)
    d[:, nb:] = 0xFF
    return eng.PackedCodes(torch.from_numpy(d).cuda(), h, packed.bits)


def _want(c, k):
    return torch.from_numpy(lo.counts_discrete(c, k).astype(np.int32)).cuda()


def _packed_counts(eng, packed, k):
    f = np.ones((1, k), dtype=np.float32)
    return eng.lev_sweep("discrete", f, 1.0, outcomes=packed, mode="log", want_data_T=False,
                         want_counts=True)["counts"]


def _check_counts(eng, c, k, bits=2):
    want = _want(c, k)
    codes = eng.encode_codes(c, n_outcomes=k)
    ref = eng.lev_sweep("discrete", np.ones((1, k), dtype=np.float32), 1.0, outcomes=codes, mode="log",
                        want_data_T=False, want_counts=True)["counts"]          # the uint8 kernel
    assert torch.equal(ref, want)
    packed = eng.pack_codes(codes, bits=bits)
    got = _packed_counts(eng, packed, k)
    assert torch.equal(got, want), f"H = {c.shape[1]}"
    got = _packed_counts(eng, _garbage_pad(eng, packed), k)
    assert torch.equal(got, want), f"H = {c.shape[1]}, garbage pad"


@pytest.mark.parametrize("k", [2, 3, 4])
def test_counts_at_every_short_horizon(eng, k):
    """H = 1 ... 300: every word (16 codes) and vector (64 codes) boundary of the first lanes' slots."""
    rs = np.random.RandomState(k)
    for h in range(1, 301):
        _check_counts(eng, _codes(rs, 37, h, k), k)


def test_coin_counts_at_every_short_horizon(eng):
    """One bit per flip: a word holds 32 flips, a vector 128."""
    rs = np.random.RandomState(5)
    for h in range(1, 301):
        _check_counts(eng, _codes(rs, 37, h, 2), 2, bits=1)


# 64 * 32 = 2048: one slot of vectors over the warp; 10240: the last H of one round (PACKED_U = 5 slots)
LONG = [2047, 2048, 2049, 4096 + 63, 8191, 10_000, 10_239, 10_240, 10_241, 10_240 + 64, 20_481, 70_001]


@pytest.mark.parametrize("h", LONG)
@pytest.mark.parametrize("k", [2, 3, 4])
def test_counts_at_long_horizons(eng, k, h):
    rs = np.random.RandomState(h + k)
    _check_counts(eng, _codes(rs, 67, h, k), k)


@pytest.mark.parametrize("h", [10_000, 20_481, 40_961, 70_001, 140_003])
def test_coin_counts_at_long_horizons(eng, h):
    rs = np.random.RandomState(h)
    _check_counts(eng, _codes(rs, 67, h, 2), 2, bits=1)


@pytest.mark.parametrize("k", [2, 3, 4])
def test_counts_past_two_to_the_sixteen(eng, k):
    """Rows of one code only: a count of H >= 65536 in one position of every lane's counters."""
    h = 70_001
    c = np.zeros((35, h), dtype=np.uint8)
    for r in range(c.shape[0]):
        c[r, :] = r % k
    c[3, ::7] = k - 1
    _check_counts(eng, c, k)


@pytest.mark.parametrize("k,bits", [(2, 2), (3, 2), (4, 2), (2, 1)])
@pytest.mark.parametrize("n", [2, 31, 33, 1000 + 3])
def test_tally_tuples_equal_the_uint8_kernel(eng, k, bits, n):
    """The tally sink: the count tuples the packed kernel inserts (and its `counts`) are the uint8 kernel's,
    and so are the statistics over them."""
    from rlmd_b200.tally import FinalTally

    rs = np.random.RandomState(n * 10 + k)
    h = 10_000
    c = _codes(rs, n, h, k)
    codes = eng.encode_codes(c, n_outcomes=k)
    f = (1.0 + 0.05 * rs.standard_normal((4, k))).astype(np.float32).clip(0.8, 1.2)
    out = {}
    for name, src in [("u8", codes), ("packed", _garbage_pad(eng, eng.pack_codes(codes, bits=bits)))]:
        t = FinalTally(n)
        cnt = torch.empty((n, k), dtype=torch.int32, device="cuda")
        t.add(src, k, counts=cnt)
        t.finalize()
        out[name] = (cnt, t.stats(f, 100.0, h, n_total=n, top=min(3, n - 1)))
        t.check()
    assert torch.equal(out["packed"][0], _want(c, k))
    assert torch.equal(out["packed"][0], out["u8"][0])
    a, b = out["packed"][1], out["u8"][1]
    assert torch.equal(a[:, 9:12], b[:, 9:12])
    assert torch.allclose(a, b, rtol=1e-14, atol=0, equal_nan=True)    # fp32 wealth overflows: inf / nan


@pytest.mark.parametrize("k", [2, 3, 4])
def test_unaligned_rows_and_strides(eng, k):
    """ld not a multiple of 16 and a base off 16-byte alignment: the byte path, with garbage around the codes."""
    rs = np.random.RandomState(40 + k)
    for n, h, off, extra in [(45, 10_000, 3, 7), (33, 1003, 1, 0), (37, 257, 5, 13), (64, 64, 15, 1)]:
        c = _codes(rs, n, h, k)
        nb = (h + 3) // 4
        host = np.full((n, off + nb + extra), 0xFF, dtype=np.uint8)
        host[:, off:off + nb] = lo.pack_codes(c)
        if h % 4:
            host[:, off + nb - 1] |= np.uint8((0xFF << (2 * (h % 4))) & 0xFF)
        buf = torch.from_numpy(host).cuda()
        got = _packed_counts(eng, eng.PackedCodes(buf[:, off:off + nb], h), k)
        assert torch.equal(got, _want(c, k)), (n, h, off)
