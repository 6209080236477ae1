"""CPU: the bit-exact restatement of the bf16-storage ingest (oracle.np_centre / np_bf16_rows) against float64 and
against its own invariants.  tests/test_gpu_ingest_exact.py holds the device to this restatement bit for bit."""
import numpy as np

import oracle as orc


def _ulp_err(mu, ref):
    """|mu - ref| in units of the float32 spacing at ref."""
    return np.abs(mu.astype(np.float64) - ref) / np.spacing(np.abs(ref).astype(np.float32)).astype(np.float64)


def test_centre_is_the_mean_within_a_few_ulp():
    rng = np.random.default_rng(3)
    for n, d in ((1, 5), (63, 7), (64, 3), (65, 9), (4097, 96), (70000, 16)):
        x = (rng.standard_normal((n, d)) * rng.uniform(0.1, 100, d) + rng.standard_normal(d) * 50).astype(np.float32)
        mu = orc.np_centre(x)
        m = min(n, orc.CENTRE_ROWS)
        ref = x[:m].astype(np.float64).mean(0)
        # error of the float32 block sums (64 terms) relative to the column's spread, plus the final rounding
        spread = np.abs(x[:m]).astype(np.float64).mean(0)
        assert np.all(np.abs(mu - ref) <= 64 * 2.0 ** -24 * spread + np.spacing(np.abs(ref).astype(np.float32))), (n, d)
        if n == 1:
            assert np.array_equal(mu, x[0])            # one row: the mean is the row itself
        if n <= 64:   # one block, no cancellation: the float32 sum is the only rounding before the last
            assert _ulp_err(mu, ref).max() <= 64, (n, d)


def test_centre_takes_the_first_65536_rows():
    rng = np.random.default_rng(4)
    x = rng.standard_normal((orc.CENTRE_ROWS + 300, 4)).astype(np.float32)
    x[orc.CENTRE_ROWS:] += 1000
    assert np.array_equal(orc.np_centre(x), orc.np_centre(x[:orc.CENTRE_ROWS]))
    assert np.abs(orc.np_centre(x)).max() < 0.05


def test_centre_is_exactly_power_of_two_equivariant():
    rng = np.random.default_rng(5)
    x = (rng.standard_normal((5000, 12)) + 3).astype(np.float32)
    mu = orc.np_centre(x)
    for s in (-60, -20, -1, 1, 20, 60):
        f = np.float32(2.0 ** s)
        assert np.array_equal(x * f / f, x)
        assert np.array_equal(orc.np_centre(x * f).view(np.uint32), (mu * f).view(np.uint32)), s


def _seq_sum(v):
    a = np.float32(0)
    for t in v:
        a = np.float32(a + t)
    return a


def test_centre_skips_non_finite_blocks_but_counts_their_rows():
    rng = np.random.default_rng(6)
    x = rng.standard_normal((200, 6)).astype(np.float32)   # blocks [0,64) [64,128) [128,192) [192,200)
    x[70, 0] = np.nan                                      # column 0 loses block 1
    x[5, 1] = np.inf                                       # column 1 loses block 0
    x[130, 2], x[131, 2] = np.inf, -np.inf                 # column 2 loses block 2 (inf - inf = NaN)
    x[:64, 3] = 1e37                                       # column 3: 64 x 1e37 overflows float32, block 0 is skipped
    mu = orc.np_centre(x)
    assert np.isfinite(mu).all()
    keep = {0: np.r_[0:64, 128:200], 1: np.r_[64:200], 2: np.r_[0:128, 192:200], 3: np.r_[64:200]}
    for c, rows in keep.items():
        ref = x[rows, c].astype(np.float64).sum() / 200   # the skipped rows still count in m
        assert abs(mu[c] - ref) <= 1e-6 * np.abs(x[rows, c]).sum() / 200, (c, mu[c], ref)
    assert np.array_equal(mu[4:], orc.np_centre(x[:, 4:]))
    # only non-finite blocks everywhere: the centre is 0
    assert np.array_equal(orc.np_centre(np.full((70, 3), np.nan, np.float32)), np.zeros(3, np.float32))
    # a partial last block of huge rows does not overflow: it alone is the sum
    big = np.full((70, 1), 1e37, np.float32)
    assert orc.np_centre(big)[0] == np.float32(np.float64(_seq_sum(big[64:, 0])) / 70)


def test_centre_of_zero_and_constant_columns():
    x = np.zeros((1000, 4), np.float32)
    x[:, 1] = -0.0
    x[:, 2] = np.float32(0.1)
    x[:, 3] = np.float32(2.0 ** -140)                      # subnormal constant
    mu = orc.np_centre(x)
    assert mu[0] == 0 and mu[1] == 0
    # 15 full blocks and one of 40 rows, each summed in float32 and added exactly
    s64, s40 = _seq_sum(x[:64, 2]), _seq_sum(x[:40, 2])
    assert mu[2] == np.float32((15 * np.float64(s64) + np.float64(s40)) / 1000)
    assert abs(float(mu[2]) - 0.1) <= 1e-6
    assert mu[3] == x[0, 3]


def test_bf16_rounding_matches_torch_cast():
    import torch

    rng = np.random.default_rng(7)
    u = np.concatenate([rng.integers(0, 2 ** 32, 200000, dtype=np.uint64).astype(np.uint32),
                        np.arange(0, 2 ** 17, dtype=np.uint32),                   # zero and subnormals
                        np.arange(0x7F7F0000, 0x7F800001, 7, dtype=np.uint32),   # the top binade, overflow to inf
                        (np.arange(0, 2 ** 16, dtype=np.uint32) << 16) | 0x8000])  # exact ties
    u = np.concatenate([u, u | np.uint32(0x80000000)])
    x = u.view(np.float32)
    got = orc.np_bf16_rne(x)
    ref = torch.from_numpy(x.copy()).to(torch.bfloat16).to(torch.float32).numpy()
    nan = np.isnan(x)
    assert np.array_equal(np.isnan(got), nan)
    assert np.array_equal(got[~nan].view(np.uint32), ref[~nan].view(np.uint32))


def test_bf16_rows_round_the_centred_value():
    rng = np.random.default_rng(8)
    x = (rng.standard_normal((3000, 10)) + 100).astype(np.float32)
    mu = orc.np_centre(x)
    r = orc.np_bf16_rows(x, mu)
    c = (x - mu).astype(np.float32)
    assert np.array_equal(r, (mu + orc.np_bf16_rne(c)).astype(np.float32))
    assert np.all(np.abs(r - x) <= 2.0 ** -8 * np.abs(c) + np.spacing(np.abs(x)))
    assert np.abs(r - x).max() > 0
