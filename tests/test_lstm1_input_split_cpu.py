"""LSTM1's operand image carries each count as two fp16 terms, x_hi = fp16(x) and x_lo = fp16(x - x_hi)
(k_xop / k_window_xop).  Counts reach 8000 (deeper columns are refused), and fp16 holds integers exactly only up to
2048, so the split must give back every such integer exactly."""
import numpy as np


def test_hi_lo_split_is_exact_for_every_count():
    x = np.arange(-8000, 8001, dtype=np.int64)
    hi = x.astype(np.float16)
    lo = (x - hi.astype(np.int64)).astype(np.float16)
    assert np.array_equal(hi.astype(np.float64) + lo.astype(np.float64), x.astype(np.float64))
    assert np.abs(lo.astype(np.float64)).max() <= 2
    # the split is needed: above 2048 one fp16 loses odd counts, above 4096 those that are not multiples of 4
    assert (hi.astype(np.int64) != x).sum() > 0 and np.all(hi.astype(np.int64)[np.abs(x) <= 2048] == x[np.abs(x) <= 2048])
