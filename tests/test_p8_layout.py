"""The fused trunk's private P8 order of the fp32 residual stream (fused_forward.to_p8 / from_p8): no GPU needed."""
import pytest


@pytest.mark.parametrize("C", [96, 128])
def test_p8_round_trip(C):
    import torch
    from minesweeper_ppo_b200.fused_forward import from_p8, to_p8
    x = torch.randn(3, C, 16, 16)
    t = to_p8(x)
    assert t.shape == (3, 2, C // 32, 4, 128, 8) and t.is_contiguous()
    assert torch.equal(from_p8(t), x)
    # element (board 1, channel c, row y, column x) sits at [1][y // 8][c // 32][(c % 32) // 8][(y % 8) * 16 + x][c % 8]
    c, y, xx = C - 3, 11, 5
    assert t[1, y // 8, c // 32, (c % 32) // 8, (y % 8) * 16 + xx, c % 8] == x[1, c, y, xx]
