"""CPU: argument checks of b200_attention / b200_attention_mc above 256 tokens (the key-tiled kernel)."""
import b200_native as nat

MAX_N = 16384  # the documented token limit of b200_attention


def test_long_attention_rejects_out_of_range_arguments_without_a_gpu():
    """< 0 before anything is launched (the pointers are never read: any non-NULL value stands for a buffer)."""
    lib, p = nat.lib(), 16
    for dh, heads in ((128, 4), (64, 12)):
        E = heads * dh
        args = lambda N: (p, 3 * E, p, E, 2, N, heads, dh, dh ** -0.5)
        for N in (MAX_N + 1, 4 * MAX_N, 0, -1, -257):
            assert lib.b200_attention(*args(N), None) < 0, (dh, N)
            assert lib.b200_attention_mc(*args(N), 0.1, 1, None) < 0, (dh, N)
        for N in (257, 1024, MAX_N):
            for bad in (-0.1, 1.0, 1.5, float("nan")):
                assert lib.b200_attention_mc(*args(N), bad, 1, None) < 0, (dh, N, bad)
    # more (case, head, 128-query tile) work items than an int holds
    assert lib.b200_attention(p, 3 * 4096, p, 4096, 1 << 20, MAX_N, 32, 128, 0.1, None) < 0
