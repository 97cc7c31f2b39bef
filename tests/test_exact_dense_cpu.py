"""The exact dense scores' value rule, emulated on the host (no GPU): ``exact_dense_values`` repeats dot_f64's
order (csrc/ccr_kernels.cu) bit for bit, so the GPU tests can compare ccr_score_dense_exact against it on
view(int32).  Also the C ABI's argument checks, which return before any device work."""
import numpy as np
import pytest
import torch


def exact_dense_values(Q, P, D):
    """float32 [B, N]: the exact value of every (row of Q, row of P) pair for the kernels' D, on numpy arrays or
    torch tensors (CPU or CUDA) holding fp32 values.

    Lane l of a warp sums acc + q_e * v_e in float64 over the float4 chunks c = l, l + 32, ... < D / 4, the four
    elements of a chunk in order, from +0.0; a product of two fp32 values is exact in float64, so each step is
    the kernel's one rounded fma.  Then the xor butterfly with offsets 16 .. 1 (lane 0's value) and the
    rounding to fp32."""
    is_torch = isinstance(Q, torch.Tensor)
    if is_torch:
        Qd, Pd = Q[:, :D].double(), P[:, :D].double()
    else:
        Qd = np.asarray(Q, dtype=np.float32)[:, :D].astype(np.float64)
        Pd = np.asarray(P, dtype=np.float32)[:, :D].astype(np.float64)
    B, N = Qd.shape[0], Pd.shape[0]
    n_chunks = D // 4
    lanes = np.arange(32)
    perms = {off: torch.as_tensor(lanes ^ off, device=Qd.device) if is_torch else lanes ^ off
             for off in (16, 8, 4, 2, 1)}
    out = torch.empty((B, N), dtype=torch.float32, device=Qd.device) if is_torch else \
        np.empty((B, N), dtype=np.float32)
    step = max(1, (1 << 21) // max(N, 1))  # rows per block: [rows, N, 32] float64 <= 512 MB
    for r0 in range(0, B, step):
        q = Qd[r0 : r0 + step]
        acc = torch.zeros((q.shape[0], N, 32), dtype=torch.float64, device=Qd.device) if is_torch else \
            np.zeros((q.shape[0], N, 32))
        for t in range(-(-n_chunks // 32)):
            live = min(32, n_chunks - 32 * t)  # lanes 0 .. live-1 own a chunk in this round
            for j in range(4):
                e = (32 * t + lanes[:live]) * 4 + j
                acc[:, :, :live] = acc[:, :, :live] + q[:, None, e] * Pd[None, :, e]
        for off in (16, 8, 4, 2, 1):
            acc = acc + acc[:, :, perms[off]]
        out[r0 : r0 + step] = acc[:, :, 0].float() if is_torch else acc[:, :, 0].astype(np.float32)
    return out


def test_emulation_follows_the_lane_and_butterfly_order():
    """D = 256: 64 chunks, lane l sums chunks l and l + 32.  Ones in the query; the item holds 2^53 at element 0
    (lane 0, chunk 0), 2^29 at element 128 (lane 0, chunk 32) and 1 at element 4 l (lane l, chunk l) for
    l = 1..31.  fp32's spacing at 2^53 is 2^30, so the fp32 result turns on which side of 2^53 + 2^29 the
    float64 sum lands.
      lane tree: lane 0 = 2^53 + 2^29, lanes 1..31 = 1; butterfly 16: lane 0 (2^53 + 2^29) + 1 -> 2^53 + 2^29
        (a tie in float64, to even), lanes 1..15 2; then + 2, + 4, + 8, + 16: 2^53 + 2^29 + 30 -> fp32 2^53 + 2^30.
      sequential float64: 2^53, every + 1 a tie to even 2^53, + 2^29: exactly 2^53 + 2^29 -> fp32 tie to 2^53.
      fp32 Q @ P.T: every product exact, 2^53 absorbs each 1 and 2^29 (a tie to even): 2^53 in any order, unless
        the 1s meet first, and 31 ones reach 2^29 + 31 -> 2^29 (fp32 spacing 64 there), so 2^53 again.
    So the tree differs from both; the next test separates all three."""
    D = 256
    q = np.ones((1, D), dtype=np.float32)
    v = np.zeros((1, D), dtype=np.float32)
    v[0, 0], v[0, 128] = 2.0 ** 53, 2.0 ** 29
    v[0, 4 * np.arange(1, 32)] = 1.0
    tree = exact_dense_values(q, v, D)[0, 0]
    seq = np.float64(0.0)
    for e in range(D):
        seq = seq + np.float64(q[0, e]) * np.float64(v[0, e])
    assert tree == np.float32(2.0 ** 53 + 2.0 ** 30)
    assert np.float32(seq) == np.float32(2.0 ** 53)
    assert (q @ v.T)[0, 0] == np.float32(2.0 ** 53)
    # torch on the host follows the same order
    assert exact_dense_values(torch.as_tensor(q), torch.as_tensor(v), D)[0, 0].item() == tree


def test_emulation_tree_sequential_and_fp32_give_three_values():
    """D = 256, ones elsewhere in the query.  Element 0 (lane 0, chunk 0): (1 + 2^-12) x -(2^54 + 2^42), product
    A = -(2^54 + 2^43 + 2^30); element 128 (lane 0, chunk 32): (1 - 2^-12) x (2^53 + 2^41), product B = 2^53 - 2^29;
    1 at element 4 l (lane l) for l = 1..31.  A + B = -(2^53 + 2^43 + 3 2^29), an fp32 midpoint (spacing 2^30).
      lane tree: lane 0 = A + B exactly, the butterfly adds the 31 ones: magnitude below the midpoint
        -> -(2^53 + 2^43 + 2^30).
      sequential float64: each 1 is lost against A (float64 spacing 4), A + B is the midpoint itself, a tie to
        even -> -(2^53 + 2^43 + 2^31).
      fp32 Q @ P.T: A rounds to -(2^54 + 2^43) (a tie to even) before it is added, A + B then lands on the
        midpoint below, a tie to even -> -(2^53 + 2^43); the ones never count, in any order of the sum."""
    D = 256
    q = np.ones((1, D), dtype=np.float32)
    v = np.zeros((1, D), dtype=np.float32)
    q[0, 0], v[0, 0] = 1 + 2.0 ** -12, -(2.0 ** 54 + 2.0 ** 42)
    q[0, 128], v[0, 128] = 1 - 2.0 ** -12, 2.0 ** 53 + 2.0 ** 41
    v[0, 4 * np.arange(1, 32)] = 1.0
    tree = exact_dense_values(q, v, D)[0, 0]
    seq = np.float64(0.0)
    for e in range(D):
        seq = seq + np.float64(q[0, e]) * np.float64(v[0, e])
    plain = (q @ v.T)[0, 0]
    assert tree == np.float32(-(2.0 ** 53 + 2.0 ** 43 + 2.0 ** 30))
    assert np.float32(seq) == np.float32(-(2.0 ** 53 + 2.0 ** 43 + 2.0 ** 31))
    assert plain == np.float32(-(2.0 ** 53 + 2.0 ** 43))


def test_emulation_matches_the_float64_sum_up_to_one_rounding():
    """On random rows the emulated value is within fp32's rounding of the float64 matmul; rows past D are
    ignored (NaN there changes nothing)."""
    rs = np.random.RandomState(0)
    for D in (8, 64, 200, 768):
        Q = rs.standard_normal((5, D + 8)).astype(np.float32)
        P = rs.standard_normal((7, D + 8)).astype(np.float32)
        Q[:, D:], P[:, D:] = np.nan, np.nan
        got = exact_dense_values(Q, P, D).astype(np.float64)
        ref = Q[:, :D].astype(np.float64) @ P[:, :D].astype(np.float64).T
        assert (np.abs(got - ref) <= np.abs(ref) * 2.0 ** -23 + 1e-300).all(), D
        np.testing.assert_array_equal(exact_dense_values(torch.as_tensor(Q), torch.as_tensor(P), D).numpy(),
                                      exact_dense_values(Q, P, D))


def test_emulation_keeps_the_sign_of_zero():
    """A sum that starts at +0.0 stays +0.0 through products of -0.0 and through exact cancellation."""
    D = 64
    q = np.zeros((2, D), dtype=np.float32)
    v = np.zeros((2, D), dtype=np.float32)
    q[0, :] = -0.0
    v[0, :] = 1.0
    q[1, 0], q[1, 4] = 1.0, 1.0
    v[1, 0], v[1, 4] = 3.0, -3.0
    got = np.diag(exact_dense_values(q, v, D))
    assert (got == 0).all() and not np.signbit(got).any()


# ---- the C ABI's argument checks (no device work happens on these paths) ----

def _call(B, ldq, N, ldi, D, ld_out, q=16, items=16, out=16):
    from ccr_b200 import _lib

    return _lib.lib().ccr_score_dense_exact(q, B, ldq, items, N, ldi, D, out, ld_out, None)


def test_abi_checks_arguments():
    from ccr_b200 import _lib

    assert _lib.EXPORTS.count("ccr_score_dense_exact") == 1
    assert _call(4, 64, 8, 64, 64, 8, q=None) == _lib.EINVAL            # null pointer
    assert _call(4, 64, 8, 64, 64, 8, out=None) == _lib.EINVAL
    assert _call(4, 68, 8, 64, 64, 8) == _lib.EINVAL                    # pitch not a multiple of 8
    assert _call(4, 64, 8, 60, 56, 8) == _lib.EINVAL
    assert _call(4, 64, 8, 64, 60, 8) == _lib.EINVAL                    # D % 8 != 0
    assert _call(4, 64, 8, 64, 72, 8) == _lib.EINVAL                    # pitch < D
    assert _call(4, 64, 8, 64, 64, 7) == _lib.EINVAL                    # ld_out < N
    assert _call(4, 64, 8, 64, 64, 8, q=24) == _lib.EINVAL              # base not 16-byte aligned
    assert _call(-1, 64, 8, 64, 64, 8) == _lib.EINVAL
    assert _call(4, 4104, 8, 4104, 4104, 8) == _lib.EUNSUPPORTED        # D > 4096
    assert _call(0, 64, 8, 64, 64, 8, q=None, items=None, out=None) == _lib.OK  # empty: nothing to do
    assert _call(4, 64, 0, 64, 64, 0, q=None, items=None, out=None) == _lib.OK
