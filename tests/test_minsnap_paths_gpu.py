"""Every kernel of K1's uniform-S dispatch (uavb_minsnap_solve_f64), reached through the C ABI by where the arrays sit.

The solve picks its kernel from S and from the 16-byte alignment of `coeffs_out`, `waypoints` and `velocity`: the tensor-store
kernels need an aligned output, the streaming kernel's bulk loads aligned inputs.  Fresh tensors are always aligned, so here every
array is a view into a padded float64 buffer that starts one element (misaligned) or two elements (aligned) in.  Each row checks the
coefficients against the NumPy oracle, that nothing outside the output views was written (the tensor stores clip rows past the batch
and the copy loops stop at its end), and that a mission solved in a batch of three gives the same bits as in the batch of 130."""
import numpy as np
import pytest

from helpers import normwise

pytestmark = pytest.mark.gpu
B = 130                    # two whole 64-mission CTAs (tiles) and a ragged one of 2
PAD = 64                   # elements of padding after every view
SENTINEL = -7.25e300

# (S, coeffs_out aligned, waypoints aligned, velocity aligned): the kernel each row selects
ROWS = {
    "S1-copy1": (1, True, True, True),            # minsnap_solve_kernel<1, one spline per flush>
    "S2-copy1": (2, False, False, False),         # minsnap_solve_kernel<2, one spline per flush>
    "S3-tma": (3, True, True, True),              # minsnap_solve_kernel<4, tensor stores, 6 CTAs>
    "S3-copy2": (3, False, True, True),           # minsnap_solve_kernel<4, two splines per flush, 6 CTAs>
    "S4-stream": (4, True, True, True),           # minsnap_solve_stream_kernel<4, 4>
    "S4-tma-wp": (4, True, False, True),          # one-shot tensor stores: the waypoints cannot be bulk-loaded
    "S4-tma-vel": (4, True, True, False),         # ... nor the velocities
    "S4-copy2": (4, False, True, True),
    "S5-tma": (5, True, True, True),              # minsnap_solve_kernel<8, tensor stores>
    "S5-copy1": (5, False, True, True),           # minsnap_solve_kernel<8, one spline per flush>
    "S8-tma": (8, True, False, False),
    "S8-copy1": (8, False, False, False),
    "S9-direct": (9, False, False, False),        # minsnap_solve_kernel<64, per-thread stores>
    "S12-direct": (12, True, True, True),
}


def _padded(n, aligned, dev):
    """A view of n elements into a sentinel-filled buffer, 16-byte aligned or 8 bytes off; the buffer and the view's offset in it."""
    import torch
    off = 2 if aligned else 1
    buf = torch.full((off + n + PAD,), SENTINEL, dtype=torch.float64, device=dev)
    view = buf[off:off + n]
    assert (view.data_ptr() % 16 == 0) == aligned
    return view, buf, off


def _solve(dev, wp, vel, S, c_al, w_al, v_al):
    import torch
    from uav_ac_b200 import _native as nat, kernels
    nb = wp.shape[0]
    w_view = _padded(wp.numel(), w_al, dev)[0]
    w_view.copy_(wp.reshape(-1))
    v_view = _padded(nb, v_al, dev)[0]
    v_view.copy_(vel)
    c_view, c_buf, c_off = _padded(nb * 24 * S, c_al, dev)
    t_view, t_buf, t_off = _padded(nb * S, True, dev)
    status = torch.full((nb,), -1, dtype=torch.int32, device=dev)
    nat.on(dev).uavb_minsnap_solve_f64(nat.ptr(w_view), nat.ptr(v_view), nb, S, float(kernels.START_END_TIME_FACTOR), nat.ptr(c_view),
                                       nat.ptr(t_view), nat.ptr(status), nat.stream_ptr(dev))
    torch.cuda.synchronize()
    c_buf, t_buf = c_buf.cpu().numpy(), t_buf.cpu().numpy()
    outside = np.concatenate([c_buf[:c_off], c_buf[c_off + c_view.numel():], t_buf[:t_off], t_buf[t_off + t_view.numel():]])
    assert (outside == SENTINEL).all(), f"{int((outside != SENTINEL).sum())} elements written outside the output views"
    return c_view.cpu().numpy().reshape(nb, 8 * S, 3), t_view.cpu().numpy().reshape(nb, S), status.cpu().numpy()


@pytest.mark.parametrize("row", list(ROWS))
def test_every_dispatch_row_matches_oracle_and_stays_in_bounds(cuda, row):
    from oracle import minsnap_np
    from uav_ac_b200 import kernels
    S, c_al, w_al, v_al = ROWS[row]
    wp, vel = kernels.mc_missions(7 + S, B, S, device=cuda)
    c, t, s = _solve(cuda, wp, vel, S, c_al, w_al, v_al)
    assert (s == 0).all()
    wp_h, vel_h = wp.cpu().numpy(), vel.cpu().numpy()
    for b in range(B):
        ref_c, ref_t = minsnap_np.solve_coeffs(wp_h[b], float(vel_h[b]), "solve")
        assert normwise(c[b], ref_c) < 1e-9, (b, normwise(c[b], ref_c))
        np.testing.assert_allclose(t[b], ref_t, rtol=1e-15, atol=0)
    for lo, hi in ((0, 3), (B - 3, B)):                 # the first CTA's head, the tail across the last whole tile and the ragged one
        c_sub, t_sub, s_sub = _solve(cuda, wp[lo:hi], vel[lo:hi], S, c_al, w_al, v_al)
        assert (s_sub == 0).all()
        assert np.array_equal(c_sub.view(np.uint64), c[lo:hi].view(np.uint64)), (lo, hi)
        assert np.array_equal(t_sub.view(np.uint64), t[lo:hi].view(np.uint64)), (lo, hi)
