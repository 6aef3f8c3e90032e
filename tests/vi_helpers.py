"""What the GPU tests of the inertial step, the window solve, the marginalisation and the slide share: guarded device copies, a small
pose rotation, the inertial-only batch, one window's inertial factors, the bytes of an array, and viml_solve_vi on device pointers."""
import ctypes as C

import numpy as np

import inertial_oracle as io


class Guarded:
    """A device copy of a host array with GUARD bytes of a fixed pattern on either side: after a call, check() reads the whole
    allocation back, fails if a byte outside the array changed (a write out of bounds by the kernels of the call), and returns the
    array."""
    GUARD = 4096

    def __init__(self, ctx, a):
        self.ctx, self.a = ctx, np.ascontiguousarray(a)
        self.n = self.a.nbytes
        self.img = np.concatenate([np.full(self.GUARD, 0xA5, np.uint8), self.a.view(np.uint8).reshape(-1),
                                   np.full(self.GUARD, 0x5A, np.uint8)])
        self.base = ctx.to_device(self.img)
        self.ptr = self.base + self.GUARD

    def check(self):
        back = np.empty_like(self.img)
        self.ctx.d2h(back, self.base)
        self.ctx.sync()
        assert np.all(back[:self.GUARD] == 0xA5) and np.all(back[self.GUARD + self.n:] == 0x5A), "write outside the buffer"
        return back[self.GUARD:self.GUARD + self.n].view(self.a.dtype).reshape(self.a.shape)

    def free(self):
        self.ctx.device_free(self.base)


def guard_all(ctx, arrays):
    """A Guarded copy of every array of the dict (None stays None)."""
    return {k: (None if a is None else Guarded(ctx, a)) for k, a in arrays.items()}


def rotate(x, th):
    """The pose x (position, then quaternion x, y, z, w) turned by the small rotation th in its own frame."""
    q = io.qmul(io.quat(x), (1.0, th[0] / 2, th[1] / 2, th[2] / 2))
    n = np.sqrt(sum(c * c for c in q))
    return np.array([x[0], x[1], x[2], q[1] / n, q[2] / n, q[3] / n, q[0] / n])


def inertial_only(pkg, batch):
    """The batch's state without its point and line factors."""
    W = batch.W
    return pkg._abi.Batch(batch.poses, batch.ex_pose, batch.inv_depth, np.zeros(W + 1, dtype=np.int32),
                          np.zeros(0, dtype=np.uint32), np.zeros((0, 4)))


def slice_vi(pkg, vi, w):
    """The inertial factors of window w alone."""
    k0, k1 = int(vi.imu_window_offset[w]), int(vi.imu_window_offset[w + 1])
    return pkg._abi.Inertial(1, vi.P, vi.X, vi.gravity, np.array([0, k1 - k0]), vi.imu_pose[k0:k1], vi.imu_sb[k0:k1],
                             vi.imu_preint[k0:k1], vi.imu_jacobian[k0:k1], vi.imu_sqrt_info[k0:k1], vi.prior_n[w:w + 1],
                             vi.prior_jacobian[w:w + 1], vi.prior_residual[w:w + 1], vi.prior_n_blocks[w:w + 1],
                             vi.prior_block[w:w + 1], vi.prior_x0[w:w + 1])


def bits(a):
    """The bytes of an array: equal bytes are equal values, NaNs and signed zeros included."""
    return np.ascontiguousarray(a).view(np.uint8)


def device_structs(ctx, batch, vi, extra):
    """Guarded device copies of the batch's and vi's arrays and of extra: (the host inputs, their guards, the batch and inertial
    structs over the copies)."""
    b_in = {k: a for k, a in batch.arrays().items() if a is not None}
    ins = {**{"b_" + k: a for k, a in b_in.items()}, **{"v_" + k: a for k, a in vi.arrays().items()}, "extra": extra}
    gi = guard_all(ctx, ins)
    s = batch.struct({**batch.arrays(), **{k: gi["b_" + k].ptr for k in b_in}})
    v = vi.struct({k: gi["v_" + k].ptr for k in vi.arrays()})
    return ins, gi, s, v


def solve_device(pkg, ctx, batch, vi, extra, opt, flags):
    """viml_solve_vi with VIML_PTRS_DEVICE | flags on guarded device copies of every input and output; the inputs must come back
    unchanged."""
    ins, gi, s, v = device_structs(ctx, batch, vi, extra)
    W, M = batch.W, opt.max_iterations
    outs = {"poses": np.full_like(batch.poses, np.nan), "ex_pose": np.full_like(batch.ex_pose, np.nan),
            "inv_depth": np.full_like(batch.inv_depth, np.nan), "extra": np.full((W, vi.X), np.nan),
            "status": np.full(W, -1, np.int32), "iterations": np.full(W, -1, np.int32), "accepted": np.full(W, -1, np.int32),
            "cost": np.full((W, 2), np.nan), "radius": np.full(W, np.nan), "trace": np.full((W, M, 4), -1.0)}
    go = guard_all(ctx, outs)
    o = pkg._abi.SolveOut()
    for k in outs:
        setattr(o, k, go[k].ptr)
    so = ctx.solve_options(**vars(opt))
    ctx._check(ctx.lib.viml_solve_vi(ctx.h, C.byref(s), C.byref(v), gi["extra"].ptr, C.byref(so), C.byref(o), flags | pkg.PTRS_DEVICE))
    ctx.sync()
    res = {k: g.check() for k, g in go.items()}
    for k, g in gi.items():
        assert np.array_equal(bits(g.check()), bits(ins[k])), k
    for g in list(gi.values()) + list(go.values()):
        g.free()
    return res
