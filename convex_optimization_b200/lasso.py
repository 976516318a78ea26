# -*- coding: utf-8 -*-
"""Solver classes of the lasso block proximal iteration, B200 edition.

Same five class names, constructor signatures, ``run()`` signature and overridable hooks
as the reference's lasso.py (ClassLassoCPU :25, ClassLasso :173, ClassLassoR :296,
ClassLassoCB_v1 :310, ClassLassoCB_v2 :357).  What each maps to here:

* ``ClassLasso`` / ``ClassLassoR`` / ``ClassLassoCB_v2``: the whole loop of
  lasso.py:228-278 / :508-599 runs on the device in ONE persistent cooperative kernel
  (``b200l_run``); only b goes up and x / the traces come back.
* ``ClassLassoCB_v1`` and any subclass that overrides ``_mtv``/``_mv``/``debug``/
  ``err_record``/``time_record`` (or ``DEBUG=True``): the step-wise loop, two device
  mat-vecs per iteration through ``GPU_Calculation`` like the reference's
  "CPU & CUDA combined" path, hooks called every iteration.
* ``ClassLassoCPU``: the host (NumPy) solver with the reference's P-way column split.
  It is a separate entry point, never a fallback of the GPU classes.

Unlike the reference (which discards it, lasso.py:167-169), the solution is kept on the
solver as ``self.x`` (K,1) together with ``self.iters`` and ``self.stopped``.
"""
import ctypes
import random
import time

import numpy as np

from . import _lib
from .cpu_calculation import (element_proj, error_crit, fun_dd_p, fun_s12,
                              fun_s22, soft_thresholding)
from . import settings

settings.init()


class ClassLassoCPU:
    """Host solver (ref lasso.py:25-169).  ``A_block_p`` is the (BLOCK,P,N,w/P) view from
    ``cpu_calculation.A_bp_get``; the P slices are processed in-process (the reference
    forks a multiprocessing.Pool per run() and pickles the slices to it, lasso.py:101-124;
    the arithmetic and its summation structure are the same)."""

    def __init__(self, A_block_p, d_ATA, A, b, mu, BLOCK, P, ITER_MAX):
        self.A_block_p = A_block_p
        self.d_ATA = d_ATA
        self.d_ATA_rec = [np.divide(1, self.d_ATA[i]) for i in range(BLOCK)]
        self.A = A
        self.A_SHAPE = A.shape
        self.b = b
        self.mu = mu
        self.BLOCK = BLOCK
        self.P = P
        self.ITER_MAX = ITER_MAX
        self.descript = 'CPU ascend index'
        self.x = None
        self.iters = 0
        self.stopped = False

    # ---- hooks (ref lasso.py:40-68) -----------------------------------------------------
    def index_get(self, t):
        return t % self.BLOCK

    def debug(self, result_s13, x_block, x, t, m, r):
        if self.DEBUG:
            self.error = error_crit(result_s13, x_block, self.mu)
            value = 0.5 * np.sum(np.power(self.A @ x - self.b, 2)) + self.mu * np.sum(np.abs(x))
            print('Loop {:-4} block {:-2} updated, with Error {:.8f}, optimum value {:4.6f}, '
                  'Stepsize {:.6f}'.format(t, m, self.error, value, r))

    def err_record(self, err_iter, result_s13, x_block, t):
        if self.ERR_RCD:
            if not self.DEBUG:
                self.error = error_crit(result_s13, x_block, self.mu)
            err_iter[t] = self.error

    def time_record(self, time_iter, t, start):
        if self.TIME_RCD:
            time_iter[t + 1] = time.time() - start

    def rlt_display(self, SILENCE, t_elapsed, t):
        if not SILENCE:
            print('{:>20}, time used: {:.8f} s, with {:-4} loops, and block number: {:-2}.'.format(
                self.descript, t_elapsed, t + 1, self.BLOCK))

    # ---- shared by every run() ----------------------------------------------------------
    def _run_flags(self, ERR_BOUND, err_iter, time_iter, DEBUG):
        self.DEBUG = DEBUG
        self.ERR_RCD = isinstance(err_iter, np.ndarray)
        self.TIME_RCD = isinstance(time_iter, np.ndarray)
        return isinstance(ERR_BOUND, float)            # ref lasso.py:74-77

    def _block_products(self, m, s11):
        """(s13, matvec) for block m on the host: P slices of A_m^T s11 stacked, and a
        closure computing sum_p A_mp d_p (ref lasso.py:107-126)."""
        slices = self.A_block_p[m]
        s13 = np.vstack([fun_s12(slices[p], s11) for p in range(self.P)])

        def matvec(descent_D):
            parts = fun_dd_p(self.P, descent_D)
            return np.sum([fun_s22(slices[p], parts[p]) for p in range(self.P)], axis=0)
        return s13, matvec

    def _stepwise(self, ERR_BOUND, err_iter, time_iter, SILENCE, products):
        """The reference loop body (lasso.py:102-157 / :228-278) on the host with the two
        mat-vecs supplied by ``products(m, s11)``; hooks are called every iteration."""
        IS_BOUNDED = isinstance(ERR_BOUND, float)
        N, K = self.A_SHAPE
        x = np.zeros((K, 1))
        x_block = np.asarray(np.vsplit(x, self.BLOCK))
        Ax = np.zeros((self.BLOCK, N, 1))
        block_Cnt = 0
        r = np.float64(0.0)
        start = time.time()
        if self.TIME_RCD:
            time_iter[0] = 0
        t = -1
        self.stopped = False
        for t in range(self.ITER_MAX):
            m = self.index_get(t)
            s11 = np.sum(Ax, axis=0) - self.b
            s13, matvec = products(m, s11)
            rx = self.d_ATA[m] * x_block[m] - s13
            Bx = self.d_ATA_rec[m] * soft_thresholding(rx, self.mu)
            descent_D = Bx - x_block[m]
            s23 = matvec(descent_D)
            r_1 = (s11.T @ s23).item() + self.mu * (np.abs(Bx).sum() - np.abs(x_block[m]).sum())
            r_2 = (s23.T @ s23).item()
            if r_2 == 0.0:
                print('r_2 is ZERO, could not divide ZERO!')
            else:
                r = np.float64(element_proj(-r_1 / r_2, 0, 1))
            self.debug(s13, x_block[m], x, t, m, r)
            self.err_record(err_iter, s13, x_block[m], t)
            if IS_BOUNDED:
                if not (self.DEBUG & self.ERR_RCD):
                    self.error = error_crit(s13, x_block[m], self.mu)
                if self.error < ERR_BOUND:
                    block_Cnt += 1
                if self.BLOCK - 1 == m:
                    if block_Cnt == self.BLOCK:
                        self.stopped = True
                        break
                    block_Cnt = 0
            x_block[m] += r * descent_D
            Ax[m] += r * s23
            self.time_record(time_iter, t, start)
        t_elapsed = time_iter[t] if self.TIME_RCD else time.time() - start
        self.x = np.vstack(x_block)
        self.iters = t + 1
        self.rlt_display(SILENCE, t_elapsed, t)
        return t_elapsed

    def run(self, ERR_BOUND=None, err_iter=None, time_iter=None, SILENCE=False, DEBUG=False):
        self._run_flags(ERR_BOUND, err_iter, time_iter, DEBUG)
        return self._stepwise(ERR_BOUND, err_iter, time_iter, SILENCE, self._block_products)


class ClassLasso(ClassLassoCPU):
    """Device solver (ref lasso.py:173-292).  ``gpu_cal`` is a ``GPU_Calculation``."""

    # set False to force the step-wise (two mat-vecs per iteration) path
    FUSED = True

    def __init__(self, gpu_cal, d_ATA, A, b, mu, BLOCK, ITER_MAX):
        ClassLassoCPU.__init__(self, None, d_ATA, A, b, mu, BLOCK, None, ITER_MAX)
        del self.A_block_p
        del self.P
        self.gpu_cal = gpu_cal
        self.descript = 'GPU ascend index'
        self.kernel_ms = 0.0
        # the fused kernel takes diag(A^T A) from the device; a caller-supplied d_ATA that differs
        # from it (the reference lets the caller pass any, lasso.py:26-30) is uploaded per run
        self._custom_diag = d_ATA is not None and not gpu_cal.is_own_diag(d_ATA)

    # matrix.T @ vector (ref lasso.py:183-184)
    def _mtv(self, s13, m, s11):
        self.gpu_cal.mat_tMulVec_DiffSize(s13, m, s11)

    # matrix @ vector (ref lasso.py:187-188)
    def _mv(self, s23, m, descent_D):
        self.gpu_cal.matMulVec_DiffSize(s23, m, descent_D)

    def _device_products(self, m, s11):
        s13 = np.zeros((self.gpu_cal.MAT_WIDTH, 1))
        self._mtv(s13, m, s11)

        def matvec(descent_D):
            s23 = np.zeros((self.gpu_cal.MAT_HEIGHT, 1))
            self._mv(s23, m, descent_D)
            return s23
        return s13, matvec

    def _hooks_overridden(self):
        cls = type(self)
        base = {'_mtv': ClassLasso._mtv, '_mv': ClassLasso._mv,
                'debug': ClassLassoCPU.debug, 'err_record': ClassLassoCPU.err_record,
                'time_record': ClassLassoCPU.time_record}
        return any(getattr(cls, k) is not v for k, v in base.items())

    def _shared_order(self, order):
        """several GPUs: every rank must run the same block order (a randomised index_get draws
        it independently per process), so rank 0's order is broadcast"""
        if getattr(self.gpu_cal, '_world', 1) <= 1:
            return order
        import torch
        import torch.distributed as dist
        t = torch.from_numpy(order.copy())
        if dist.get_backend(self.gpu_cal._group) == "nccl":
            t = t.to(self.gpu_cal.device)
        dist.broadcast(t, src=dist.get_global_rank(self.gpu_cal._group, 0) if self.gpu_cal._group is not None else 0,
                       group=self.gpu_cal._group)
        return np.ascontiguousarray(t.cpu().numpy().astype(np.int32))

    def _fused_supported(self):
        """the fused kernel has shape limits the reference does not (a row of a block must fit a
        32 KiB tile, w <= 64 * #SM, N / #SM <= 1024 fp32 / 512 fp64 entries for the pre-transposed layout, and for the
        row-major layout N / #SM rows small enough that their buffers leave two tile slots in shared memory: on a B200
        about 1,500-5,300 rows in fp64 and 2,400-6,700 in fp32 depending on w, INTEGRATION.md section 4); shapes beyond
        them run the step-wise path on the library's mat-vec kernels instead, with a warning"""
        try:
            self.gpu_cal.run_config()
            return True
        except _lib.B200LassoError as e:
            import warnings
            warnings.warn("fused kernel not available for this shape (%s); running the step-wise device path" % e)
            return False

    def _fused(self, ERR_BOUND, err_iter, time_iter, SILENCE):
        """Whole solve in one persistent kernel (b200l_run)."""
        lib = self.gpu_cal._lib
        ctx = self.gpu_cal.ctx
        K = self.gpu_cal.MAT_WIDTH_ALL
        if tuple(self.A_SHAPE) != (self.gpu_cal.MAT_HEIGHT, K) or self.BLOCK != self.gpu_cal.Block:
            raise ValueError("A%s / BLOCK=%d do not match the GPU_Calculation (%d x %d, %d blocks)"
                             % (tuple(self.A_SHAPE), self.BLOCK, self.gpu_cal.MAT_HEIGHT, K,
                                self.gpu_cal.Block))
        bounded = isinstance(ERR_BOUND, float)
        if type(self).index_get is ClassLassoCPU.index_get:
            order = None         # the cyclic order t % BLOCK (ref lasso.py:40-41) is the kernel's own
        else:
            order = np.fromiter((self.index_get(t) for t in range(self.ITER_MAX)),
                                dtype=np.int32, count=self.ITER_MAX)
            order = self._shared_order(order)
        if self._custom_diag:
            self.gpu_cal._use_custom_diag(self.d_ATA)
        else:
            self.gpu_cal._use_own_diag()
        b = np.ascontiguousarray(self.b, dtype=np.float64).reshape(-1)
        errs = np.zeros(self.ITER_MAX) if self.ERR_RCD else None
        times = np.zeros(self.ITER_MAX) if self.TIME_RCD else None
        steps = ctypes.c_int64(0)
        stopped = ctypes.c_int32(0)
        kms = ctypes.c_double(0.0)
        x = np.empty((K, 1), np.float64)

        start = time.time()
        if self.TIME_RCD:
            time_iter[0] = 0
        _lib.check(lib.b200l_set_problem(ctx, _lib.dptr(b)))            # H2D b, x = 0, r = -b
        t_launch = time.time() - start
        _lib.check(lib.b200l_run(
            ctx, order.ctypes.data_as(ctypes.POINTER(ctypes.c_int32)) if order is not None else None, self.ITER_MAX,
            float(self.mu), float(ERR_BOUND) if bounded else -1.0,
            _lib.dptr(errs) if errs is not None else None,
            _lib.dptr(times) if times is not None else None,
            ctypes.byref(steps), ctypes.byref(stopped), ctypes.byref(kms)))
        _lib.check(lib.b200l_get_x(ctx, _lib.dptr(x)))                  # D2H x
        wall = time.time() - start

        n = int(steps.value)
        t = n - 1
        self.iters = n
        self.stopped = bool(stopped.value)
        self.kernel_ms = float(kms.value)
        self.x = x
        if self.ERR_RCD:
            err_iter[:n] = errs[:n]
            self.error = errs[n - 1] if n else 0.0
        if self.TIME_RCD:
            # time_iter[t+1] is written at the end of every completed iteration
            # (ref lasso.py:60-62,157); the breaking iteration does not get one
            done = n - 1 if self.stopped else n
            time_iter[1:done + 1] = t_launch + times[:done]
            t_elapsed = time_iter[t]                                     # ref lasso.py:161-162
        else:
            t_elapsed = wall
        self.rlt_display(SILENCE, t_elapsed, t)
        return t_elapsed

    def run(self, ERR_BOUND=None, err_iter=None, time_iter=None, SILENCE=False, DEBUG=False):
        self._run_flags(ERR_BOUND, err_iter, time_iter, DEBUG)
        if self.FUSED and not DEBUG and not self._hooks_overridden() and self._fused_supported():
            return self._fused(ERR_BOUND, err_iter, time_iter, SILENCE)
        return self._stepwise(ERR_BOUND, err_iter, time_iter, SILENCE, self._device_products)


class ClassLassoR(ClassLasso):
    """Random block order, reshuffled every BLOCK iterations (ref lasso.py:296-306)."""

    def __init__(self, gpu_cal, d_ATA, A, b, mu, BLOCK, ITER_MAX):
        ClassLasso.__init__(self, gpu_cal, d_ATA, A, b, mu, BLOCK, ITER_MAX)
        self.idx_shuffle = np.arange(self.BLOCK)
        self.descript = 'GPU random index'

    def index_get(self, t):
        if t % self.BLOCK == 0:
            random.shuffle(self.idx_shuffle)
        return self.idx_shuffle[t % self.BLOCK]


class ClassLassoCB_v1(ClassLasso):
    """Host loop + device mat-vecs (the reference's "Cublas CPU combined", lasso.py:310-353).
    ``h`` is the cuBLAS handle of the reference signature; it is stored and unused: the
    two GEMVs (cublasDgemv 'N' / 'T', lasso.py:336,342) are the library's own kernels."""

    def __init__(self, h, gpu_cal, d_ATA, A, b, mu, BLOCK, ITER_MAX):
        ClassLasso.__init__(self, gpu_cal, d_ATA, A, b, mu, BLOCK, ITER_MAX)
        self.descript = 'Cublas CPU combined'
        self.h = h
        self.idx_m = self.gpu_cal.MAT_HEIGHT
        self.idx_n = self.gpu_cal.MAT_WIDTH

    # The reference overrides the two mat-vecs with cublasDgemv on device vectors (lasso.py:334-344).
    # Here they are the same library mat-vecs as the parent's; the overrides exist so that
    # _hooks_overridden() routes this class to the step-wise "host loop + device mat-vecs" path,
    # which is what "Cublas CPU combined" is.
    def _mtv(self, result_s13, m, result_s11):
        self.gpu_cal.mat_tMulVec_DiffSize(result_s13, m, result_s11)

    def _mv(self, result_s23, m, descent_D):
        self.gpu_cal.matMulVec_DiffSize(result_s23, m, descent_D)


class ClassLassoCB_v2(ClassLasso):
    """Everything on the device (the reference's "Pure Cublas", lasso.py:357-613, ~15+BLOCK
    library launches and 4 scalar read-backs per iteration) -- here the fused kernel.
    The reference left the stop test commented out in this class (lasso.py:578-591);
    here ``ERR_BOUND`` is honoured."""

    def __init__(self, h, gpu_cal, d_ATA, A, b, mu, BLOCK, ITER_MAX):
        ClassLasso.__init__(self, gpu_cal, d_ATA, A, b, mu, BLOCK, ITER_MAX)
        self.descript = 'Pure Cublas'
        self.h = h
        self.idx_m = self.gpu_cal.MAT_HEIGHT
        self.idx_n = self.gpu_cal.MAT_WIDTH

    def run(self, ERR_BOUND=None, err_iter=None, time_iter=None, SILENCE=False, DEBUG=False):
        self._run_flags(ERR_BOUND, err_iter, time_iter, False)
        if not self._fused_supported():
            return self._stepwise(ERR_BOUND, err_iter, time_iter, SILENCE, self._device_products)
        return self._fused(ERR_BOUND, err_iter, time_iter, SILENCE)
