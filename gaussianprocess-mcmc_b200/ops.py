"""Torch-tensor level wrappers over the C ABI: device memory and streams come from PyTorch,
the arithmetic is libgpmc's hand-written sm_100a kernels."""
import ctypes

import numpy as np

from . import _lib
from ._lib import (KIND_SE_ISO, KIND_SE_ARD, ASM_ADD_S, ASM_LOWER_ONLY, JITTER_NONE, JITTER_PYGPS,
                   OP_POTRF, OP_LOGLIK, OP_LOGLIK_GRAD, GpmcError)


def _stream_ptr(torch):
    return ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)


def _f64_cuda(torch, a, name):
    t = torch.as_tensor(a)
    if t.dtype != torch.float64:
        t = t.to(torch.float64)
    if not t.is_cuda:
        t = t.cuda()
    if not t.is_contiguous():
        t = t.contiguous()
    return t


def kind_of(D, P):
    if P == 3:
        return KIND_SE_ISO
    if P == D + 2:
        return KIND_SE_ARD
    raise ValueError('hyp has %d columns; expected 3 (iso) or D+2=%d (ARD)' % (P, D + 2))


class Workspace(object):
    """Caller-owned device scratch, grown on demand and reused across calls."""

    def __init__(self):
        self.buf = None

    def get(self, torch, nbytes):
        if self.buf is None or self.buf.numel() < nbytes:
            self.buf = None
            self.buf = torch.empty(int(nbytes), dtype=torch.uint8, device='cuda')
        return self.buf


_default_ws = Workspace()


def cov_assemble(x, hyp, add_S=False, lower_only=False, jitter=None, out=None, ld=None):
    """Batched K (or K+S) for ``hyp[B,P]`` over inputs ``x[N,D]`` -> ``A[B,N,ld]`` (device tensor).

    Mirrors ``covK.RBF(np.log(ll), np.log(sf)).getCovMatrix(x, mode='train')`` (+ the S diagonal of
    ``aux_var_model``), ``sliceSample.py:104-105,136-137,183-190``."""
    torch = _lib.require_cuda()
    lib = _lib.load()
    x = _f64_cuda(torch, x, 'x')
    if x.dim() == 1:
        x = x.reshape(-1, 1)
    hyp = _f64_cuda(torch, hyp, 'hyp')
    if hyp.dim() == 1:
        hyp = hyp.reshape(1, -1)
    N, D = x.shape
    B, P = hyp.shape
    if ld is None:
        ld = N + (N & 1)
    if out is None:
        out = torch.empty((B, N, ld), dtype=torch.float64, device='cuda')
        if ld != N:
            out[:, :, N:] = 0.0
    jit = None if jitter is None else _f64_cuda(torch, jitter, 'jitter')
    flags = (ASM_ADD_S if add_S else 0) | (ASM_LOWER_ONLY if lower_only else 0)
    rc = lib.gpmc_cov_assemble(x.data_ptr(), N, D, hyp.data_ptr(), B, P, kind_of(D, P), flags,
                               None if jit is None else jit.data_ptr(), out.data_ptr(), ld, _stream_ptr(torch))
    _lib.check(rc, 'gpmc_cov_assemble')
    return out


def potrf_batched(A, jitter_policy=JITTER_NONE, zero_upper=True, n=None, workspace=None):
    """In-place batched lower Cholesky of ``A[B,N,ld]`` (device, FP64).  Returns ``info[B]`` (device int32).

    Mirrors ``kcGP.tools.jitchol`` (``sliceSample.py:196,205``)."""
    torch = _lib.require_cuda()
    lib = _lib.load()
    if not (A.is_cuda and A.dtype == torch.float64 and A.is_contiguous() and A.dim() == 3):
        raise ValueError('A must be a contiguous CUDA float64 tensor [B, N, ld]')
    B, N, ld = A.shape
    if n is not None:
        N = n
    info = torch.empty((B,), dtype=torch.int32, device='cuda')
    need = B * 128 * 128 * 8
    if jitter_policy == JITTER_PYGPS:
        need += B * N * ld * 8 + 4 * ((B * 8 + 255) // 256 * 256) + 256
    ws = (workspace or _default_ws).get(torch, need)
    rc = lib.gpmc_potrf_batched(A.data_ptr(), N, ld, B, info.data_ptr(), jitter_policy, 1 if zero_upper else 0,
                                ws.data_ptr(), ws.numel(), _stream_ptr(torch))
    _lib.check(rc, 'gpmc_potrf_batched')
    return info


def loglik_batched(x, g, hyp, jitter_policy=JITTER_PYGPS, workspace=None, max_wave=None):
    """``loglik[b] = log N(g_b; 0, K(hyp_b) + S(hyp_b))`` for device tensors; returns ``(loglik[B], info[B])``.

    The metric's unit (``sliceSample.py:136-137,183-190,196,147``), B items in waves."""
    torch = _lib.require_cuda()
    lib = _lib.load()
    x = _f64_cuda(torch, x, 'x')
    if x.dim() == 1:
        x = x.reshape(-1, 1)
    g = _f64_cuda(torch, g, 'g')
    hyp = _f64_cuda(torch, hyp, 'hyp')
    if g.dim() == 1:
        g = g.reshape(1, -1)
    if hyp.dim() == 1:
        hyp = hyp.reshape(1, -1)
    N, D = x.shape
    B, P = hyp.shape
    if g.shape != (B, N):
        raise ValueError('g must be [B=%d, N=%d], got %s' % (B, N, tuple(g.shape)))
    out = torch.empty((B,), dtype=torch.float64, device='cuda')
    info = torch.empty((B,), dtype=torch.int32, device='cuda')
    if B == 0:
        return out, info
    wsobj = workspace or _default_ws
    need = lib.gpmc_workspace_bytes(OP_LOGLIK, N, D, B if max_wave is None else min(B, max_wave))
    have = 0 if wsobj.buf is None else wsobj.buf.numel()
    if max_wave is None and have < need:
        # growing: never ask for more than 60 % of what is free (cudaMemGetInfo is slow, so only look when growing)
        free, _ = torch.cuda.mem_get_info()
        one = lib.gpmc_workspace_bytes(OP_LOGLIK, N, D, 1)
        need = max(one, min(need, (free + have) * 6 // 10))
    ws = wsobj.get(torch, need)
    use_bytes = need if max_wave is not None else ws.numel()       # max_wave: really limit the wave (tests)
    rc = lib.gpmc_loglik_batched(x.data_ptr(), N, D, g.data_ptr(), hyp.data_ptr(), B, P, kind_of(D, P), jitter_policy,
                                 out.data_ptr(), info.data_ptr(), ws.data_ptr(), use_bytes, _stream_ptr(torch))
    _lib.check(rc, 'gpmc_loglik_batched')
    return out, info


def loglik_grad_batched(x, g, hyp, jitter_policy=JITTER_PYGPS, workspace=None, max_wave=None):
    """``log N(g_b; 0, K(hyp_b) + sn_b^2 I)`` and its gradient with respect to the natural-scale row ``hyp[b] = (ell..,
    sf, sn)``; returns ``(loglik[B], grad[B,P], info[B])`` CUDA tensors (``gpmc_loglik_grad_batched``, include/gpmc.h).

    ``max_wave`` limits the items factored at once (the workspace is sized for that many)."""
    torch = _lib.require_cuda()
    lib = _lib.load()
    x = _f64_cuda(torch, x, 'x')
    if x.dim() == 1:
        x = x.reshape(-1, 1)
    g = _f64_cuda(torch, g, 'g')
    hyp = _f64_cuda(torch, hyp, 'hyp')
    if g.dim() == 1:
        g = g.reshape(1, -1)
    if hyp.dim() == 1:
        hyp = hyp.reshape(1, -1)
    N, D = x.shape
    B, P = hyp.shape
    if g.shape != (B, N):
        raise ValueError('g must be [B=%d, N=%d], got %s' % (B, N, tuple(g.shape)))
    out = torch.empty((B,), dtype=torch.float64, device='cuda')
    grad = torch.empty((B, P), dtype=torch.float64, device='cuda')
    info = torch.empty((B,), dtype=torch.int32, device='cuda')
    if B == 0:
        return out, grad, info
    wsobj = workspace or _default_ws
    need = lib.gpmc_workspace_bytes(OP_LOGLIK_GRAD, N, D, B if max_wave is None else min(B, max_wave))
    have = 0 if wsobj.buf is None else wsobj.buf.numel()
    if max_wave is None and have < need:
        free, _ = torch.cuda.mem_get_info()
        one = lib.gpmc_workspace_bytes(OP_LOGLIK_GRAD, N, D, 1)
        need = max(one, min(need, (free + have) * 6 // 10))
    ws = wsobj.get(torch, need)
    use_bytes = need if max_wave is not None else ws.numel()
    rc = lib.gpmc_loglik_grad_batched(x.data_ptr(), N, D, g.data_ptr(), hyp.data_ptr(), B, P, kind_of(D, P), jitter_policy,
                                      out.data_ptr(), grad.data_ptr(), info.data_ptr(), ws.data_ptr(), use_bytes,
                                      _stream_ptr(torch))
    _lib.check(rc, 'gpmc_loglik_grad_batched')
    return out, grad, info


def loglik_host(x, g, hyp, jitter_policy=JITTER_PYGPS):
    """Same unit for numpy inputs through the library's own pinned staging + stream (the end-to-end call)."""
    _lib.require_cuda()
    lib = _lib.load()
    x = np.ascontiguousarray(x, dtype=np.float64)
    if x.ndim == 1:
        x = x.reshape(-1, 1)
    g = np.ascontiguousarray(np.atleast_2d(g), dtype=np.float64)
    hyp = np.ascontiguousarray(np.atleast_2d(hyp), dtype=np.float64)
    N, D = x.shape
    B, P = hyp.shape
    if g.shape[0] == 0:
        g = g.reshape(0, N)
    if g.shape != (B, N):
        raise ValueError('g must be [B=%d, N=%d], got %s' % (B, N, g.shape))
    out = np.empty(B, dtype=np.float64)
    info = np.empty(B, dtype=np.int32)
    if B == 0:
        return out, info
    rc = lib.gpmc_loglik_host(x.ctypes.data, N, D, g.ctypes.data, hyp.ctypes.data, B, P, kind_of(D, P), jitter_policy,
                              out.ctypes.data, info.ctypes.data)
    _lib.check(rc, 'gpmc_loglik_host')
    return out, info


def prior_constants(n_ell):
    """Hyper-prior shape/scale for P = n_ell + 2 (``sliceSample.py:124-125``: k = [1, 3, 3], theta = [1, 1.5, 3];
    every extra ARD length-scale reuses the length-scale entry)."""
    k = np.array([1.0] * n_ell + [3.0, 3.0])
    th = np.array([1.0] * n_ell + [1.5, 3.0])
    return k, th


class Tape(object):
    """Explicit randomness of one sweep for B chains, in the reference's draw order
    (``sliceSample.py:194,110,127,132``): ``z[B,N]`` N(0,1); ``v[B,P]``, ``u0[B]``, ``U[B,T,P]`` U(0,1)."""

    def __init__(self, z, v, u0, U):
        self.z = np.ascontiguousarray(np.atleast_2d(z), dtype=np.float64)
        self.v = np.ascontiguousarray(np.atleast_2d(v), dtype=np.float64)
        self.u0 = np.ascontiguousarray(np.atleast_1d(u0), dtype=np.float64)
        U = np.asarray(U, dtype=np.float64)
        self.U = np.ascontiguousarray(U[None] if U.ndim == 2 else U)


def sds_sweep(x, y, F, Hyp, scale, it, my=None, tape=None, seed=0, chain0=0, max_trips=64, prior_k=None,
              prior_theta=None, jitter_policy=JITTER_PYGPS, workspace=None, chains_per_wave=None):
    """One surrogate-data slice-sampling transition for every chain (``sliceSample.py:76-163``), in place.

    ``F[B,N]`` and ``Hyp[B,P]`` are CUDA float64 tensors holding the chains' current ``(f, theta)``; on return
    they hold the accepted ``(f', theta')``.  Returns ``(ntrips[B], loglik[B], status[B])`` device tensors."""
    torch = _lib.require_cuda()
    lib = _lib.load()
    x = _f64_cuda(torch, x, 'x')
    if x.dim() == 1:
        x = x.reshape(-1, 1)
    N, D = x.shape
    if not (F.is_cuda and F.dtype == torch.float64 and F.is_contiguous() and F.dim() == 2 and F.shape[1] == N):
        raise ValueError('F must be a contiguous CUDA float64 tensor [B, N]')
    if not (Hyp.is_cuda and Hyp.dtype == torch.float64 and Hyp.is_contiguous() and Hyp.dim() == 2):
        raise ValueError('Hyp must be a contiguous CUDA float64 tensor [B, P]')
    B, P = Hyp.shape
    if F.shape[0] != B:
        raise ValueError('F and Hyp disagree on the number of chains')
    kind = kind_of(D, P)
    if my is None:
        my = float(np.mean(np.asarray(y.cpu() if hasattr(y, 'cpu') else y, dtype=np.float64)))      # sliceSample.py:102
    y = _f64_cuda(torch, y, 'y').reshape(-1)
    k, th = prior_constants(P - 2)
    k = _f64_cuda(torch, k if prior_k is None else prior_k, 'prior_k')
    th = _f64_cuda(torch, th if prior_theta is None else prior_theta, 'prior_theta')
    scale = _f64_cuda(torch, scale, 'scale').reshape(-1)
    if scale.numel() != P:
        raise ValueError('scale must have P=%d entries' % P)
    ntrips = torch.zeros((B,), dtype=torch.int32, device='cuda')
    loglik = torch.empty((B,), dtype=torch.float64, device='cuda')
    status = torch.zeros((B,), dtype=torch.int32, device='cuda')
    if B == 0:
        return ntrips, loglik, status
    tz = tv = tu = tU = None
    ttrips = 0
    if tape is not None:
        if tape.z.shape != (B, N) or tape.v.shape != (B, P) or tape.u0.shape != (B,) or tape.U.shape[0] != B or tape.U.shape[2] != P:
            raise ValueError('tape shapes do not match B=%d N=%d P=%d' % (B, N, P))
        tz, tv, tu, tU = (torch.tensor(a).cuda() for a in (tape.z, tape.v, tape.u0, tape.U))
        ttrips = tape.U.shape[1]
    wsobj = workspace or _default_ws
    have = 0 if wsobj.buf is None else wsobj.buf.numel()
    explicit_wave = chains_per_wave is not None
    if chains_per_wave is None:
        chains_per_wave = B
        if lib.gpmc_sds_workspace_bytes(N, P, B) > have:
            free, _ = torch.cuda.mem_get_info()
            budget = (free + have) * 6 // 10
            while chains_per_wave > 1 and lib.gpmc_sds_workspace_bytes(N, P, chains_per_wave) > max(budget, have):
                chains_per_wave = (chains_per_wave + 1) // 2
    need = lib.gpmc_sds_workspace_bytes(N, P, min(B, chains_per_wave))
    ws = wsobj.get(torch, need)
    # the library sizes its waves from ws_bytes: an explicit chains_per_wave must really limit the wave even when the
    # shared workspace is already larger
    ws_bytes = need if explicit_wave else ws.numel()
    ptr = lambda t: None if t is None else t.data_ptr()
    rc = lib.gpmc_sds_sweep(x.data_ptr(), y.data_ptr(), N, D, F.data_ptr(), Hyp.data_ptr(), B, P, kind,
                            scale.data_ptr(), k.data_ptr(), th.data_ptr(), int(it),
                            my, 0.0 - my, 100.0 - my, int(seed), int(chain0),
                            ptr(tz), ptr(tv), ptr(tu), ptr(tU), ttrips, int(max_trips), jitter_policy,
                            ntrips.data_ptr(), loglik.data_ptr(), status.data_ptr(),
                            ws.data_ptr(), ws_bytes, _stream_ptr(torch))
    _lib.check(rc, 'gpmc_sds_sweep')
    return ntrips, loglik, status


def sds_run(x, y, F, Hyp, scale, it0, n_iters, my=None, seed=0, chain0=0, max_trips=64, prior_k=None, prior_theta=None,
            jitter_policy=JITTER_PYGPS, workspace=None, chains_per_wave=None, keep_f_every=0):
    """``n_iters`` surrogate-data slice-sampling transitions per chain in ONE call (``gpmc_sds_run``): the caller loop of
    ``framework.py:68-75`` for every chain, each chain advancing on its own inside the resident device loop.

    ``F[B,N]`` / ``Hyp[B,P]`` hold the state on entry and the final state on return.  Returns device tensors
    ``(hist_hyp[B, n_iters, P], hist_loglik[B, n_iters], hist_trips[B, n_iters], hist_f[B, n_keep, N] or None, n_exhausted)``.
    Results are those of ``n_iters`` calls of :func:`sds_sweep` with ``it = it0 .. it0 + n_iters - 1`` bit for bit."""
    torch = _lib.require_cuda()
    lib = _lib.load()
    x = _f64_cuda(torch, x, 'x')
    if x.dim() == 1:
        x = x.reshape(-1, 1)
    N, D = x.shape
    if not (F.is_cuda and F.dtype == torch.float64 and F.is_contiguous() and F.dim() == 2 and F.shape[1] == N):
        raise ValueError('F must be a contiguous CUDA float64 tensor [B, N]')
    if not (Hyp.is_cuda and Hyp.dtype == torch.float64 and Hyp.is_contiguous() and Hyp.dim() == 2):
        raise ValueError('Hyp must be a contiguous CUDA float64 tensor [B, P]')
    B, P = Hyp.shape
    kind = kind_of(D, P)
    if my is None:
        my = float(np.mean(np.asarray(y.cpu() if hasattr(y, 'cpu') else y, dtype=np.float64)))
    y = _f64_cuda(torch, y, 'y').reshape(-1)
    k, th = prior_constants(P - 2)
    k = _f64_cuda(torch, k if prior_k is None else prior_k, 'prior_k')
    th = _f64_cuda(torch, th if prior_theta is None else prior_theta, 'prior_theta')
    scale = _f64_cuda(torch, scale, 'scale').reshape(-1)
    n_iters = int(n_iters)
    hist_hyp = torch.zeros((B, n_iters, P), dtype=torch.float64, device='cuda')
    hist_ll = torch.zeros((B, n_iters), dtype=torch.float64, device='cuda')
    hist_trips = torch.zeros((B, n_iters), dtype=torch.int32, device='cuda')
    n_keep = (n_iters + keep_f_every - 1) // keep_f_every if keep_f_every else 0
    hist_f = torch.zeros((B, n_keep, N), dtype=torch.float64, device='cuda') if n_keep else None
    n_exh = torch.zeros((1,), dtype=torch.int32, device='cuda')
    if B == 0 or n_iters == 0:
        return hist_hyp, hist_ll, hist_trips, hist_f, 0
    wsobj = workspace or _default_ws
    have = 0 if wsobj.buf is None else wsobj.buf.numel()
    explicit_wave = chains_per_wave is not None
    if chains_per_wave is None:
        chains_per_wave = B
        if lib.gpmc_sds_workspace_bytes(N, P, B) > have:
            free, _ = torch.cuda.mem_get_info()
            budget = (free + have) * 6 // 10
            while chains_per_wave > 1 and lib.gpmc_sds_workspace_bytes(N, P, chains_per_wave) > max(budget, have):
                chains_per_wave = (chains_per_wave + 1) // 2
    need = lib.gpmc_sds_workspace_bytes(N, P, min(B, chains_per_wave))
    ws = wsobj.get(torch, need)
    ws_bytes = need if explicit_wave else ws.numel()
    rc = lib.gpmc_sds_run(x.data_ptr(), y.data_ptr(), N, D, F.data_ptr(), Hyp.data_ptr(), B, P, kind,
                          scale.data_ptr(), k.data_ptr(), th.data_ptr(), int(it0), n_iters, my, 0.0 - my, 100.0 - my,
                          int(seed), int(chain0), int(max_trips), jitter_policy,
                          hist_hyp.data_ptr(), hist_ll.data_ptr(), hist_trips.data_ptr(),
                          None if hist_f is None else hist_f.data_ptr(), int(keep_f_every), int(n_keep),
                          n_exh.data_ptr(), ws.data_ptr(), ws_bytes, _stream_ptr(torch))
    _lib.check(rc, 'gpmc_sds_run')
    return hist_hyp, hist_ll, hist_trips, hist_f, int(n_exh.item())


def _pad_matrix(torch, A, ld):
    """Copy a host/device [N, N] matrix into a zero-padded CUDA [N, ld] buffer."""
    A = _f64_cuda(torch, A, 'A')
    N = A.shape[0]
    out = torch.zeros((N, ld), dtype=torch.float64, device='cuda')
    out[:, :A.shape[1]] = A
    return out


def aux_var_model_device(K, Sdiag, g):
    """L = chol(K+S), m = R S^-1 g, C = chol(R + 1e-11 I) for one caller-supplied K (``sliceSample.py:196-205``).

    Returns device tensors ``(L[N,N], m[N], C[N,N], info[2])``; no jitter retry (see kcMCMC.sliceSample.aux_var_model)."""
    torch = _lib.require_cuda()
    lib = _lib.load()
    N = int(K.shape[0])
    ld = (N + 15) // 16 * 16
    Kp = _pad_matrix(torch, K, ld)
    Sv = torch.zeros((ld,), dtype=torch.float64, device='cuda')
    Sv[:N] = _f64_cuda(torch, Sdiag, 'S').reshape(-1)
    gv = torch.zeros((ld,), dtype=torch.float64, device='cuda')
    gv[:N] = _f64_cuda(torch, g, 'g').reshape(-1)
    L = torch.zeros((N, ld), dtype=torch.float64, device='cuda')
    C = torch.zeros((N, ld), dtype=torch.float64, device='cuda')
    m = torch.zeros((ld,), dtype=torch.float64, device='cuda')
    info = torch.zeros((2,), dtype=torch.int32, device='cuda')
    ws = _default_ws.get(torch, lib.gpmc_aux_workspace_bytes(N))
    rc = lib.gpmc_aux_var_model(Kp.data_ptr(), N, ld, Sv.data_ptr(), gv.data_ptr(), L.data_ptr(), m.data_ptr(), C.data_ptr(),
                                info.data_ptr(), ws.data_ptr(), ws.numel(), _stream_ptr(torch))
    _lib.check(rc, 'gpmc_aux_var_model')
    return L[:, :N], m[:N], C[:, :N], info


def trsv_lower(L, rhs, want_lognormal=False):
    """Solve ``L x = b`` for every row ``b`` of ``rhs[B, N]`` with ONE lower-triangular ``L[N, N]`` (device tensors out)."""
    torch = _lib.require_cuda()
    lib = _lib.load()
    N = int(L.shape[0])
    ld = (N + 15) // 16 * 16
    Lp = _pad_matrix(torch, L, ld)
    rhs = _f64_cuda(torch, rhs, 'rhs')
    if rhs.dim() == 1:
        rhs = rhs.reshape(1, -1)
    B = rhs.shape[0]
    R = torch.zeros((B, ld), dtype=torch.float64, device='cuda')
    R[:, :N] = rhs
    out = torch.empty((B, ld), dtype=torch.float64, device='cuda')
    quad = torch.empty((B,), dtype=torch.float64, device='cuda') if want_lognormal else None
    rc = lib.gpmc_trsv_lower_batched(Lp.data_ptr(), N, ld, 0, R.data_ptr(), ld, B, out.data_ptr(),
                                     None if quad is None else quad.data_ptr(), _stream_ptr(torch))
    _lib.check(rc, 'gpmc_trsv_lower_batched')
    return (out[:, :N], quad) if want_lognormal else out[:, :N]


def cov_cross(x, z, hyp):
    """``covK.RBF(...).getCovMatrix(x=x, z=z, mode='cross')`` -> device tensor ``[N, M]`` (``sliceSample.py:263``)."""
    torch = _lib.require_cuda()
    lib = _lib.load()
    x = _f64_cuda(torch, x, 'x'); z = _f64_cuda(torch, z, 'z')
    if x.dim() == 1:
        x = x.reshape(-1, 1)
    if z.dim() == 1:
        z = z.reshape(-1, 1)
    hyp = _f64_cuda(torch, hyp, 'hyp').reshape(-1)
    N, D = x.shape
    M = z.shape[0]
    out = torch.empty((N, M), dtype=torch.float64, device='cuda')
    rc = lib.gpmc_cov_cross(x.data_ptr(), N, z.data_ptr(), M, D, hyp.data_ptr(), hyp.numel(), kind_of(D, hyp.numel()),
                            out.data_ptr(), M, _stream_ptr(torch))
    _lib.check(rc, 'gpmc_cov_cross')
    return out


def tg2_loglik(y, mu, sn, lower, upper, my=0.0):
    """``likK.TruncatedGauss2(upper, lower, ...).evaluate(y=y - my, mu=mu_b)`` for every row of ``mu[B, N]``."""
    torch = _lib.require_cuda()
    lib = _lib.load()
    y = _f64_cuda(torch, y, 'y').reshape(-1)
    mu = _f64_cuda(torch, mu, 'mu')
    if mu.dim() == 1:
        mu = mu.reshape(1, -1)
    B, N = mu.shape
    sn = _f64_cuda(torch, np.broadcast_to(np.asarray(sn, dtype=np.float64), (B,)).copy(), 'sn')
    out = torch.empty((B,), dtype=torch.float64, device='cuda')
    rc = lib.gpmc_tg2_loglik(y.data_ptr(), float(my), mu.data_ptr(), N, N, B, sn.data_ptr(), float(lower), float(upper),
                             out.data_ptr(), _stream_ptr(torch))
    _lib.check(rc, 'gpmc_tg2_loglik')
    return out


def predict_batched(x, xs, fm, hyp, jitter_policy=JITTER_PYGPS, workspace=None):
    """``inf_mcmc``'s linear algebra (``sliceSample.py:256-270``) for S stored samples at once.

    ``fm[S, N]`` = ``f_s - m`` (centred latent samples), ``hyp[S, P]`` their hyper-parameters, ``xs[M, D]`` test inputs.
    Returns device tensors ``(fmu[S, M], fs2[S, M], info[S])`` with ``fmu = Ks^T alpha`` (add ``ms`` yourself) and
    ``fs2 = kss - sum V^2`` (unclamped)."""
    torch = _lib.require_cuda()
    lib = _lib.load()
    x = _f64_cuda(torch, x, 'x')
    xs = _f64_cuda(torch, xs, 'xs')
    if x.dim() == 1:
        x = x.reshape(-1, 1)
    if xs.dim() == 1:
        xs = xs.reshape(-1, 1)
    fm = _f64_cuda(torch, fm, 'fm')
    hyp = _f64_cuda(torch, hyp, 'hyp')
    if fm.dim() == 1:
        fm = fm.reshape(1, -1)
    if hyp.dim() == 1:
        hyp = hyp.reshape(1, -1)
    N, D = x.shape
    M = xs.shape[0]
    S, P = hyp.shape
    if fm.shape != (S, N) or xs.shape[1] != D:
        raise ValueError('fm must be [S=%d, N=%d] and xs [M, D=%d]' % (S, N, D))
    fmu = torch.empty((S, M), dtype=torch.float64, device='cuda')
    fs2 = torch.empty((S, M), dtype=torch.float64, device='cuda')
    info = torch.zeros((S,), dtype=torch.int32, device='cuda')
    if S == 0 or M == 0:
        return fmu, fs2, info
    ws = (workspace or _default_ws).get(torch, lib.gpmc_predict_workspace_bytes(N, M, S))
    rc = lib.gpmc_predict_batched(x.data_ptr(), N, D, xs.data_ptr(), M, fm.data_ptr(), hyp.data_ptr(), S, P, kind_of(D, P),
                                  jitter_policy, fmu.data_ptr(), fs2.data_ptr(), info.data_ptr(), ws.data_ptr(), ws.numel(),
                                  _stream_ptr(torch))
    _lib.check(rc, 'gpmc_predict_batched')
    return fmu, fs2, info


class EssTape(object):
    """Explicit randomness of one elliptical-slice update for B chains in the reference's draw order
    (``sliceSample.py:41,51,54,74``): ``nu[B,N]`` (the N(0,K) draw itself) or ``z[B,N]`` (nu = chol(K) z),
    ``u[B]`` (slice level), ``theta[B,T]`` (initial angle, then one redraw per rejected proposal), all U(0,1)/N(0,1)."""

    def __init__(self, u, theta, nu=None, z=None):
        self.u = np.ascontiguousarray(np.atleast_1d(u), dtype=np.float64)
        self.theta = np.ascontiguousarray(np.atleast_2d(theta), dtype=np.float64)
        self.nu = None if nu is None else np.ascontiguousarray(np.atleast_2d(nu), dtype=np.float64)
        self.z = None if z is None else np.ascontiguousarray(np.atleast_2d(z), dtype=np.float64)


def ess_sweep(x, y, F, Hyp, it=0, my=None, tape=None, seed=0, chain0=0, max_trips=256, jitter_policy=JITTER_PYGPS, workspace=None):
    """One elliptical-slice update of ``F[B,N]`` in place (``sliceSample.py:15-74``) for B chains with ``Hyp[B,P]``.
    Returns ``(ntrips[B], status[B], info[B])`` device tensors."""
    torch = _lib.require_cuda()
    lib = _lib.load()
    x = _f64_cuda(torch, x, 'x')
    if x.dim() == 1:
        x = x.reshape(-1, 1)
    N, D = x.shape
    if not (F.is_cuda and F.dtype == torch.float64 and F.is_contiguous() and F.dim() == 2 and F.shape[1] == N):
        raise ValueError('F must be a contiguous CUDA float64 tensor [B, N]')
    Hyp = _f64_cuda(torch, Hyp, 'Hyp')
    if Hyp.dim() == 1:
        Hyp = Hyp.reshape(1, -1)
    B, P = Hyp.shape
    if F.shape[0] != B:
        raise ValueError('F and Hyp disagree on the number of chains')
    if my is None:
        my = float(np.mean(np.asarray(y.cpu() if hasattr(y, 'cpu') else y, dtype=np.float64)))
    y = _f64_cuda(torch, y, 'y').reshape(-1)
    ntrips = torch.zeros((B,), dtype=torch.int32, device='cuda')
    status = torch.zeros((B,), dtype=torch.int32, device='cuda')
    info = torch.zeros((B,), dtype=torch.int32, device='cuda')
    if B == 0:
        return ntrips, status, info
    t_nu = t_z = t_u = t_th = None
    ttrips = 0
    if tape is not None:
        if tape.u.shape != (B,) or tape.theta.shape[0] != B:
            raise ValueError('tape shapes do not match B=%d' % B)
        t_u, t_th = torch.tensor(tape.u).cuda(), torch.tensor(tape.theta).cuda()
        ttrips = tape.theta.shape[1]
        if tape.nu is not None:
            t_nu = torch.tensor(tape.nu).cuda()
        if tape.z is not None:
            t_z = torch.tensor(tape.z).cuda()
    ws = (workspace or _default_ws).get(torch, lib.gpmc_ess_workspace_bytes(N, B))
    ptr = lambda t: None if t is None else t.data_ptr()
    rc = lib.gpmc_ess_sweep(x.data_ptr(), y.data_ptr(), N, D, F.data_ptr(), Hyp.data_ptr(), B, P, kind_of(D, P),
                            my, 0.0 - my, 100.0 - my, int(seed), int(chain0), int(it),
                            ptr(t_nu), ptr(t_z), ptr(t_u), ptr(t_th), ttrips, int(max_trips), jitter_policy,
                            ntrips.data_ptr(), status.data_ptr(), info.data_ptr(), ws.data_ptr(), ws.numel(), _stream_ptr(torch))
    _lib.check(rc, 'gpmc_ess_sweep')
    return ntrips, status, info


def set_tuning(key, value):
    _lib.check(_lib.load().gpmc_set_tuning(int(key), int(value)), 'gpmc_set_tuning')


def fp64_peak(which='dmma', iters=4096):
    _lib.require_cuda()
    lib = _lib.load()
    tf, ms = ctypes.c_double(), ctypes.c_double()
    _lib.check(lib.gpmc_bench_fp64_peak(0 if which == 'dmma' else 1, iters, ctypes.byref(tf), ctypes.byref(ms)), 'gpmc_bench_fp64_peak')
    return tf.value, ms.value


def profile(on):
    lib = _lib.load()
    lib.gpmc_profile_reset()
    lib.gpmc_profile_enable(1 if on else 0)


def profile_timeline(origin='assemble', capacity=65536):
    """{class name: float64[launches, 2]} -- (start, end) of every recorded launch in ms after the first launch of
    class ``origin`` began.  Streams of the look-ahead schedule overlap in time."""
    lib = _lib.load()
    o = _lib.KC_NAMES.index(origin)
    out = {}
    for k, name in enumerate(_lib.KC_NAMES):
        buf = np.zeros((capacity, 2))
        n = ctypes.c_longlong()
        _lib.check(lib.gpmc_profile_timeline(k, o, buf.ctypes.data_as(ctypes.POINTER(ctypes.c_double)), capacity, ctypes.byref(n)),
                   'gpmc_profile_timeline')
        out[name] = buf[:n.value].copy()
    return out


def profile_read():
    """{class name: (total_ms, launches)} of the library's own kernels since the last reset."""
    lib = _lib.load()
    out = {}
    for k, name in enumerate(_lib.KC_NAMES):
        ms, n = ctypes.c_double(), ctypes.c_longlong()
        _lib.check(lib.gpmc_profile_read(k, ctypes.byref(ms), ctypes.byref(n)), 'gpmc_profile_read')
        out[name] = (ms.value, n.value)
    return out
