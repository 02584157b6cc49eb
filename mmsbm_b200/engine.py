"""Device-resident EM engine: the host-side owner of the buffers the sm_100a kernels
work on.  PyTorch is used for plumbing only (device memory, streams, and -- in
parallel.py -- torch.distributed); every computation is a call into
libmmsbm_b200.so through the device-pointer C ABI (include/mmsbm_b200.h).

One ``Engine`` = one encoded training set on one GPU + the parameters of S runs
(``sampling``) in the padded device layout theta [S][U][ldk], eta [S][I][ldl],
pr [S][K][L][R].  It stands where the reference keeps ``train`` plus the per-run
numpy arrays of ``run_one_sampling`` (src/mmsbm.py:187-269).
"""
import numpy as np
import torch

from . import _lib



class Engine:
    def __init__(self, data, n_users, n_items, n_levels, K, L, device=None):
        """``data``: int [N,3] encoded (user, item, rating) rows (numpy, host)."""
        self.lib = _lib.load(require_device=True)
        if not torch.cuda.is_available():
            raise ImportError("mmsbm_b200: torch sees no CUDA device; there is no CPU fallback")
        self.device = torch.device("cuda", torch.cuda.current_device()) if device is None \
            else torch.device(device)
        data = np.asarray(data)
        if data.ndim != 2 or data.shape[1] != 3:
            raise ValueError("data must have shape [N,3]")
        self.N = int(data.shape[0])
        self.U, self.I, self.R, self.K, self.L = int(n_users), int(n_items), int(n_levels), int(K), int(L)
        self.ldk, self.ldl = self.lib.mmsbm_row_stride(self.K), self.lib.mmsbm_row_stride(self.L)
        self.S = 0
        self.theta = self.eta = self.pr = None
        self._alt = None
        self._ws = None
        with torch.cuda.device(self.device):
            # the int64 [N,3] rows go up as they are; the int32 split and the id range check
            # run on the device (mmsbm_split_triples)
            raw = torch.from_numpy(np.ascontiguousarray(data, dtype=np.int64)).to(self.device)
            self.cols = torch.empty((3, max(self.N, 1)), dtype=torch.int32, device=self.device)
            bad = torch.zeros(1, dtype=torch.int32, device=self.device)
            _lib.check(self.lib.mmsbm_split_triples(
                raw.data_ptr(), self.N, self.U, self.I, self.R, self.cols[0].data_ptr(),
                self.cols[1].data_ptr(), self.cols[2].data_ptr(), bad.data_ptr(), self._stream()),
                "split_triples")
            if int(bad.item()):
                raise ValueError("data holds an id outside [0,U) x [0,I) x [0,R)")
            del raw
            self._build_graph()

    @classmethod
    def for_prediction(cls, n_users, n_items, n_levels, K, L, device=None):
        """An engine without a training set: holds parameters (``set_params``) and serves
        ``prod_dist_device`` / ``mean_over_runs`` -- what a model restored by ``MMSBM.load``
        needs for ``predict``.  ``run`` / ``likelihood`` need the ratings and refuse."""
        self = cls.__new__(cls)
        self.lib = _lib.load(require_device=True)
        if not torch.cuda.is_available():
            raise ImportError("mmsbm_b200: torch sees no CUDA device; there is no CPU fallback")
        self.device = torch.device("cuda", torch.cuda.current_device()) if device is None \
            else torch.device(device)
        self.N = 0
        self.U, self.I, self.R, self.K, self.L = int(n_users), int(n_items), int(n_levels), int(K), int(L)
        self.ldk, self.ldl = self.lib.mmsbm_row_stride(self.K), self.lib.mmsbm_row_stride(self.L)
        self.S = 0
        self.theta = self.eta = self.pr = None
        self._alt = None
        self._ws = None
        self.cols = None
        self.useg = None                          # no index structure
        return self

    def _need_ratings(self):
        if getattr(self, "useg", None) is None:
            raise RuntimeError("this engine holds parameters only (restored model): "
                               "fit again to iterate or to compute a likelihood")

    # ------------------------------------------------------------------ plumbing
    def _stream(self):
        return torch.cuda.current_stream(self.device).cuda_stream

    def _empty(self, n, dtype):
        return torch.empty(max(int(n), 1), dtype=dtype, device=self.device)

    def _bytes(self, n):
        return torch.empty(max(int(n), 16), dtype=torch.uint8, device=self.device)

    def _build_graph(self):
        i32 = torch.int32
        N, U, I, R = self.N, self.U, self.I, self.R
        self.useg, self.uadj, self.uperm, self.udeg = (
            self._empty(U * R + 1, i32), self._empty(N, i32), self._empty(N, i32), self._empty(U, i32))
        self.iseg, self.iadj, self.iperm, self.ideg = (
            self._empty(I * R + 1, i32), self._empty(N, i32), self._empty(N, i32), self._empty(I, i32))
        n_u, n_i = _lib.C.c_int64(0), _lib.C.c_int64(0)
        _lib.check(self.lib.mmsbm_sched_elems(N, U, _lib.C.byref(n_u)), "sched_elems")
        _lib.check(self.lib.mmsbm_sched_elems(N, I, _lib.C.byref(n_i)), "sched_elems")
        self.usched, self.isched = self._empty(n_u.value, i32), self._empty(n_i.value, i32)
        need = _lib.C.c_size_t(0)
        _lib.check(self.lib.mmsbm_graph_workspace_bytes(N, U, I, R, _lib.C.byref(need)), "graph_workspace_bytes")
        ws = self._bytes(need.value)
        _lib.check(self.lib.mmsbm_graph_build(
            self.cols[0].data_ptr(), self.cols[1].data_ptr(), self.cols[2].data_ptr(), N, U, I, R,
            self.useg.data_ptr(), self.uadj.data_ptr(), self.uperm.data_ptr(), self.udeg.data_ptr(),
            self.iseg.data_ptr(), self.iadj.data_ptr(), self.iperm.data_ptr(), self.ideg.data_ptr(),
            self.usched.data_ptr(), self.isched.data_ptr(),
            ws.data_ptr(), need.value, self._stream()), "graph_build")
        torch.cuda.current_stream(self.device).synchronize()   # ws is released on return
        del ws
        self.cols = None            # the int32 columns are only an input of the build

    def _graph_args(self):
        return (self.useg.data_ptr(), self.uadj.data_ptr(), self.udeg.data_ptr(),
                self.iseg.data_ptr(), self.iadj.data_ptr(), self.ideg.data_ptr(),
                self.usched.data_ptr(), self.isched.data_ptr())

    # ---------------------------------------------------------------- parameters
    def _pad(self, x, ld):
        x = np.ascontiguousarray(x, dtype=np.float64)
        if x.shape[-1] == ld:
            return x
        out = np.zeros(x.shape[:-1] + (ld,), dtype=np.float64)
        out[..., :x.shape[-1]] = x
        return out

    def set_params(self, theta, eta, pr):
        """theta [S,U,K], eta [S,I,L], pr [S,K,L,R] (numpy, host layout of the reference)."""
        theta, eta, pr = np.asarray(theta), np.asarray(eta), np.asarray(pr)
        if theta.ndim == 2:
            theta, eta, pr = theta[None], eta[None], pr[None]
        S = theta.shape[0]
        if theta.shape != (S, self.U, self.K) or eta.shape != (S, self.I, self.L) \
                or pr.shape != (S, self.K, self.L, self.R):
            raise ValueError("parameter shapes do not match the engine")
        dev = self.device
        self.S = S
        self.theta = torch.from_numpy(self._pad(theta, self.ldk)).to(dev)
        self.eta = torch.from_numpy(self._pad(eta, self.ldl)).to(dev)
        self.pr = torch.from_numpy(np.ascontiguousarray(pr, dtype=np.float64)).to(dev)
        self._alt = (torch.empty_like(self.theta), torch.empty_like(self.eta), torch.empty_like(self.pr))
        if getattr(self, "useg", None) is None:   # prediction-only engine: no EM workspace
            self._ws, self._ws_bytes = None, 0
            return
        need = _lib.C.c_size_t(0)
        _lib.check(self.lib.mmsbm_em_workspace_bytes(self.N, self.U, self.I, self.R, self.K, self.L, S,
                                                     _lib.C.byref(need)), "em_workspace_bytes")
        self._ws = self._bytes(need.value)
        self._ws_bytes = need.value

    def get_params(self):
        """numpy (theta [S,U,K], eta [S,I,L], pr [S,K,L,R])."""
        th = self.theta.cpu().numpy()[..., :self.K]
        et = self.eta.cpu().numpy()[..., :self.L]
        return np.ascontiguousarray(th), np.ascontiguousarray(et), self.pr.cpu().numpy()

    # ------------------------------------------------------------------- EM loop
    def run(self, iterations):
        """``iterations`` EM steps for all S runs, asynchronous on the current stream."""
        if iterations <= 0:
            return
        self._need_ratings()
        a = (self.theta, self.eta, self.pr)
        b = self._alt
        _lib.check(self.lib.mmsbm_em_run(
            *self._graph_args(), self.N, self.U, self.I, self.R, self.K, self.L, self.S, int(iterations),
            a[0].data_ptr(), a[1].data_ptr(), a[2].data_ptr(),
            b[0].data_ptr(), b[1].data_ptr(), b[2].data_ptr(),
            self._ws.data_ptr(), self._ws_bytes, self._stream()), "em_run")
        if iterations % 2:
            self.swap()

    def step_raw(self, flags):
        """One step into the alternate buffers with ``flags`` (RAW_THETA / RAW_ETA_PR);
        returns the three output tensors without swapping."""
        self._need_ratings()
        b = self._alt
        _lib.check(self.lib.mmsbm_em_step(
            *self._graph_args(), self.N, self.U, self.I, self.R, self.K, self.L, self.S,
            self.theta.data_ptr(), self.eta.data_ptr(), self.pr.data_ptr(),
            b[0].data_ptr(), b[1].data_ptr(), b[2].data_ptr(), int(flags),
            self._ws.data_ptr(), self._ws_bytes, self._stream()), "em_step")
        return b

    def finalize(self, eta, pr, ideg=None):
        """Post-all-reduce epilogue, in place."""
        ideg = self.ideg if ideg is None else ideg
        _lib.check(self.lib.mmsbm_em_finalize(eta.data_ptr(), ideg.data_ptr(), self.I, self.L,
                                              pr.data_ptr(), self.K, self.R, self.S, self._stream()),
                   "em_finalize")

    def swap(self):
        (self.theta, self.eta, self.pr), self._alt = self._alt, (self.theta, self.eta, self.pr)

    # ------------------------------------------------------------------- fold-in
    def fold_in(self, side, rows, init, iterations):
        """Rows for ids the engine has not seen, with the parameters it holds fixed.

        ``side`` 0: new users, ``rows`` int [n,3] (user, item, rating) with the new users numbered
        0..n_new-1 and known item ids; ``init`` [S,n_new,K].  ``side`` 1: new items, mirror case,
        ``init`` [S,n_new,L].  Runs ``iterations`` EM steps of the new rows alone (csrc/fold_in.cu)
        and returns them as numpy [S,n_new,K or L]; the engine's parameters are not changed."""
        if side not in (0, 1):
            raise ValueError("side must be 0 (users) or 1 (items)")
        if self.theta is None:
            raise RuntimeError("the engine holds no parameters: set_params first")
        rows, init = np.asarray(rows), np.asarray(init, dtype=np.float64)
        width, ld = (self.K, self.ldk) if side == 0 else (self.L, self.ldl)
        if rows.ndim != 2 or rows.shape[1] != 3:
            raise ValueError("rows must have shape [N,3]")
        if init.ndim != 3 or init.shape[0] != self.S or init.shape[1] < 1 or init.shape[2] != width:
            raise ValueError(f"init must have shape [{self.S}, n_new, {width}]")
        n_new, n = int(init.shape[1]), int(rows.shape[0])
        n_other = self.I if side == 0 else self.U
        i32 = torch.int32
        with torch.cuda.device(self.device):
            raw = torch.from_numpy(np.ascontiguousarray(rows, dtype=np.int64)).to(self.device)
            cols = torch.empty((3, max(n, 1)), dtype=i32, device=self.device)
            bad = torch.zeros(1, dtype=i32, device=self.device)
            nu, ni = (n_new, self.I) if side == 0 else (self.U, n_new)
            _lib.check(self.lib.mmsbm_split_triples(
                raw.data_ptr(), n, nu, ni, self.R, cols[0].data_ptr(), cols[1].data_ptr(), cols[2].data_ptr(),
                bad.data_ptr(), self._stream()), "split_triples")
            if int(bad.item()):
                raise ValueError("rows hold an id outside the new ids, the known ids or the rating levels")
            seg, adj, perm, deg = (self._empty(n_new * self.R + 1, i32), self._empty(n, i32),
                                   self._empty(n, i32), self._empty(n_new, i32))
            n_sched = _lib.C.c_int64(0)
            _lib.check(self.lib.mmsbm_sched_elems(n, n_new, _lib.C.byref(n_sched)), "sched_elems")
            sched = self._empty(n_sched.value, i32)
            need = _lib.C.c_size_t(0)
            _lib.check(self.lib.mmsbm_graph_workspace_bytes(n, n_new, n_new, self.R, _lib.C.byref(need)),
                       "graph_workspace_bytes")
            gws = self._bytes(need.value)
            _lib.check(self.lib.mmsbm_graph_build_side(
                cols[side].data_ptr(), cols[1 - side].data_ptr(), cols[2].data_ptr(), n, n_new, self.R,
                seg.data_ptr(), adj.data_ptr(), perm.data_ptr(), deg.data_ptr(), sched.data_ptr(),
                gws.data_ptr(), need.value, self._stream()), "graph_build_side")
            own = torch.from_numpy(self._pad(init, ld)).to(self.device)
            _lib.check(self.lib.mmsbm_fold_in_workspace_bytes(n, side, n_new, n_other, self.R, self.K, self.L,
                                                              self.S, _lib.C.byref(need)),
                       "fold_in_workspace_bytes")
            ws = self._bytes(need.value)
            _lib.check(self.lib.mmsbm_fold_in(
                seg.data_ptr(), adj.data_ptr(), deg.data_ptr(), n, side, n_new, n_other, self.R, self.K, self.L,
                self.S, int(iterations), (self.eta if side == 0 else self.theta).data_ptr(), self.pr.data_ptr(),
                own.data_ptr(), ws.data_ptr(), need.value, self._stream()), "fold_in")
            return np.ascontiguousarray(own.cpu().numpy()[..., :width])

    def append_rows(self, side, rows):
        """Append ``rows`` [S,n,K] to theta (side 0) or [S,n,L] to eta (side 1) of every run, on the
        device; the new ids follow the existing ones.  The index structure of the training rows
        does not cover them, so the engine becomes parameters-only (like ``for_prediction``):
        ``predict`` serves every id, ``run`` / ``likelihood`` need a new fit."""
        rows = np.asarray(rows, dtype=np.float64)
        width, ld, cur = (self.K, self.ldk, self.theta) if side == 0 else (self.L, self.ldl, self.eta)
        if rows.ndim != 3 or rows.shape[0] != self.S or rows.shape[2] != width:
            raise ValueError(f"rows must have shape [{self.S}, n, {width}]")
        if rows.shape[1] == 0:
            return
        new = torch.cat([cur, torch.from_numpy(self._pad(rows, ld)).to(self.device)], dim=1)
        if side == 0:
            self.theta, self.U = new, self.U + rows.shape[1]
        else:
            self.eta, self.I = new, self.I + rows.shape[1]
        self._alt = (torch.empty_like(self.theta), torch.empty_like(self.eta), torch.empty_like(self.pr))
        self.useg = self.uadj = self.uperm = self.udeg = self.usched = None
        self.iseg = self.iadj = self.iperm = self.ideg = self.isched = None
        self._ws, self._ws_bytes = None, 0

    # ---------------------------------------------------------------- reductions
    def likelihood_device(self):
        self._need_ratings()
        out = self._empty(self.S, torch.float64)
        dims = (self.N, self.U, self.I, self.R, self.K, self.L, self.S)
        need = _lib.C.c_size_t(0)
        _lib.check(self.lib.mmsbm_likelihood_min_workspace_bytes(*dims, _lib.C.byref(need)),
                   "likelihood_min_workspace_bytes")
        if self._ws is not None and self._ws_bytes >= need.value:
            # the EM workspace is idle between iterations (same stream): the likelihood batches its
            # runs to whatever it is given
            ws, ws_bytes = self._ws, self._ws_bytes
        else:
            _lib.check(self.lib.mmsbm_likelihood_workspace_bytes(*dims, _lib.C.byref(need)),
                       "likelihood_workspace_bytes")
            ws, ws_bytes = self._bytes(need.value), need.value
        _lib.check(self.lib.mmsbm_likelihood(
            self.useg.data_ptr(), self.uadj.data_ptr(), self.usched.data_ptr(), self.N, self.U, self.I,
            self.R, self.K, self.L, self.S, self.theta.data_ptr(), self.eta.data_ptr(), self.pr.data_ptr(),
            out.data_ptr(), ws.data_ptr(), ws_bytes, self._stream()), "likelihood")
        ws.record_stream(torch.cuda.current_stream(self.device))
        return out[:self.S]

    def likelihood(self):
        return self.likelihood_device().cpu().numpy()

    def loglik_device(self):
        """Observed-data log-likelihood of every run, sum_n log max(sum_kl theta eta pr, eps): the
        objective EM increases.  [S] float64 on the device."""
        self._need_ratings()
        out = self._empty(self.S, torch.float64)
        dims = (self.N, self.U, self.I, self.R, self.K, self.L, self.S)
        need = _lib.C.c_size_t(0)
        _lib.check(self.lib.mmsbm_loglik_workspace_bytes(*dims, _lib.C.byref(need)), "loglik_workspace_bytes")
        ws = self._bytes(need.value)
        _lib.check(self.lib.mmsbm_loglik(
            self.useg.data_ptr(), self.uadj.data_ptr(), self.usched.data_ptr(), *dims,
            self.theta.data_ptr(), self.eta.data_ptr(), self.pr.data_ptr(),
            out.data_ptr(), ws.data_ptr(), need.value, self._stream()), "loglik")
        ws.record_stream(torch.cuda.current_stream(self.device))
        return out[:self.S]

    def loglik(self):
        return self.loglik_device().cpu().numpy()

    def run_converge(self, max_iterations, tol, check_every=10):
        """EM until each run's log-likelihood changes by at most ``tol`` (relative) between two
        checks ``check_every`` steps apart, or ``max_iterations`` steps (mmsbm_em_run_converge).
        The final parameters of every run are left in theta / eta / pr.  Returns numpy
        (iterations [S] int, converged [S] bool, trace [S, checks + 1]): the log-likelihood at
        each check, NaN after the run's stop.  Synchronous."""
        self._need_ratings()
        max_iterations, check_every = int(max_iterations), int(check_every)
        checks = -(-max_iterations // check_every) if max_iterations > 0 else 0
        dims = (self.N, self.U, self.I, self.R, self.K, self.L, self.S)
        need = _lib.C.c_size_t(0)
        _lib.check(self.lib.mmsbm_em_converge_workspace_bytes(*dims, _lib.C.byref(need)),
                   "em_converge_workspace_bytes")
        ws = self._bytes(need.value)
        trace = torch.empty((self.S, checks + 1), dtype=torch.float64, device=self.device)
        iters = self._empty(self.S, torch.int32)
        conv = self._empty(self.S, torch.int32)
        a, b = (self.theta, self.eta, self.pr), self._alt
        _lib.check(self.lib.mmsbm_em_run_converge(
            *self._graph_args(), *dims, max_iterations, check_every, float(tol),
            a[0].data_ptr(), a[1].data_ptr(), a[2].data_ptr(), b[0].data_ptr(), b[1].data_ptr(), b[2].data_ptr(),
            trace.data_ptr(), iters.data_ptr(), conv.data_ptr(), ws.data_ptr(), need.value, self._stream()),
            "em_run_converge")
        return (iters.cpu().numpy()[:self.S].astype(np.int64), conv.cpu().numpy()[:self.S] != 0,
                trace.cpu().numpy())

    def prod_dist_device(self, test):
        """rat [S,M,R] on the device for int [M,3] (or [M,2]) test rows."""
        test = np.asarray(test)
        M = int(test.shape[0])
        if M and (test[:, 0].min() < 0 or test[:, 0].max() >= self.U
                  or test[:, 1].min() < 0 or test[:, 1].max() >= self.I):
            raise ValueError("test rows hold an id unseen in training")
        tu = torch.from_numpy(np.ascontiguousarray(test[:, 0], dtype=np.int32)).to(self.device)
        ti = torch.from_numpy(np.ascontiguousarray(test[:, 1], dtype=np.int32)).to(self.device)
        rat = torch.empty((self.S, M, self.R), dtype=torch.float64, device=self.device)
        _lib.check(self.lib.mmsbm_prod_dist(
            tu.data_ptr(), ti.data_ptr(), M, self.U, self.I, self.R, self.K, self.L, self.S,
            self.theta.data_ptr(), self.eta.data_ptr(), self.pr.data_ptr(), rat.data_ptr(),
            self._stream()), "prod_dist")
        for t in (tu, ti):
            t.record_stream(torch.cuda.current_stream(self.device))
        return rat

    def mean_over_runs(self, rat):
        S, M, R = rat.shape
        out = torch.empty((M, R), dtype=torch.float64, device=self.device)
        _lib.check(self.lib.mmsbm_mean_over_runs(rat.data_ptr(), M * R, S, out.data_ptr(), self._stream()),
                   "mean_over_runs")
        return out


def predict_stats(rat, real, device=None, want_pred=False):
    """Prediction statistics of src/mmsbm.py:488-539 on the GPU.

    ``rat``: torch cuda tensor or numpy, [S,M,R] or [M,R]; ``real``: encoded ratings [M].
    Returns a list of S dicts (numpy scalars as in the reference) and, optionally, the
    argmax predictions [S,M] (numpy int32)."""
    lib = _lib.load(require_device=True)
    if not isinstance(rat, torch.Tensor):
        dev = torch.device("cuda", torch.cuda.current_device()) if device is None else torch.device(device)
        rat = torch.from_numpy(np.ascontiguousarray(rat, dtype=np.float64)).to(dev)
    if rat.dim() == 2:
        rat = rat[None]
    rat = rat.contiguous()
    dev = rat.device
    S, M, R = rat.shape
    real_d = torch.from_numpy(np.ascontiguousarray(real, dtype=np.int32)).to(dev)
    counts = torch.empty((S, 5), dtype=torch.int64, device=dev)
    s2p = torch.empty((S,), dtype=torch.float64, device=dev)
    pred = torch.empty((S, max(M, 1)), dtype=torch.int32, device=dev) if want_pred else None
    need = _lib.C.c_size_t(0)
    _lib.check(lib.mmsbm_stats_workspace_bytes(M, S, _lib.C.byref(need)), "stats_workspace_bytes")
    ws = torch.empty(max(need.value, 16), dtype=torch.uint8, device=dev)
    stream = torch.cuda.current_stream(dev).cuda_stream
    _lib.check(lib.mmsbm_predict_stats(rat.data_ptr(), real_d.data_ptr(), M, R, S, counts.data_ptr(),
                                       s2p.data_ptr(), pred.data_ptr() if want_pred else None,
                                       ws.data_ptr(), need.value, stream), "predict_stats")
    c = counts.cpu().numpy()
    s = s2p.cpu().numpy()
    out = []
    for k in range(S):
        n = c[k, 0]
        with np.errstate(divide="ignore", invalid="ignore"):
            out.append({
                "accuracy": np.float64(c[k, 1]) / n,
                "one_off_accuracy": np.float64(c[k, 2]) / n,
                "mae": 1 - np.float64(c[k, 4]) / n,
                "s2": np.int64(c[k, 3]),
                "s2pond": np.float64(s[k]),
            })
    if want_pred:
        return out, pred.cpu().numpy()[:, :M]
    return out
