"""Mixed-Membership Stochastic Block Model with the public API of the reference
(src/mmsbm.py:15-553): ``MMSBM(user_groups, item_groups, iterations, sampling, seed,
debug, backend).fit / cv_fit / predict / score``.

What differs is where the work runs.  The reference fans ``sampling`` runs out to a
spawn pool and loops ``update_coefficients`` + three normalisations in numpy
(src/mmsbm.py:182-185, 243-250); here all runs of a rank are batched on one B200:
the index structure, the fused EM iterations, the likelihood, prod_dist and the
prediction statistics are CUDA kernels of libmmsbm_b200.so (engine.py), and runs
shard over GPUs when torch.distributed is initialised (parallel.py).  Kept on the
host, verbatim in behaviour: the string-rank encoding, the seeded initial draws
(numpy PCG64 streams of the SeedSequence children, src/mmsbm.py:82-85,224-233 -- so run
s starts from the same theta0/eta0/pr0 as in the reference) and the fold construction
of cv_fit (it consumes ``self.rng`` sequentially).
"""
from datetime import datetime

import numpy as np

from .data_handler import DataHandler
from .engine import Engine, predict_stats
from .expectation_maximization import ExpectationMaximization
from .helpers import get_n_per_group, structure_folds
from .logger import setup_logger
from .parallel import ShardedEngine, broadcast_seed, dist_info, gather_runs, shard_jobs, shard_runs


class MMSBM:
    """
    Parameters
    ----------
    user_groups, item_groups : int
        Number of latent user / item groups (K, L).
    iterations : int, default=400
        EM iterations per run.
    sampling : int, default=1
        Independent randomly initialised runs; all are kept, the best one (by accuracy
        on the data given to ``predict``, src/mmsbm.py:306,474-478) provides theta/eta/pr.
    seed : int or None
        Seed of the parent generator; run s uses the s-th SeedSequence child.
    debug : bool
        Log the likelihood every 50 iterations (with ``tol``: the log-likelihood of every check).
    backend : str, default="auto"
        "auto" or "b200".  There is no CPU backend.
    shard : str, default="runs"  (extension; only matters under torch.distributed)
        "runs": independent runs round-robin over ranks, no per-iteration communication.
        "ratings": all runs are split over all ranks by user range x item range (each rank owns
        the ratings of its users and of its items); parameter rows travel between GPUs by
        copy-engine DMA and one small all-reduce of the pr accumulator closes every iteration
        (for a fit too slow or too large for one GPU; parallel.ShardedEngine).
    """

    data_handler = None
    results = None
    test = None
    theta = None
    eta = None
    pr = None
    likelihood = None
    prediction_matrix = None
    rng = None

    def __init__(self, user_groups, item_groups, iterations=400, sampling=1, seed=None,
                 debug=False, backend="auto", shard="runs"):
        self.start_time = datetime.now()
        self.user_groups = user_groups
        self.item_groups = item_groups
        self.iterations = iterations
        self.sampling = sampling
        self.debug = debug
        self.backend = backend
        assert shard in ("runs", "ratings"), "shard must be 'runs' or 'ratings'"
        self.shard = shard

        # under torch.distributed every rank must draw the same child seeds and folds: with
        # seed=None rank 0's entropy is used by all
        self.rng = np.random.default_rng(broadcast_seed(seed))
        self.child_states = self.rng.bit_generator._seed_seq.spawn(sampling)

        self.logger = setup_logger("MMSBM")

        self._normalization_factors = None
        self._engine = None
        self._index_cache = None
        self._resident = None       # run ids whose fitted parameters the engine still holds
        self.timings = {}           # wall seconds of the stages of the last fit

    # ------------------------------------------------------------------ preparation
    _MAX_GROUPS = 256
    _MAX_LEVELS = 31

    def _check_shape(self, n_levels):
        """The shapes the kernels are built for, checked before any GPU work so that an
        unsupported one fails here with the limits spelled out (the reference has none)."""
        K, L = self.user_groups, self.item_groups
        if K > self._MAX_GROUPS or L > self._MAX_GROUPS or n_levels > self._MAX_LEVELS:
            raise ValueError(
                f"mmsbm_b200 supports user_groups, item_groups <= {self._MAX_GROUPS} and at most "
                f"{self._MAX_LEVELS} distinct ratings (got K={K}, L={L}, {n_levels} ratings); "
                "see INTEGRATION.md, 'Supported shapes'")
        ld = 4 * ((max(K, L) + 3) // 4)
        if ld > 32 and n_levels * ld > 1024:
            raise ValueError(
                f"mmsbm_b200: with more than 32 groups on a side, ratings x groups must stay <= 1024 "
                f"(got {n_levels} x {ld}); see INTEGRATION.md, 'Supported shapes'")

    def _prepare_objects(self, train, build_engine=True, counts=None):
        """Sizes, degree factors and the on-device index structure
        (replaces src/mmsbm.py:93-146; the O((U+I)N) scans become one GPU sort).
        ``build_engine=False`` (rating-sharded fits): no single-GPU index of all ratings is
        built; the degrees come from a host bincount.  ``counts`` = (users, items, levels) when
        the rows need not reach the top codes or every level (refit); by default they are
        derived from the rows."""
        if counts is None:
            self.ratings = list(np.unique(train[:, 2]))      # = sorted(set(train[:, 2])), src/mmsbm.py:95
            self.p = int(train[:, 0].max())
            self.m = int(train[:, 1].max())
        else:
            self.ratings = list(range(counts[2]))
            self.p, self.m = counts[0] - 1, counts[1] - 1
        self.r = max(self.ratings)
        self.train = train
        self._dims = {
            'n_samples': len(train),
            'n_user_groups': self.user_groups,
            'n_item_groups': self.item_groups,
            'n_ratings': len(self.ratings),
        }
        self.em = ExpectationMaximization(
            dims=self._dims, user_indices=None, item_indices=None, rating_indices=None,
            norm_factors=None, backend=self.backend, debug=self.debug)
        self._check_shape(self._dims['n_ratings'])
        self._resident = None
        if build_engine:
            self._engine = Engine(train, self.p + 1, self.m + 1, self._dims['n_ratings'],
                                  self.user_groups, self.item_groups)
            du = np.maximum(self._engine.udeg.cpu().numpy()[:self.p + 1].astype(np.int64), 1)
            di = np.maximum(self._engine.ideg.cpu().numpy()[:self.m + 1].astype(np.int64), 1)
        else:
            self._engine = None
            du = np.maximum(np.bincount(train[:, 0], minlength=self.p + 1).astype(np.int64), 1)
            di = np.maximum(np.bincount(train[:, 1], minlength=self.m + 1).astype(np.int64), 1)
        self._normalization_factors = {
            'user': np.repeat(du[:, None], self.user_groups, axis=1),
            'item': np.repeat(di[:, None], self.item_groups, axis=1),
        }
        self.em._normalization_factors = self._normalization_factors
        self._index_cache = None

    def _index_lists(self):
        """Per-id row lists of the reference (src/mmsbm.py:114-122), derived on demand
        from the device index structure."""
        if self._index_cache is None:
            e, R = self._engine, self._dims['n_ratings']
            out = {}
            for name, seg, perm, n_ids in (("user", e.useg, e.uperm, e.U), ("item", e.iseg, e.iperm, e.I)):
                seg, perm = seg.cpu().numpy(), perm.cpu().numpy()[:e.N]
                out[name] = [np.sort(perm[seg[a * R]:seg[(a + 1) * R]]).astype(np.int64)
                             for a in range(n_ids)]
            seg, perm = e.useg.cpu().numpy(), e.uperm.cpu().numpy()[:e.N]
            out["rating"] = [np.sort(np.concatenate(
                [perm[seg[a * R + r]:seg[a * R + r + 1]] for a in range(e.U)] or [perm[:0]])).astype(np.int64)
                for r in range(R)]
            self._index_cache = out
        return self._index_cache

    def _has_index(self):
        return self._engine is not None and self._engine.useg is not None

    @property
    def _user_indices(self):
        return self._index_lists()["user"] if self._has_index() else None

    @property
    def _item_indices(self):
        return self._index_lists()["item"] if self._has_index() else None

    @property
    def _rating_indices(self):
        return self._index_lists()["rating"] if self._has_index() else None

    def _initial_parameters(self, seed):
        """theta0, eta0, pr0 of one run: three draws in this order from
        default_rng(seed) (src/mmsbm.py:224-233)."""
        rng = np.random.default_rng(seed)
        K, L, R = self.user_groups, self.item_groups, self._dims['n_ratings']
        theta = self.em.normalize_with_d(rng.random((self.p + 1, K)), 'user')
        eta = self.em.normalize_with_d(rng.random((self.m + 1, L)), 'item')
        pr = self.em.normalize_with_self(rng.random((K, L, R)))
        return theta, eta, pr

    # -------------------------------------------------------------------------- fit
    def _tick(self, stage, t0):
        """Wall seconds of a stage of the last fit, accumulated in ``self.timings`` (bench.py's
        api_e2e reports them; the device is synchronised so the split is meaningful)."""
        import time
        import torch
        if torch.cuda.is_available():
            torch.cuda.synchronize()
        now = time.perf_counter()
        self.timings[stage] = self.timings.get(stage, 0.0) + (now - t0)
        return now

    def _initial_batch(self, seeds):
        """theta0/eta0/pr0 of several runs, stacked.  The draws of different runs come from
        independent generators (one SeedSequence child each), so they run in threads (numpy's
        Generator releases the GIL while filling an array); every run's stream is untouched."""
        if len(seeds) > 1 and (self.p + 1) * self.user_groups >= 200_000:
            from concurrent.futures import ThreadPoolExecutor
            with ThreadPoolExecutor(max_workers=min(len(seeds), 8)) as ex:
                inits = list(ex.map(self._initial_parameters, seeds))
        else:
            inits = [self._initial_parameters(s) for s in seeds]
        return tuple(np.stack([a[j] for a in inits]) for j in range(3))

    def _check_convergence_args(self, tol, check_every):
        """The stopping rule's arguments, checked before any GPU work."""
        if tol is not None:
            if isinstance(tol, bool) or not isinstance(tol, (int, float, np.integer, np.floating)) \
                    or not np.isfinite(tol) or tol < 0:
                raise ValueError(f"tol must be a finite number >= 0 or None (got {tol!r})")
            if dist_info()[1] > 1 and self.shard == "ratings":
                raise ValueError("tol is not supported with shard='ratings' under torch.distributed; "
                                 "use shard='runs' or a fixed iteration count")
        if isinstance(check_every, bool) or not isinstance(check_every, (int, np.integer)) \
                or check_every < 2 or check_every % 2:
            raise ValueError(f"check_every must be an even integer >= 2 (got {check_every!r})")

    def _run_batch(self, engine, seeds, run_ids, init=None, iterations=None, tol=None, check_every=10):
        """EM runs ``run_ids`` on ``engine``: from the seeded draws of ``seeds``, or from ``init`` =
        stacked (theta0, eta0, pr0) when given; ``iterations`` defaults to ``self.iterations``.
        With ``tol``, ``iterations`` is the maximum and each run stops on its own at convergence
        (Engine.run_converge); its result then also holds "iterations", "converged" and "loglik"."""
        import time
        iterations = self.iterations if iterations is None else iterations
        t = time.perf_counter()
        theta0, eta0, pr0 = self._initial_batch(seeds) if init is None else init
        t = self._tick("init_draws", t)
        engine.set_params(theta0, eta0, pr0)
        t = self._tick("params_h2d", t)
        conv = None
        if tol is not None:
            n_it, converged, trace = engine.run_converge(iterations, tol, check_every)
            conv = {}
            for j, i in enumerate(run_ids):
                checks = trace[j][~np.isnan(trace[j])]
                conv[i] = {"iterations": int(n_it[j]), "converged": bool(converged[j]), "loglik": checks}
                if self.debug:
                    for c, v in enumerate(checks):
                        self.logger.debug(f"\nLog-likelihood at run {i} after "
                                          f"{min(c * check_every, iterations)} iterations is {v:.6f}")
        elif self.debug:
            done = 0
            while done < iterations:
                step = 1 if done == 0 else min(50, iterations - done)
                engine.run(step)
                done += step
                if (done - 1) % 50 == 0:
                    for i, lik in zip(run_ids, engine.likelihood()):
                        self.logger.debug(f"\nLikelihood at run {i} is {lik:.0f}")
        else:
            engine.run(iterations)
        t = self._tick("em_iterations", t)
        lik = engine.likelihood()
        t = self._tick("likelihood", t)
        theta, eta, pr = engine.get_params()
        t = self._tick("results_d2h", t)
        self._resident = list(run_ids) if engine is self._engine else None
        out = {i: {"likelihood": np.float64(lik[j]), "pr": pr[j], "theta": theta[j], "eta": eta[j]}
               for j, i in enumerate(run_ids)}
        if conv is not None:
            for i in run_ids:
                out[i].update(conv[i])
        return out

    def fit(self, data, silent=False, tol=None, check_every=10):
        """Fit ``sampling`` EM runs on a DataFrame with columns [users, items, ratings].

        ``tol``: stop each run at convergence.  The observed-data log-likelihood (the quantity EM
        increases) is evaluated at the start and every ``check_every`` steps (even, >= 2); a run stops
        at the first check where it changed by at most ``tol`` times its magnitude since the previous
        one, and ``self.iterations`` becomes the maximum.  Every ``results[s]`` then also holds
        ``"iterations"`` (steps run), ``"converged"`` (False: stopped at the maximum) and ``"loglik"``
        (the log-likelihood at each check up to the stop).  ``None`` (default): exactly
        ``self.iterations`` steps, as before."""
        self._check_convergence_args(tol, check_every)
        if not silent:
            self.logger.info(f"Running {self.sampling} runs of {self.iterations} iterations.")
        import time
        self.timings = {}
        t = time.perf_counter()
        self.data_handler = DataHandler()
        train = self.data_handler.format_train_data(data)
        t = self._tick("encode", t)
        rank, world = dist_info()
        if world > 1 and self.shard == "ratings":
            self._prepare_objects(train, build_engine=False)
            eng = ShardedEngine(train, self.p + 1, self.m + 1, self._dims['n_ratings'],
                                self.user_groups, self.item_groups)
            every = list(range(self.sampling))
            try:
                done = self._run_batch(eng, [self.child_states[i] for i in every], every)
            finally:
                eng.close()
            self.results = [done[i] for i in every]
            return
        self._prepare_objects(train)
        self._tick("rows_h2d_index_build", t)
        mine = shard_runs(self.sampling, rank, world)
        local = self._run_batch(self._engine, [self.child_states[i] for i in mine], mine,
                                tol=tol, check_every=check_every) if mine else {}
        self.results = gather_runs(local, self.sampling)

    def run_one_sampling(self, data, seed, i):
        """One EM run from ``seed`` on the encoded array ``data`` (in-process; the
        reference's unit of work, src/mmsbm.py:187-269)."""
        engine = self._engine
        if engine is None or data is not self.train:
            engine = Engine(data, self.p + 1, self.m + 1, self._dims['n_ratings'],
                            self.user_groups, self.item_groups)
        return self._run_batch(engine, [seed], [i])[i]

    def _check_is_fitted(self):
        assert self.results is not None, "You need to fit the model before predicting."

    def _check_has_predictions(self):
        assert self.prediction_matrix is not None, (
            "You need to predict before computing the goodness of fit " "parameters.")

    # ---------------------------------------------------------------------- predict
    def predict(self, data):
        """Rating distribution [M,R] for the rows of ``data`` (mean over runs); the best
        run (highest accuracy on ``data``, first on ties) provides theta / eta / pr."""
        self._check_is_fitted()
        test = self.data_handler.format_test_data(data)
        self.test = test

        prs = np.array([a["pr"] for a in self.results])
        likelihoods = np.array([a["likelihood"] for a in self.results])
        thetas = np.array([a["theta"] for a in self.results])
        etas = np.array([a["eta"] for a in self.results])

        engine = self._engine
        if engine is None:                                    # rating-sharded fit: parameters only
            engine = self._engine = Engine.for_prediction(self.p + 1, self.m + 1, self._dims['n_ratings'],
                                                          self.user_groups, self.item_groups)
        if self._resident != list(range(len(self.results))) or engine.S != len(self.results):
            engine.set_params(thetas, etas, prs)              # else: still on the device from fit
            self._resident = list(range(len(self.results)))
        rat = engine.prod_dist_device(test)                   # [S,M,R] on the GPU
        accuracies = [s["accuracy"] for s in predict_stats(rat, test[:, 2])]
        best = accuracies.index(max(accuracies))

        self.theta = self.data_handler.return_theta_indices(thetas[best])
        self.eta = self.data_handler.return_eta_indices(etas[best])
        self.pr = self.data_handler.return_pr_indices(prs[best])
        self.likelihood = likelihoods[best]

        self.prediction_matrix = engine.mean_over_runs(rat).cpu().numpy()
        return self.prediction_matrix

    def score(self, silent=False):
        """{"stats": {accuracy, one_off_accuracy, mae, s2, s2pond, likelihood},
        "objects": {theta, eta, pr}} for the last prediction."""
        self._check_has_predictions()
        stats = self._compute_stats(self.prediction_matrix)
        stats["likelihood"] = self.likelihood
        if not silent:
            self.logger.debug(
                f"Done {self.sampling} runs in {(datetime.now() - self.start_time).total_seconds() / 60.0:.2f} "
                f"minutes.")
            self.logger.info(
                f"The final accuracy is {stats['accuracy']}, the one off accuracy is {stats['one_off_accuracy']} "
                f"and the MAE is {stats['mae']}.")
        return {"stats": stats, "objects": {"theta": self.theta, "eta": self.eta, "pr": self.pr}}

    # ---------------------------------------------------------------------- fold_in
    def fold_in(self, data, iterations=None, seed=0):
        """Parameters for users and items the fitted model has not seen, without refitting.

        ``data``: a DataFrame read by position like ``fit``.  A row of a new user with a known item
        is used for that user's theta, a row of a known user with a new item for that item's eta;
        the rest is dropped or ignored with a warning (DataHandler.plan_fold_in).  With eta and pr
        (theta and pr) fixed, ``iterations`` (default: ``self.iterations``) EM steps run on the new
        rows alone, for every run; the known rows of every run stay as they are.  Run s starts from
        ``default_rng(SeedSequence(seed).spawn(S)[s])``: ``random((new users, K))`` then
        ``random((new items, L))``, each row divided by max(its fold-in rows, 1).  ``self.rng`` is
        not used.  Afterwards ``predict`` / ``score`` / ``save`` serve the new ids.

        Returns {"users": [...], "items": [...]}: the labels added, in code order."""
        self._check_is_fitted()
        iterations = self.iterations if iterations is None else int(iterations)
        plan = self.data_handler.plan_fold_in(data)
        added = {"users": plan["users"], "items": plan["items"]}
        nu, ni = len(plan["users"]), len(plan["items"])
        if not nu and not ni:
            return added
        S, K, L = len(self.results), self.user_groups, self.item_groups
        engine = self._engine
        if engine is None:                                    # rating-sharded fit: parameters only
            engine = self._engine = Engine.for_prediction(self.p + 1, self.m + 1, self._dims['n_ratings'],
                                                          K, L)
        if self._resident != list(range(S)) or engine.S != S:
            engine.set_params(np.array([a["theta"] for a in self.results]),
                              np.array([a["eta"] for a in self.results]),
                              np.array([a["pr"] for a in self.results]))
            self._resident = list(range(S))
        du = np.maximum(np.bincount(plan["user_rows"][:, 0], minlength=nu), 1)[:, None]
        di = np.maximum(np.bincount(plan["item_rows"][:, 1], minlength=ni), 1)[:, None]
        init_u, init_i = np.empty((S, nu, K)), np.empty((S, ni, L))
        for s, child in enumerate(np.random.SeedSequence(seed).spawn(S)):
            rng = np.random.default_rng(child)
            init_u[s] = rng.random((nu, K)) / du
            init_i[s] = rng.random((ni, L)) / di
        # both sets are computed from the known rows only, so neither depends on the other
        new_theta = engine.fold_in(0, plan["user_rows"], init_u, iterations) if nu else init_u
        new_eta = engine.fold_in(1, plan["item_rows"], init_i, iterations) if ni else init_i
        engine.append_rows(0, new_theta)
        engine.append_rows(1, new_eta)
        for s, res in enumerate(self.results):
            res["theta"] = np.concatenate([res["theta"], new_theta[s]])
            res["eta"] = np.concatenate([res["eta"], new_eta[s]])
        self.data_handler.add_fold_in_ids(plan["users"], plan["items"])
        self.p, self.m = self.p + nu, self.m + ni
        self._index_cache = None
        return added

    # ------------------------------------------------------------------------ refit
    def refit(self, data, iterations=None, seed=0, tol=None, check_every=10):
        """Fit on ``data`` again, starting from this model's parameters instead of random draws.

        ``data`` is the whole rating set the model should describe from now on -- normally the old
        ratings plus the new ones, NOT only the new rows.  It is read by position like ``fit`` and
        encoded against the model's dictionaries (DataHandler.plan_refit): known ids keep their
        codes, new users and items get the codes after the existing ones (ranked among themselves by
        ``sorted(set(str))``), rows with a rating value the model does not have are dropped with a
        warning.  Run s starts from its current theta / eta / pr; new ids draw from
        ``default_rng(SeedSequence(seed).spawn(S)[s])``: ``random((new users, K))`` then
        ``random((new items, L))``, each row divided by max(its rows in ``data``, 1).  ``self.rng``
        is not used.  ``iterations`` (default: ``self.iterations``) EM steps then run over all rows,
        for every run.  Known ids without a row in ``data`` keep their parameters (with a warning);
        a rating level without a row gets a zero pr slab, as in EM.  Calling ``fold_in(data)`` first
        gives the new ids a fold-in start instead of a random one.

        ``tol`` / ``check_every``: stop each run at convergence, with ``iterations`` as the maximum
        (see ``fit``).

        Afterwards ``results``, ``train`` and the degree factors describe ``data``, and
        ``likelihood`` / ``predict`` / ``score`` / ``save`` / ``refit`` work as after ``fit``.
        Returns {"users": [...], "items": [...]}: the labels added, in code order."""
        import time
        self._check_is_fitted()
        self._check_convergence_args(tol, check_every)
        iterations = self.iterations if iterations is None else int(iterations)
        self.timings = {}
        t = time.perf_counter()
        plan = self.data_handler.plan_refit(data)
        t = self._tick("encode_plan", t)
        rows = plan["rows"]
        S, K, L, R = len(self.results), self.user_groups, self.item_groups, self._dims['n_ratings']
        U0, I0 = self.p + 1, self.m + 1
        U, I = U0 + len(plan["users"]), I0 + len(plan["items"])
        deg_u, deg_i = np.bincount(rows[:, 0], minlength=U), np.bincount(rows[:, 1], minlength=I)
        du, di = np.maximum(deg_u[U0:], 1)[:, None], np.maximum(deg_i[I0:], 1)[:, None]
        theta0, eta0 = np.empty((S, U, K)), np.empty((S, I, L))
        for s, (res, child) in enumerate(zip(self.results, np.random.SeedSequence(seed).spawn(S))):
            rng = np.random.default_rng(child)
            theta0[s, :U0], theta0[s, U0:] = res["theta"], rng.random((U - U0, K)) / du
            eta0[s, :I0], eta0[s, I0:] = res["eta"], rng.random((I - I0, L)) / di
        pr0 = np.stack([res["pr"] for res in self.results])
        absent_u, absent_i = np.flatnonzero(deg_u[:U0] == 0), np.flatnonzero(deg_i[:I0] == 0)
        if len(absent_u) or len(absent_i):
            self.logger.warning(f"{len(absent_u)} users and {len(absent_i)} items of the model have no rows in "
                                f"the refit set so they keep their parameters.")
        t = self._tick("init_draws", t)

        rank, world = dist_info()
        if world > 1 and self.shard == "ratings":
            self._prepare_objects(rows, build_engine=False, counts=(U, I, R))
            eng = ShardedEngine(rows, U, I, R, K, L)
            every = list(range(S))
            try:
                done = self._run_batch(eng, None, every, init=(theta0, eta0, pr0), iterations=iterations)
            finally:
                eng.close()
            results = [done[s] for s in every]
        else:
            self._prepare_objects(rows, counts=(U, I, R))
            self._tick("rows_h2d_index_build", t)
            mine = shard_runs(S, rank, world)
            local = self._run_batch(self._engine, None, mine, init=(theta0[mine], eta0[mine], pr0[mine]),
                                    iterations=iterations, tol=tol, check_every=check_every) if mine else {}
            # EM leaves a zero row where an id has no rating: put the old rows back, on the device too
            # when the engine still holds these runs for predict
            if self._resident is not None:
                import torch
                e = self._engine
                for absent, cur, init, width in ((absent_u, e.theta, theta0, K), (absent_i, e.eta, eta0, L)):
                    if len(absent):
                        cur[:, torch.from_numpy(absent).to(e.device), :width] = \
                            torch.from_numpy(init[np.ix_(mine, absent)]).to(e.device)
            results = gather_runs(local, S)
        for s, res in enumerate(results):
            res["theta"][absent_u] = theta0[s, absent_u]
            res["eta"][absent_i] = eta0[s, absent_i]
        self.results = results
        self.data_handler.add_fold_in_ids(plan["users"], plan["items"])
        return {"users": plan["users"], "items": plan["items"]}

    # ----------------------------------------------------------------------- cv_fit
    def _make_folds(self, data, folds):
        """(train, test) DataFrames of every fold, built as the reference does
        (src/mmsbm.py:415-439): per user (groups in sorted key order) up to items_per_fold
        held-out rows, drawn from ``self.rng`` in that order; index label 0 is never held out
        (the reference filters str(a) != "0", :435).  The fits do not touch ``self.rng``, so
        building all folds first consumes it exactly as the reference's interleaved loop.

        Fast path (SURVEY.md section 8 f3): ``rng.choice(x.index, k, replace=False)`` draws
        positions from the group SIZE only, so the same stream is consumed by
        ``rng.choice(len(x), k, replace=False)`` on row positions kept in numpy arrays -- no
        pandas groupby / .loc / .isin per fold.  Taken when the frame has a unique index and a
        plain integer / float-without-NaN / str user column (where ``np.unique`` orders the
        groups exactly like ``groupby``); anything else goes through pandas as before."""
        items_per_fold = structure_folds(data, folds)
        fast = self._make_folds_fast(data, folds, items_per_fold)
        if fast is not None:
            return fast
        temp = data
        pairs = []
        for _ in range(folds):
            picked = []
            for _, group in temp.groupby(temp.columns[0]):
                chosen = get_n_per_group(group, n=items_per_fold, rng=self.rng)
                picked.extend(chosen)
            test_indices = [a for a in picked if str(a) != "0"]
            test = temp.loc[test_indices, :]
            train = data[~data.index.isin(test.index)]
            temp = temp[~temp.index.isin(test_indices)]
            pairs.append((train, test))
        return pairs

    def _make_folds_fast(self, data, folds, items_per_fold):
        if not data.index.is_unique or items_per_fold <= 0:
            return None
        users = data.iloc[:, 0].to_numpy()
        kind = users.dtype.kind
        if kind == "f" and np.isnan(users).any():
            return None
        if kind == "O":
            import pandas as pd
            if not len(users) or pd.api.types.infer_dtype(users, skipna=False) != "string":
                return None
        elif kind not in "iuf":
            return None
        _, codes = np.unique(users, return_inverse=True)           # sorted keys, like groupby
        order = np.argsort(codes, kind="stable")                   # rows of a group in frame order
        bounds = np.flatnonzero(np.diff(codes[order], prepend=-1, append=codes.max(initial=-1) + 1))
        groups = [order[bounds[j]:bounds[j + 1]] for j in range(len(bounds) - 1)]
        labels = data.index
        zero_label = np.fromiter((str(a) == "0" for a in labels), dtype=bool, count=len(labels)) \
            if labels.dtype.kind not in "iu" else (labels.to_numpy() == 0)
        alive = np.ones(len(data), dtype=bool)
        pairs = []
        for _ in range(folds):
            picked = []
            for rows in groups:
                rows = rows[alive[rows]]
                take = min(items_per_fold, len(rows))
                if take > 0:
                    picked.append(rows[self.rng.choice(len(rows), take, replace=False)])
            picked = np.concatenate(picked) if picked else np.zeros(0, dtype=np.int64)
            picked = picked[~zero_label[picked]]
            held = np.zeros(len(data), dtype=bool)
            held[picked] = True
            pairs.append((data.iloc[~held], data.iloc[picked]))
            alive[picked] = False
        return pairs

    def cv_fit(self, data, folds=5, tol=None, check_every=10):
        """k-fold cross-validation; returns the accuracy of every fold and keeps the objects of
        the most accurate one (src/mmsbm.py:371-472).  Under torch.distributed the folds x runs
        jobs shard over the ranks (SURVEY.md section 8e.2); the result is the same.  ``tol`` /
        ``check_every``: every fit stops at convergence (see ``fit``)."""
        self._check_convergence_args(tol, check_every)
        return self._cv_execute(self._make_folds(data, folds), tol, check_every)

    def _cv_execute(self, pairs, tol=None, check_every=10):
        """Fit / predict / score every (train, test) pair and keep the best fold: the part of
        ``cv_fit`` after the fold construction (src/mmsbm.py:441-472)."""
        folds = len(pairs)
        rank, world = dist_info()
        sharded_cv = world > 1 and self.shard == "runs"
        done = {}
        if sharded_cv:
            mine = shard_jobs(folds, self.sampling, rank, world)
            local = {}
            for f in sorted({f for f, _ in mine}):
                self.data_handler = DataHandler()
                self._prepare_objects(self.data_handler.format_train_data(pairs[f][0]))
                runs = [s for (ff, s) in mine if ff == f]
                out = self._run_batch(self._engine, [self.child_states[s] for s in runs], runs,
                                      tol=tol, check_every=check_every)
                local.update({(f, s): out[s] for s in runs})
            import torch.distributed as dist
            boxes = [None] * world
            dist.all_gather_object(boxes, local)
            for b in boxes:
                done.update(b)

        all_results = []
        for f, (train, test) in enumerate(pairs):
            self.logger.info(f"Running fold {f + 1} of {folds}...")
            if sharded_cv:
                # the runs of this fold were fitted on some ranks: only the encoding and a
                # parameters-only engine (created by predict) are needed here
                self.data_handler = DataHandler()
                self._prepare_objects(self.data_handler.format_train_data(train), build_engine=False)
                self.results = [done[(f, s)] for s in range(self.sampling)]
            else:
                self.fit(train, silent=True, tol=tol, check_every=check_every)
            self.prediction_matrix = self.predict(test)
            results = self.score(silent=True)
            all_results.append({
                "stats": results["stats"],
                "objects": {"theta": self.theta, "eta": self.eta, "pr": self.pr,
                            "rat": self.prediction_matrix},
            })

        accuracies = [a["stats"]["accuracy"] for a in all_results]
        best = accuracies.index(max(accuracies))
        self.theta = all_results[best]["objects"]["theta"]
        self.eta = all_results[best]["objects"]["eta"]
        self.pr = all_results[best]["objects"]["pr"]
        self.prediction_matrix = all_results[best]["objects"]["rat"]

        self.logger.info(f"Ran {folds} folds with accuracies {accuracies}.")
        self.logger.info(f"They have mean {np.mean(accuracies)} and sd {np.std(accuracies)}.")
        return accuracies

    # ------------------------------------------------------------------ save / load
    def save(self, path):
        """Write the fitted model to one ``.npz`` file: the parameters and likelihood of every run,
        the three id dictionaries and the constructor arguments.  (The reference has no on-disk
        format; this is the adjacent feature of SURVEY.md section 8 f4.)  ``MMSBM.load(path)``
        gives a model that can ``predict`` and ``score``."""
        import json
        self._check_is_fitted()
        config = {"user_groups": self.user_groups, "item_groups": self.item_groups,
                  "iterations": self.iterations, "sampling": self.sampling, "debug": self.debug,
                  "backend": self.backend, "shard": self.shard}
        dicts = [list(d.items()) for d in self.data_handler.return_dicts()]
        with open(path, "wb") as fh:
            np.savez_compressed(
                fh, format_version=np.int64(1), config=np.array(json.dumps(config)),
                dicts=np.array(json.dumps(dicts)),
                theta=np.stack([a["theta"] for a in self.results]),
                eta=np.stack([a["eta"] for a in self.results]),
                pr=np.stack([a["pr"] for a in self.results]),
                likelihood=np.array([a["likelihood"] for a in self.results], dtype=np.float64))

    @classmethod
    def load(cls, path):
        """Restore a model written by ``save`` (prediction side only: no training rows are kept)."""
        import json
        with np.load(path, allow_pickle=False) as z:
            if int(z["format_version"]) != 1:
                raise ValueError(f"unknown mmsbm_b200 model format {int(z['format_version'])}")
            config = json.loads(str(z["config"]))
            dicts = [dict((k, int(v)) for k, v in d) for d in json.loads(str(z["dicts"]))]
            theta, eta, pr, lik = z["theta"], z["eta"], z["pr"], z["likelihood"]
        self = cls(**config)
        self.data_handler = DataHandler()
        self.data_handler.obs_dict, self.data_handler.items_dict, self.data_handler.ratings_dict = dicts
        self.results = [{"likelihood": np.float64(lik[s]), "pr": pr[s], "theta": theta[s], "eta": eta[s]}
                        for s in range(theta.shape[0])]
        self.p, self.m = theta.shape[1] - 1, eta.shape[1] - 1
        self.ratings = list(range(pr.shape[3]))
        self.r = pr.shape[3] - 1
        self._dims = {'n_samples': 0, 'n_user_groups': self.user_groups,
                      'n_item_groups': self.item_groups, 'n_ratings': pr.shape[3]}
        self._engine = Engine.for_prediction(self.p + 1, self.m + 1, pr.shape[3],
                                             self.user_groups, self.item_groups)
        return self

    # ------------------------------------------------------------------------ stats
    def choose_best_run(self, rats):
        """Index of the run with the highest accuracy (first on ties)."""
        accuracies = [self._compute_stats(a)["accuracy"] for a in rats]
        return accuracies.index(max(accuracies))

    def _compute_stats(self, rat):
        """accuracy, one_off_accuracy, mae, s2, s2pond of one [M,R] distribution against
        ``self.test`` -- an on-device reduction (src/mmsbm.py:480-539)."""
        return predict_stats(rat, self.test[:, 2])[0]

    def compute_likelihood(self, data, theta, eta, pr):
        return self.em.compute_likelihood(data, theta, eta, pr)
