"""KMeans -- drop-in for `sklearn.cluster.KMeans` as get_basis.py:210 uses it: `KMeans(n_clusters=, init='k-means++').fit(X).labels_`.

Lloyd iterations run on the GPU: gfs_kmeans_assign (fp32 pinned-order E-step) + gfs_kmeans_accumulate (deterministic
sums) per iteration; the control flow mirrors sklearn 1.9.0 (_kmeans.py:1487-1490 mean-centring, :289-296 tolerance,
:630-759 Lloyd loop / convergence, _k_means_common.pyx:167-260 empty-cluster relocation and centre averaging).

Up to 512 clusters with at most 192 features (up to 192 clusters with 193..256 features).  Beyond 192 clusters the E-step
runs the panelled tensor-core path, which needs a multiple of 64 channels: the channel-major copies of the points and the
centres then carry zero channels up to the next multiple of 64, which leave the pinned fp32 chains (and so the labels)
unchanged, since fmaf(0, 0, s) == s.

Multi-GPU: pass `process_group` (or have torch.distributed initialised and shard=True): X is then THIS rank's shard of
the points; the only exchange per iteration is an NCCL all-reduce of the (K*D + K) fp64 sums/counts (+ the mean/variance
once), every rank applies the identical centroid update.

Beyond get_basis.py: the rest of sklearn's KMeans interface -- `sample_weight` (weighted seeding, M-step, relocation and
inertia: _k_means_lloyd.pyx:216-218, _kmeans.py:_kmeans_plusplus), `init='random'`, the `n_init` loop (_kmeans.py:1504-1545),
`inertia_`, `predict`, `transform`, `fit_transform` and `score`.  Numpy inputs give numpy results, tensors give tensors.

Inject for the reference script without editing it:   import get_basis; get_basis.KMeans = gfs3d.kmeans.KMeans
"""
import warnings
from typing import Optional

import numpy as np
import torch

from . import ops


def _dist():
    import torch.distributed as dist
    return dist


class KMeans:
    def __init__(self, n_clusters=8, *, init="k-means++", n_init="auto", max_iter=300, tol=1e-4, verbose=0,
                 random_state=None, copy_x=True, algorithm="lloyd", device=None, shard=False, process_group=None):
        if algorithm not in ("lloyd", "auto", "full"):
            raise NotImplementedError(f"algorithm={algorithm!r}: only Lloyd is built")
        self.n_clusters, self.init, self.n_init = n_clusters, init, n_init
        self.max_iter, self.tol, self.verbose, self.random_state = max_iter, tol, verbose, random_state
        self.device = device
        self.shard = shard or process_group is not None
        self.process_group = process_group

    # ------------------------------------------------------------------ helpers
    def _allreduce(self, t):
        if self.shard:
            _dist().all_reduce(t, group=self.process_group)
        return t

    def _rng(self):
        rs = self.random_state
        if rs is None:
            return np.random.mtrand._rand          # numpy global state, as sklearn's check_random_state(None)
        if isinstance(rs, np.random.RandomState):
            return rs
        return np.random.RandomState(rs)

    def _world(self):
        if not self.shard:
            return 1, 0
        d = _dist()
        return d.get_world_size(self.process_group), d.get_rank(self.process_group)

    def _gather_sizes(self, n, dev):
        world, rank = self._world()
        sizes = torch.tensor([n], dtype=torch.int64, device=dev)
        if world > 1:
            allsz = [torch.empty_like(sizes) for _ in range(world)]
            _dist().all_gather(allsz, sizes, group=self.process_group)
            sizes = torch.cat(allsz)
        return sizes.tolist()

    def _gather_weights(self, w, sizes):
        """the weights of all ranks in rank order (4 bytes per point, once per seeding), as float32 numpy"""
        world, _ = self._world()
        if world == 1:
            return w.cpu().numpy()
        parts = [torch.empty(s_, dtype=torch.float32, device=w.device) for s_ in sizes]
        _dist().all_gather(parts, w.contiguous(), group=self.process_group)
        return torch.cat(parts).cpu().numpy()

    def _broadcast0(self, t):
        if self._world()[0] > 1:
            _dist().broadcast(t, src=_dist().get_global_rank(self.process_group, 0) if self.process_group else 0,
                              group=self.process_group)
        return t

    def _owned_rows(self, Xc, n, pos, mine):
        """(T, D) rows Xc[pos] where this rank owns the pick, zero elsewhere; summed over the ranks"""
        rows = Xc[pos.clamp(0, n - 1)] * mine.to(torch.float32).unsqueeze(1)
        if self._world()[0] > 1:
            _dist().all_reduce(rows, group=self.process_group)
        return rows.contiguous()

    def _seed_random(self, Xc, rng, n, w=None):
        """sklearn _kmeans.py:1030-1037: K distinct rows drawn with choice(n, size=K, replace=False, p=w/sum(w)) -- p is passed
        with unit weights too, as sklearn does (numpy draws differently without it).  Sharded: drawn on rank 0 over the points
        of all ranks in rank order, each row contributed by its owner rank."""
        K = self.n_clusters
        dev = Xc.device
        _, rank = self._world()
        sizes = self._gather_sizes(n, dev)
        n_tot, lo = sum(sizes), sum(sizes[:rank])
        wall = self._gather_weights(w, sizes) if w is not None else None
        idx = torch.empty(K, dtype=torch.int64)
        if rank == 0:
            wa = wall if wall is not None else np.ones(n_tot, dtype=np.float32)
            idx[:] = torch.from_numpy(rng.choice(n_tot, size=K, replace=False, p=wa / wa.sum()).astype(np.int64))
        idx = self._broadcast0(idx.to(dev))
        pos = idx - lo
        return self._owned_rows(Xc, n, pos, (pos >= 0) & (pos < n))

    def _seed_plusplus(self, Xc, xt, rng, n=None, w=None):
        """k-means++ exactly as sklearn's _kmeans_plusplus consumes its random stream (sklearn 1.9.0 _kmeans.py:_kmeans_plusplus):
        first centre through `choice(n, p=w/sum(w))`, then `uniform(size=2+ln K)` per centre; candidates = searchsorted of
        u * potential in the cumulative sum of the closest squared distances; all candidates of a centre scored in ONE pass over
        the resident channel-major copy (gfs_kmeans_pp_trial: fp64-accumulated distances rounded to fp32, like sklearn's upcast
        path), the best kept.  What is NOT bit-pinned: sklearn sums the potential with a float32 BLAS dot and the cumulative sum in
        float32; here both are fp64 (parallel, order-independent to 1e-16), so a pick can differ where u * pot lands within that
        rounding of a boundary (tests/golden: 31 of 32 seeded problems give identical picks for all centres).

        Sharded (multi-GPU): the points of all ranks form ONE sequence in rank order; every rank searches its own slice of the
        global cumulative sum, the owner contributes the candidate rows (all-reduce), potentials are all-reduced: the picks equal
        the single-GPU picks.  The random numbers are drawn on rank 0 and broadcast.  No host synchronisation inside the loop.

        Weighted (w: this rank's (n,) fp32 weights): the first centre is choice(n, p=w/sum(w)) over the weights of all ranks
        (all-gathered once), the potentials are sum_i w_i * closest_i (gfs_kmeans_pp_trial with the weights) and the candidates
        come from the cumulative sum of w * closest; `closest` itself stays unweighted, as in sklearn."""
        D = Xc.shape[1]
        n = Xc.shape[0] if n is None else n
        K = self.n_clusters
        trials = 2 + int(np.log(K))
        if trials > 8:
            raise NotImplementedError(f"k-means++ with {trials} local trials (n_clusters={K}) is not built")
        dev = Xc.device
        world, rank = self._world()
        sizes = self._gather_sizes(n, dev)
        n_tot, lo = sum(sizes), sum(sizes[:rank])
        # the random stream (rank 0's generator; the other ranks receive the draws)
        draws = torch.empty(1 + (K - 1) * trials, dtype=torch.float64)
        wall = self._gather_weights(w, sizes) if w is not None else None
        if rank == 0:
            wa = wall if wall is not None else np.ones(n_tot, dtype=np.float32)
            draws[0] = float(rng.choice(n_tot, p=wa / wa.sum()))
            draws[1:] = torch.from_numpy(rng.uniform(size=(K - 1) * trials)) if K > 1 else draws[1:]
        draws = self._broadcast0(draws.to(dev))
        U = draws[1:].view(K - 1, trials)
        npad = xt.shape[1]
        xsq = torch.zeros(npad, dtype=torch.float64, device=dev)
        xsq[:n] = (Xc[:n].double() ** 2).sum(1)
        centers = torch.empty(K, D, dtype=torch.float32, device=dev)
        m = torch.empty(8, npad, dtype=torch.float32, device=dev)
        pots = torch.zeros(8, dtype=torch.float64, device=dev)
        first = draws[0].long() - lo
        centers[0] = self._owned_rows(Xc, n, first.view(1), ((first >= 0) & (first < n)).view(1))[0]
        ops.kmeans_pp_trial(xt, n, xsq, centers[0:1].contiguous(), None, m, pots, weights=w)
        if world > 1:
            _dist().all_reduce(pots, group=self.process_group)
        closest, pot = m[0].clone(), pots[0].clone()
        for c in range(1, K):
            # this rank's slice of the global cumulative sum (of w * closest when weighted: an exact fp64 product), minus P[rank]
            cs = torch.cumsum(closest[:n].double() if w is None else closest[:n].double() * w.double(), 0)
            tots = cs[-1:].contiguous()
            if world > 1:
                gathered = [torch.empty_like(tots) for _ in range(world)]
                _dist().all_gather(gathered, tots, group=self.process_group)
                tots = torch.cat(gathered)
            P = torch.cumsum(tots, 0)                              # identical on every rank: ownership is decided from the same numbers
            rv = U[c - 1] * pot
            owner = torch.searchsorted(P, rv).clamp_max(world - 1)  # first rank whose slice reaches rv (the last one if none: numpy's clip)
            mine = owner == rank
            pos = torch.searchsorted(cs, rv - (P[rank] - tots[rank])).clamp_max(n - 1)   # first i with cumsum[i] >= rv (side='left')
            cand = self._owned_rows(Xc, n, pos, mine)
            pots.zero_()
            ops.kmeans_pp_trial(xt, n, xsq, cand, closest, m, pots, weights=w)
            if world > 1:
                _dist().all_reduce(pots, group=self.process_group)
            best = torch.argmin(pots[:trials]).view(1)
            pot = pots.index_select(0, best)[0]
            closest = m.index_select(0, best)[0]
            centers[c] = cand.index_select(0, best)[0]
        return centers

    # ------------------------------------------------------------------ fit
    def _check_weight(self, sample_weight, n):
        """sklearn's _check_sample_weight(..., dtype=float32) plus the checks its seeding relies on; runs before the data
        touch the device.  -> None, or the (n,) float32 weights as a CPU or CUDA tensor (a CUDA tensor stays where it is)"""
        if sample_weight is None:
            return None
        if isinstance(sample_weight, torch.Tensor):
            w = sample_weight.detach().to(torch.float32)
        else:
            w = torch.from_numpy(np.ascontiguousarray(np.asarray(sample_weight, dtype=np.float32)))
        if tuple(w.shape) != (n,):
            raise ValueError(f"sample_weight has shape {tuple(w.shape)}, expected ({n},)")
        if not bool(torch.isfinite(w).all()):
            raise ValueError("sample_weight must be finite")
        if bool((w < 0).any()):
            raise ValueError("sample_weight must be non-negative")
        if not self.shard and not bool((w > 0).any()):
            raise ValueError("sample_weight must contain at least one positive entry")
        return w.contiguous()

    def _n_runs(self):
        """sklearn _kmeans.py:_check_params_vs_input: 'auto' is 10 runs for init='random', else 1; an array init runs once"""
        array_init = isinstance(self.init, (np.ndarray, torch.Tensor))
        if self.n_init == "auto":
            runs = 10 if (isinstance(self.init, str) and self.init == "random") else 1
        else:
            runs = int(self.n_init)
            if runs < 1:
                raise ValueError(f"n_init={self.n_init!r} must be 'auto' or a positive integer")
        if array_init and runs != 1:
            warnings.warn(f"Explicit initial center position passed: performing only one init in KMeans instead of n_init={runs}.",
                          RuntimeWarning, stacklevel=3)
            runs = 1
        return runs

    def _as_device(self, X, dev):
        if isinstance(X, np.ndarray):
            return torch.from_numpy(np.ascontiguousarray(X, dtype=np.float32)).to(dev, non_blocking=True)
        return X.to(dev, torch.float32).contiguous()

    def fit(self, X, y=None, sample_weight=None):
        """sample_weight: None or (n,) non-negative finite weights (numpy or tensor), cast to float32; with shard=True, the
        weights of this rank's shard.  Mean-centring and the tolerance stay unweighted, as in sklearn."""
        w_in = self._check_weight(sample_weight, X.shape[0])
        K = self.n_clusters
        if K > 512:
            raise NotImplementedError(f"n_clusters={K} > 512 is not built")
        if K > 192 and X.shape[1] > 192:
            raise NotImplementedError(f"n_clusters={K} > 192 with {X.shape[1]} > 192 features is not built")
        dev = torch.device(self.device) if self.device is not None else torch.device("cuda", torch.cuda.current_device())
        Xd = self._as_device(X, dev)
        n, D = Xd.shape
        runs = self._n_runs()
        w = w_in.to(dev) if w_in is not None else None
        if w is not None and self.shard:
            wtot = w.double().sum().view(1)
            self._allreduce(wtot)
            if not float(wtot) > 0:
                raise ValueError("sample_weight must contain at least one positive entry")

        # mean-centring and tolerance (global over all shards)
        stat = torch.cat([Xd.double().sum(0), (Xd.double() ** 2).sum(0), torch.tensor([float(n)], dtype=torch.float64, device=dev)])
        self._allreduce(stat)
        n_tot = float(stat[-1])
        mean = (stat[:D] / n_tot)
        var = stat[D:2 * D] / n_tot - mean ** 2
        tol_abs = float(var.mean()) * self.tol
        mean32 = mean.float()
        Xc = Xd - mean32
        npad = (n + 3) // 4 * 4
        xt = torch.zeros(self._e_channels(D), npad, dtype=torch.float32, device=dev)   # E-step copy; xt[:D] is the data
        xt[:D, :n] = Xc.t()

        rng = self._rng() if isinstance(self.init, str) else None
        best = None
        for _ in range(runs):
            # initial centres
            if isinstance(self.init, str) and self.init == "k-means++":
                centers = self._seed_plusplus(Xc, xt[:D], rng, n, w=w)
            elif isinstance(self.init, str) and self.init == "random":
                centers = self._seed_random(Xc, rng, n, w=w)
            elif isinstance(self.init, (np.ndarray, torch.Tensor)):
                centers = torch.as_tensor(self.init, dtype=torch.float32).to(dev) - mean32
                if centers.shape != (K, D):
                    raise ValueError(f"init has shape {tuple(centers.shape)}, expected {(K, D)}")
            else:
                raise NotImplementedError(f"init={self.init!r} is not built")
            labels, centers, n_iter, lloyd_ms = self._lloyd(Xc, xt, n, centers.contiguous(), w, tol_abs)
            inertia = self._allreduce(ops.kmeans_inertia(Xc, labels, centers, w, n_valid=n))
            inertia = float(inertia)
            # sklearn _kmeans.py:1534-1538: a later run wins only with a lower inertia AND a different partition
            if best is None or (inertia < best[0] and not self._same_clustering(labels[:n], best[1][:n])):
                best = (inertia, labels, centers, n_iter, lloyd_ms)

        inertia, labels, centers, n_iter, lloyd_ms = best
        self.labels_ = labels[:n].cpu().numpy().astype(np.int32)
        self.lloyd_ms_ = lloyd_ms
        self.labels_device_ = labels[:n]
        self.cluster_centers_ = (centers + mean32).cpu().numpy()
        self.inertia_ = inertia
        self.n_iter_ = n_iter
        self.n_features_in_ = D
        self.mean_device_ = mean32                      # predict centres new data with the fit's fp32 mean ...
        self.centers_centered_ = centers               # ... against these: cluster_centers_ - mean does not round back to them
        return self

    def _e_channels(self, D):
        """channels of the E-step's channel-major copies: D, or D padded with zeros to a multiple of 64 for the panelled
        tensor-core path (n_clusters > 192)"""
        return (D + 63) // 64 * 64 if self.n_clusters > 192 else D

    def _same_clustering(self, a, b):
        """sklearn _k_means_common.pyx:_is_same_clustering (every label of a maps to one label of b), over all shards"""
        K = self.n_clusters
        pairs = torch.bincount(a.long() * K + b.long(), minlength=K * K).view(K, K)
        self._allreduce(pairs)
        return bool(((pairs > 0).sum(1) <= 1).all())

    def _lloyd(self, Xc, xt, n, centers, w, tol_abs):
        """one Lloyd run from the (centred) initial centres -> (labels (npad) int32, centres (K, D), n_iter, Lloyd ms)"""
        K, D = self.n_clusters, Xc.shape[1]
        dev = Xc.device
        npad = xt.shape[1]
        # Lloyd iterations.  Per iteration: E-step (4 launches), M-step sums (2), pack (1), ONE collective of the packed
        # [sums | weight sums | labels changed] buffer when sharded, centre update (1) and ONE device->host read of
        # (labels changed, centre shift, empty clusters).  All buffers are allocated once.  Unweighted, the weight sums are
        # the counts, which pack copies into their slot; weighted, the M-step writes them there.
        Kp = (K + 3) // 4 * 4
        ct = torch.zeros(xt.shape[0], Kp, dtype=torch.float32, device=dev)
        ct[:D, :K] = centers.t()
        centers = centers.contiguous()
        centers_new = torch.empty_like(centers)
        labels_old = torch.full((npad,), -1, dtype=torch.int32, device=dev)
        packed = torch.empty(K * D + K + 1, dtype=torch.float64, device=dev)
        sums, wsums = packed[:K * D].view(K, D), packed[K * D:K * D + K]
        if w is None:
            counts = torch.empty(K, dtype=torch.int64, device=dev)
            acc_ws = ops.kmeans_accumulate_workspace(K, D, dev)
        else:
            counts = None
            acc_ws = ops.kmeans_accumulate_weighted_workspace(K, D, dev)
        scratch = torch.zeros(2, dtype=torch.int64, device=dev)
        result = torch.empty(3, dtype=torch.float64, device=dev)
        # E-step over the channel-major copy: tensor-core product when the shape allows, same labels as the fp32 kernel.  (The
        # row-major entry, ops.kmeans_assign_rows, measured slower: 32 rows per load instruction instead of one 128-byte line.)
        assign = lambda: ops.kmeans_assign(xt, ct, K)
        strict = False
        n_iter = 0
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        ev0.record()
        for n_iter in range(1, self.max_iter + 1):
            labels = assign()                                          # ct holds the current centres, transposed
            if w is None:
                ops.kmeans_accumulate(Xc, labels, K, n_valid=n, sums=sums, counts=counts, ws=acc_ws)
            else:
                ops.kmeans_accumulate_weighted(Xc, labels, w, K, n_valid=n, sums=sums, wsums=wsums, ws=acc_ws)
            ops.kmeans_pack(labels, labels_old, n, K, D, packed, scratch, counts=counts)
            if self.shard:
                _dist().all_reduce(packed, group=self.process_group)
            ops.kmeans_update(packed, centers, K, D, Kp, centers_new, ct, result)
            n_changed, shift_h, n_empty = result.tolist()
            if n_empty > 0:           # rare: sklearn moves the empty clusters onto the points farthest from their centres
                gsums, gw = self._relocate_empty(Xc, n, labels, centers, sums.clone(), wsums.clone(), w)
                # clusters that are still empty keep the zero sum (sklearn _k_means_common.pyx:_average_centers)
                new = torch.where(gw[:, None] > 0, gsums / torch.where(gw > 0, gw, 1.0)[:, None], torch.zeros_like(gsums)).float()
                shift_h = float(((new - centers).double() ** 2).sum())
                centers_new.copy_(new)
                ct[:D, :K] = new.t()
            centers, centers_new = centers_new, centers
            if self.verbose:
                print(f"Iteration {n_iter - 1}, center shift {shift_h:.6g}")
            if n_changed == 0:
                strict = True
                break
            if shift_h <= tol_abs:
                break
            labels_old = labels
        ev1.record()
        if not strict:
            labels = assign()                                          # ct already holds the final centres
        torch.cuda.synchronize(dev)
        return labels, centers, n_iter, ev0.elapsed_time(ev1)

    def _relocate_empty(self, Xc, n, labels, centers, sums, wsums, w):
        """sklearn _k_means_common.pyx:167-211: every empty cluster (weight sum 0) is moved onto one of the points farthest,
        by unweighted distance, from its own (old) centre, and that point is taken out of its old cluster: sums[old] -= w x,
        sums[e] = w x (an fp32 product, as sklearn), wsums[e] = w, wsums[old] -= w.  w None: unit weights, for which these
        are the counts' updates.  Rare path, plain device ops.  Sharded: each rank offers its n_empty farthest points
        (distance, old label, weight, coordinates), the candidates are all-gathered and every rank applies the same global
        choice to the (already all-reduced) sums / weight sums."""
        empty = (wsums == 0).nonzero().flatten()
        ne = int(empty.numel())
        D = Xc.shape[1]
        dist = ((Xc - centers[labels[:n].long()]) ** 2).sum(1)
        m = min(ne, n)
        vals, idxs = torch.topk(dist, m)
        cand = torch.full((ne, 3 + D), float("-inf"), dtype=torch.float64, device=Xc.device)
        cand[:m, 0] = vals.double()
        cand[:m, 1] = labels[idxs].double()
        cand[:m, 2] = w[idxs].double() if w is not None else 1.0
        cand[:m, 3:] = Xc[idxs].double()
        if self.shard:
            world = _dist().get_world_size(self.process_group)
            gathered = [torch.empty_like(cand) for _ in range(world)]
            _dist().all_gather(gathered, cand, group=self.process_group)
            cand = torch.cat(gathered, 0)
        if float(cand[:, 0].max()) <= 0:
            return sums, wsums
        order = torch.argsort(cand[:, 0], descending=True, stable=True)[:ne]
        for e, row in zip(empty.tolist(), order.tolist()):
            old = int(cand[row, 1])
            wx = (cand[row, 3:].float() * cand[row, 2].float()).double()
            sums[old] -= wx
            sums[e] = wx
            wsums[e] = cand[row, 2]
            wsums[old] -= cand[row, 2]
        return sums, wsums

    def fit_predict(self, X, y=None, sample_weight=None):
        return self.fit(X, sample_weight=sample_weight).labels_

    # ------------------------------------------------------------------ fitted-model queries
    def _fitted_device(self):
        if not hasattr(self, "centers_centered_"):
            raise RuntimeError("this KMeans instance is not fitted yet: call fit first")
        return self.centers_centered_.device

    @staticmethod
    def _like_input(X, t):
        """numpy in -> numpy out, tensor in -> tensor on the input's device"""
        return t.to(X.device) if isinstance(X, torch.Tensor) else t.cpu().numpy()

    def _predict_device(self, X):
        dev = self._fitted_device()
        Xc = self._as_device(X, dev) - self.mean_device_
        n, D = Xc.shape
        if D != self.n_features_in_:
            raise ValueError(f"X has {D} features, the model was fitted with {self.n_features_in_}")
        K = self.n_clusters
        De = self._e_channels(D)
        xt = torch.zeros(De, (n + 3) // 4 * 4, dtype=torch.float32, device=dev)
        xt[:D, :n] = Xc.t()
        ct = torch.zeros(De, (K + 3) // 4 * 4, dtype=torch.float32, device=dev)
        ct[:D, :K] = self.centers_centered_.t()
        return Xc.contiguous(), ops.kmeans_assign(xt, ct, K)[:n]

    def predict(self, X):
        """nearest centre of each row: X is centred with the fit's fp32 mean and labelled by the pinned E-step against the
        fit's centred fp32 centres (labels defined bit for bit by oracle.kmeans_assign_exact on the centred data)"""
        return self._like_input(X, self._predict_device(X)[1])

    def transform(self, X):
        """(n, K) Euclidean distances to cluster_centers_ on the uncentred data, as sklearn's euclidean_distances evaluates
        float32 input: (|x|^2 - 2 x.c) + |c|^2 in fp64, one rounding to fp32, a clip at 0, an fp32 sqrt.  Runs
        gfs_kmeans_pp_trial (closest = NULL) over groups of 8 centres."""
        dev = self._fitted_device()
        Xd = self._as_device(X, dev)
        n, D = Xd.shape
        if D != self.n_features_in_:
            raise ValueError(f"X has {D} features, the model was fitted with {self.n_features_in_}")
        K = self.n_clusters
        npad = (n + 3) // 4 * 4
        xt = torch.zeros(D, npad, dtype=torch.float32, device=dev)
        xt[:, :n] = Xd.t()
        xsq = (Xd.double() ** 2).sum(1)
        C = torch.from_numpy(np.ascontiguousarray(self.cluster_centers_, dtype=np.float32)).to(dev)
        m = torch.empty(8, npad, dtype=torch.float32, device=dev)
        pots = torch.zeros(8, dtype=torch.float64, device=dev)
        out = torch.empty(n, K, dtype=torch.float32, device=dev)
        for g in range(0, K, 8):
            T = min(8, K - g)
            ops.kmeans_pp_trial(xt, n, xsq, C[g:g + T].contiguous(), None, m, pots)
            out[:, g:g + T] = m[:T, :n].t()
        return self._like_input(X, torch.sqrt(out))

    def fit_transform(self, X, y=None, sample_weight=None):
        return self.fit(X, sample_weight=sample_weight).transform(X)

    def score(self, X, y=None, sample_weight=None):
        """-inertia of predict(X) on X (centred as in predict), weighted by sample_weight"""
        w = self._check_weight(sample_weight, X.shape[0])
        Xc, labels = self._predict_device(X)
        if w is not None:
            w = w.to(Xc.device)
        return -float(ops.kmeans_inertia(Xc, labels, self.centers_centered_, w))
