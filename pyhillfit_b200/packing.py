"""Dataset packer: reference-shaped inputs -> the packed device layouts of include/pyhillfit_b200.h.

Single-level: (concs, responses, masks) as built at python/PyHillFit.py:661-677 / python/PyHillTemp.py:132-140
become one phf_dose_group per unique dose (sufficient statistics of the replicates) and one phf_dataset.
Hierarchical: the list of per-experiment arrays from dr.load_crumb_data (python/doseresponse.py:60-67)
becomes one phf_hier_point per measurement.  Statistics are accumulated in extended precision on the host
so that the compressed likelihood agrees with the reference's per-point sum to ~1 ulp.
"""
import numpy as np

from . import _lib

_LD = np.longdouble
_EXTENDED = np.finfo(_LD).nmant >= 63


def _ln_hi_lo(c):
    """ln(c) as a double-double (hi, lo)."""
    c = float(c)
    if c == 0.0:
        return -np.inf, 0.0
    if c < 0 or not np.isfinite(c):
        raise ValueError("dose must be finite and >= 0, got %r" % c)
    if _EXTENDED:
        full = np.log(_LD(c))
        hi = np.float64(full)
        lo = np.float64(full - _LD(hi))
    else:  # pragma: no cover - non-x86 hosts
        import mpmath
        mpmath.mp.prec = 120
        full = mpmath.log(mpmath.mpf(c))
        hi = np.float64(float(full))
        lo = np.float64(float(full - mpmath.mpf(float(hi))))
    return float(hi), float(lo)


_ln_cache = {}


def ln_hi_lo(c):
    c = float(c)
    v = _ln_cache.get(c)
    if v is None:
        v = _ln_cache[c] = _ln_hi_lo(c)
    return v


def masks(responses):
    """The three reference masks (PyHillFit.py:675-677); a response outside [0,100] is in none."""
    r = np.asarray(responses, dtype=np.float64)
    return r == 0, r == 100, (0 < r) & (r < 100)


def pack_single_one(concs, responses, where_0=None, where_100=None, where_other=None, pi_bit=None):
    """-> (groups[D] structured array, pi_bit, n_other_total)."""
    concs = np.asarray(concs, dtype=np.float64).ravel()
    y = np.asarray(responses, dtype=np.float64).ravel()
    if concs.shape != y.shape:
        raise ValueError("concs and responses differ in length")
    if where_0 is None:
        where_0, where_100, where_other = masks(y)
    where_0 = np.asarray(where_0, dtype=bool)
    where_100 = np.asarray(where_100, dtype=bool)
    where_other = np.asarray(where_other, dtype=bool)
    if pi_bit is None:  # doseresponse.py:299-301 called with the mask -> N_total
        pi_bit = 0.5 * len(where_other) * np.log(2 * np.pi)
    uniq = []
    seen = {}
    for cval in concs:  # order of first appearance
        if cval not in seen:
            seen[cval] = len(uniq)
            uniq.append(cval)
    g = np.zeros(len(uniq), dtype=_lib.DOSE_GROUP_DTYPE)
    for k, cval in enumerate(uniq):
        m = concs == cval
        yo = y[m & where_other].astype(_LD)
        hi, lo = ln_hi_lo(cval)
        g["lnc_hi"][k], g["lnc_lo"][k], g["conc"][k] = hi, lo, cval
        g["n_other"][k] = len(yo)
        if len(yo):
            ybar = yo.sum() / _LD(len(yo))
            g["ybar"][k] = np.float64(ybar)
            # centre on the *rounded* mean so that ss + n (ybar - p)^2 is the exact expansion
            yb = _LD(np.float64(ybar))
            g["ss"][k] = np.float64(((yo - yb) ** 2).sum())
            # first-order term 2 (ybar_r - p) sum(y - ybar_r) is < n ulp(ybar) |ybar - p|: below double rounding
        g["n0"][k] = np.count_nonzero(m & where_0)
        g["n100"][k] = np.count_nonzero(m & where_100)
    return g, float(pi_bit), float(np.count_nonzero(where_other))


POINT_ZERO, POINT_HUNDRED, POINT_OTHER, POINT_NONE = 0, 1, 2, 3


def point_kinds(where_0, where_100, where_other):
    """phf_point.kind of each point from the three masks (the reference builds them disjoint; a point in none of them
    is POINT_NONE)."""
    k = np.full(np.shape(where_0), POINT_NONE, dtype=np.int32)
    k[np.asarray(where_other, dtype=bool)] = POINT_OTHER
    k[np.asarray(where_100, dtype=bool)] = POINT_HUNDRED
    k[np.asarray(where_0, dtype=bool)] = POINT_ZERO
    return k


def point_list(concs, responses, where_0=None, where_100=None, where_other=None):
    """-> phf_point records [N] of one dataset, in the order of its responses; `group` is the index of the point's dose
    among the dataset's dose groups as pack_single_one orders them (order of first appearance)."""
    concs = np.asarray(concs, dtype=np.float64).ravel()
    y = np.asarray(responses, dtype=np.float64).ravel()
    if where_0 is None:
        where_0, where_100, where_other = masks(y)
    index = {}
    for cval in concs:
        index.setdefault(cval, len(index))
    pts = np.zeros(len(y), dtype=_lib.POINT_DTYPE)
    pts["group"] = [index[cval] for cval in concs]
    pts["kind"] = point_kinds(where_0, where_100, where_other)
    pts["y"] = y
    return pts


class SinglePack:
    """Packed single-level datasets, host copies plus (lazily) device tensors."""

    def __init__(self, items):
        """items: iterable of (concs, responses) or dicts with optional masks / pi_bit."""
        groups, ds, points = [], [], []
        begin = 0
        for it in items:
            kw = dict(it) if isinstance(it, dict) else dict(zip(("concs", "responses", "where_0", "where_100",
                                                                 "where_other", "pi_bit"), it))
            g, pb, no = pack_single_one(**kw)
            kw.pop("pi_bit", None)
            pts = point_list(**kw)
            pts["group"] += begin
            groups.append(g)
            points.append(pts)
            ds.append((begin, len(g), pb, no, 0.0))
            begin += len(g)
        self.groups = np.concatenate(groups) if groups else np.zeros(0, dtype=_lib.DOSE_GROUP_DTYPE)
        self.datasets = np.array(ds, dtype=_lib.DATASET_DTYPE)
        self.points = np.concatenate(points) if points else np.zeros(0, dtype=_lib.POINT_DTYPE)
        self.point_offsets = np.concatenate(([0], np.cumsum([len(p) for p in points], dtype=np.int64))).astype(np.int64)
        self._dev = {}

    @classmethod
    def from_uniform(cls, concs, responses):
        """Vectorised packer for many datasets that share one dose design (the synthetic scale-up, BASELINE
        config 5): concs [N], responses [n_datasets, N].  Same statistics as pack_single_one, computed for all
        datasets at once in extended precision."""
        concs = np.asarray(concs, dtype=np.float64).ravel()
        Y = np.atleast_2d(np.asarray(responses, dtype=np.float64))
        if Y.shape[1] != len(concs):
            raise ValueError("responses must be [n_datasets, len(concs)]")
        n_ds = Y.shape[0]
        uniq = []
        for cval in concs:
            if cval not in uniq:
                uniq.append(cval)
        D = len(uniq)
        g = np.zeros((n_ds, D), dtype=_lib.DOSE_GROUP_DTYPE)
        w0, w100, wo = masks(Y)
        for k, cval in enumerate(uniq):
            cols = np.nonzero(concs == cval)[0]
            hi, lo = ln_hi_lo(cval)
            g["lnc_hi"][:, k], g["lnc_lo"][:, k], g["conc"][:, k] = hi, lo, cval
            yo = Y[:, cols].astype(_LD)
            m = wo[:, cols]
            cnt = m.sum(axis=1)
            ybar = np.where(cnt > 0, (yo * m).sum(axis=1) / np.maximum(cnt, 1), 0)
            yb = ybar.astype(np.float64).astype(_LD)      # centre on the rounded mean (see pack_single_one)
            g["n_other"][:, k] = cnt
            g["ybar"][:, k] = ybar.astype(np.float64)
            g["ss"][:, k] = ((((yo - yb[:, None]) ** 2) * m).sum(axis=1)).astype(np.float64)
            g["n0"][:, k] = w0[:, cols].sum(axis=1)
            g["n100"][:, k] = w100[:, cols].sum(axis=1)
        self = cls([])
        self.groups = g.reshape(-1)
        ds = np.zeros(n_ds, dtype=_lib.DATASET_DTYPE)
        ds["group_begin"] = np.arange(n_ds, dtype=np.int64) * D
        ds["n_groups"] = D
        ds["pi_bit"] = 0.5 * len(concs) * np.log(2 * np.pi)
        ds["n_other_total"] = wo.sum(axis=1)
        self.datasets = ds
        # point list: dataset k's points in column order, each pointing at its dose's group
        first = np.array([uniq.index(cval) for cval in concs], dtype=np.int32)
        pts = np.zeros((n_ds, len(concs)), dtype=_lib.POINT_DTYPE)
        pts["group"] = np.arange(n_ds, dtype=np.int32)[:, None] * D + first[None, :]
        pts["kind"] = point_kinds(w0, w100, wo)
        pts["y"] = Y
        self.points = pts.reshape(-1)
        self.point_offsets = np.arange(n_ds + 1, dtype=np.int64) * len(concs)
        return self

    @property
    def n_datasets(self):
        return len(self.datasets)

    def device(self, device=None):
        torch = _lib.require_cuda()
        device = torch.device("cuda", torch.cuda.current_device()) if device is None else torch.device(device)
        key = str(device)
        if key not in self._dev:
            g = torch.from_numpy(self.groups.view(np.float64).reshape(-1, 8).copy()).to(device)
            d = torch.from_numpy(self.datasets.view(np.uint8).reshape(-1, 32).copy()).to(device)
            self._dev[key] = (d, g)
        return self._dev[key]

    def points_device(self, device=None):
        """The point list as a device tensor (16-byte phf_point records, viewed as int64 pairs)."""
        torch = _lib.require_cuda()
        device = torch.device("cuda", torch.cuda.current_device()) if device is None else torch.device(device)
        key = "points:" + str(device)
        if key not in self._dev:
            self._dev[key] = torch.from_numpy(self.points.view(np.int64).reshape(-1, 2).copy()).to(device)
        return self._dev[key]

    def dataset_cost(self, model=2):
        """Relative cost of one adaptive-Metropolis iteration per dataset (SURVEY.md section 8d's cost table: a Hill
        curve per unique dose, an erfcx + log per censored dose, plus the fixed proposal / accept / adapt work) --
        the weight ranks are balanced by when a chain list is sharded (dist.shard_bounds)."""
        gb, ng = self.datasets["group_begin"].astype(np.int64), self.datasets["n_groups"].astype(np.int64)
        cens = ((self.groups["n0"] > 0).astype(np.float64) + (self.groups["n100"] > 0)).cumsum()
        cens = np.concatenate(([0.0], cens))
        n_cens = cens[gb + ng] - cens[gb]
        fixed = 560.0 if model == 2 else 470.0
        return fixed + 58.0 * ng + 133.0 * n_cens

    def stage_groups_needed(self, dataset_id, block_threads):
        """max over CTAs of the contiguous dose-group range they touch (chains sorted by dataset)."""
        ids = np.asarray(dataset_id)
        if len(ids) == 0:
            return 0
        lo = ids[::block_threads]
        hi = ids[np.minimum(np.arange(block_threads - 1, len(ids) + block_threads - 1, block_threads), len(ids) - 1)]
        gb = self.datasets["group_begin"]
        ng = self.datasets["n_groups"]
        return int(np.max(gb[hi] + ng[hi] - gb[lo]))


def pack_hier_one(experiments):
    pts = []
    for e, arr in enumerate(experiments):
        arr = np.asarray(arr, dtype=np.float64)
        for cval, yval in arr:
            hi, lo = ln_hi_lo(cval)
            pts.append((hi, lo, yval, e, 0))
    return np.array(pts, dtype=_lib.HIER_POINT_DTYPE), len(experiments)


class HierPack:
    def __init__(self, experiment_lists):
        pts, ds = [], []
        begin = 0
        for ex in experiment_lists:
            p, ne = pack_hier_one(ex)
            pts.append(p)
            ds.append((begin, len(p), ne, 0))
            begin += len(p)
        self.points = np.concatenate(pts) if pts else np.zeros(0, dtype=_lib.HIER_POINT_DTYPE)
        self.datasets = np.array(ds, dtype=_lib.HIER_DATASET_DTYPE)
        self._dev = {}

    @property
    def n_datasets(self):
        return len(self.datasets)

    def device(self, device=None):
        torch = _lib.require_cuda()
        device = torch.device("cuda", torch.cuda.current_device()) if device is None else torch.device(device)
        key = str(device)
        if key not in self._dev:
            p = torch.from_numpy(self.points.view(np.uint8).reshape(-1, 32).copy()).to(device)
            d = torch.from_numpy(self.datasets.view(np.uint8).reshape(-1, 16).copy()).to(device)
            self._dev[key] = (d, p)
        return self._dev[key]
