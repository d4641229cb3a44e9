"""Host-side mirror of the reference's L1-L3 layers for the particle hot path, over the C ABI.

Reference (all under /root/reference/src):
  DeviceColumnStore  <- ColumnStore / AbstractParticleStore          stores.jl:28-35,70-111
  SMCState, run      <- SMCState, run!, advance!, score_logpdf        types.jl:48-78,120-126,183-206
  Assign ... Move    <- the ParticleTransformer subtypes + apply!/score!  transformers.jl
  Normal/MvNormal/Exponential, importance_kernel  <- default_kernels  default_kernels.jl:69-102
  RW, autoRW         <- proposals                                     move_kernels.jl:189-265

Every ``apply`` body is one C-ABI call; nothing here touches particle data on the host.  Python
is the host language because no Julia toolchain exists in the build image; ``julia/WSB200.jl`` is
the ``ccall`` shim with the same structure (INTEGRATION.md).
"""
from __future__ import annotations

import ctypes as C
import os
import math

import numpy as np

from . import _lib as L
from ._lib import UnsupportedModelError, WsError, check
from .expr import CExprs, Col, Const, Expr, NotAProbabilityVector, Tokens, lower, wrap

__all__ = [
    "DeviceColumnStore", "ColumnStore", "SMCState", "ParticleTransformer", "Assign", "AccessorAssign", "Sample",
    "AccessorSample", "Observe", "Weight", "Sequence", "Loop", "Cond", "Resample", "Move", "ScoreCtx", "apply",
    "score", "run", "score_logpdf", "marginal_diversity", "WeightedKernel", "Normal", "MvNormal", "Exponential",
    "importance_kernel", "default_kernels", "RW", "autoRW", "default_proposals", "nparticles", "hascol", "getcol",
    "colnames", "resample", "nccl_unique_id", "shard_bounds", "sharded_state",
]


def _unsupported(msg):
    return UnsupportedModelError(L.WS_EUNSUPPORTED, msg)


# --------------------------------------------------------------------------------------------------
# L1: particle store
# --------------------------------------------------------------------------------------------------
class DeviceColumnStore:
    """``ColumnStore`` whose columns are device-resident Float64 planes (stores.jl:70-111).

    ``getcol`` returns a host COPY (download); device-resident access is through statements.
    """

    def __init__(self, n, *, device=0, seed=0, ess_perc_min=0.5, resampler="stratified", rank=0, nranks=1, nccl_id=None):
        """``n`` is the GLOBAL particle count; with ``nranks > 1`` this rank owns the slots
        [rank*n/nranks, (rank+1)*n/nranks) and ``nccl_id`` is the 128-byte id from :func:`nccl_unique_id`."""
        lib = L.load()
        self._lib = lib
        self._ctx = C.c_void_p()
        if nranks > 1:
            if nccl_id is None or len(nccl_id) != 128:
                raise ValueError("a sharded state needs the 128-byte NCCL unique id created by rank 0")
            idbuf = C.create_string_buffer(bytes(nccl_id), 128)
            rc = lib.ws_create_sharded(C.byref(self._ctx), int(n), int(rank), int(nranks), idbuf, int(device),
                                       int(seed) & (2 ** 64 - 1), float(ess_perc_min), L.RESAMPLER[resampler])
        else:
            rc = lib.ws_create(C.byref(self._ctx), int(n), int(device), int(seed) & (2 ** 64 - 1), float(ess_perc_min),
                               L.RESAMPLER[resampler])
        if rc != 0:
            msg = lib.ws_last_error(None)
            raise WsError(rc, msg.decode() if msg else "")
        nl, ng = C.c_int64(), C.c_int64()
        check(self._ctx, lib.ws_n_particles(self._ctx, C.byref(nl), C.byref(ng)))
        self.n = nl.value           # local shard size: every host buffer of this store has this length
        self.n_global = ng.value
        self.rank, self.nranks = int(rank), int(nranks)

    # -- C-ABI plumbing ---------------------------------------------------------------------------
    def _call(self, name, *args):
        check(self._ctx, getattr(self._lib, name)(self._ctx, *args))

    def _lookup(self, name):
        cid, width = C.c_int32(), C.c_int32()
        self._call("ws_col_lookup", name.encode(), C.byref(cid), C.byref(width))
        return cid.value, width.value

    def _ensure(self, name, width):
        cid = C.c_int32()
        self._call("ws_col_ensure", name.encode(), int(width), C.byref(cid))
        return cid.value

    def _table_id(self, tab):
        """the context's id of a build-time table (uploaded on first use; ws_table deduplicates by content)"""
        ids = self.__dict__.setdefault("_tables", {})
        key = (tab.values.shape, tab.values.tobytes())
        if key not in ids:
            tid = C.c_int32()
            self._call("ws_table", tab.values.ctypes.data_as(C.c_void_p), int(tab.values.shape[0]), int(tab.values.shape[1]),
                       C.byref(tid))
            ids[key] = tid.value
        return ids[key]

    def _new_index_faults(self):
        """table index faults since the last call (0 without a call to the device when no table exists)"""
        if not self.__dict__.get("_tables"):
            return 0
        n = C.c_int64()
        self._call("ws_get_index_faults", C.byref(n))
        new, self._faults_seen = n.value - self.__dict__.get("_faults_seen", 0), n.value
        return new

    def close(self):
        if getattr(self, "_ctx", None) is not None and self._ctx:
            self._lib.ws_destroy(self._ctx)
            self._ctx = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # -- AbstractParticleStore interface (stores.jl:28-35) ----------------------------------------
    def nparticles(self):
        return self.n

    def hascol(self, name):
        return self._lookup(str(name))[0] >= 0

    def colnames(self):
        cnt = C.c_int32()
        self._call("ws_col_count", C.byref(cnt))
        out = []
        buf = C.create_string_buffer(256)
        for i in range(cnt.value):
            w = C.c_int32()
            self._call("ws_col_info", i, buf, 256, C.byref(w))
            out.append(buf.value.decode())
        return out

    def colwidth(self, name):
        return self._lookup(str(name))[1]

    def getcol(self, name):
        cid, width = self._lookup(str(name))
        if cid < 0:
            raise KeyError(name)
        out = np.empty((width, self.n), dtype=np.float64)
        self._call("ws_col_download", cid, out.ctypes.data_as(C.c_void_p))
        return out[0].copy() if width == 1 else np.ascontiguousarray(out.T)  # vector columns: (n, d)

    def setcol(self, name, values):
        """``broadcast_setcol!(store, name, identity, (values,))`` with host data (upload)."""
        v = np.asarray(values, dtype=np.float64)
        if v.ndim == 0:
            v = np.full(self.n, float(v))
        if v.ndim == 1:
            if v.shape[0] != self.n:
                raise ValueError(f"column length {v.shape[0]} != n_particles {self.n}")
            planes = np.ascontiguousarray(v[None, :])
        else:
            if v.shape[0] != self.n:
                raise ValueError(f"column length {v.shape[0]} != n_particles {self.n}")
            planes = np.ascontiguousarray(v.T)
        cid = self._ensure(str(name), planes.shape[0])
        self._call("ws_col_upload", cid, planes.ctypes.data_as(C.c_void_p))

    def resample(self, indices):
        """``resample!(store, indices)`` (stores.jl:105-111), 0-based indices."""
        idx = np.ascontiguousarray(indices, dtype=np.int32)
        if idx.shape != (self.n,):
            raise ValueError("indices must have one entry per particle")
        if idx.min() < 0 or idx.max() >= self.n:
            raise IndexError("ancestor index out of range")
        self._call("ws_gather", idx.ctypes.data_as(C.c_void_p))

    def __repr__(self):
        return f"ColumnStore(n={self.n}, columns={self.colnames()})"


ColumnStore = DeviceColumnStore


def nccl_unique_id():
    """128-byte ncclUniqueId (create on rank 0, hand to every rank's SMCState)."""
    buf = C.create_string_buffer(128)
    rc = L.load().ws_nccl_unique_id(buf)
    if rc != 0:
        msg = L.load().ws_last_error(None)
        raise WsError(rc, msg.decode() if msg else "")
    return buf.raw


def shard_bounds(n_global, rank, nranks):
    """global slot range [lo, hi) owned by ``rank`` (same arithmetic as ws_create_sharded)."""
    return (n_global * rank) // nranks, (n_global * (rank + 1)) // nranks


def sharded_state(n_global, *, make_id=nccl_unique_id, **kw):
    """SMCState sharded over the ranks of an initialised ``torch.distributed`` process group (one rank per
    GPU): rank 0 creates the NCCL id, it is broadcast as an object, every rank builds its shard."""
    import torch.distributed as dist
    rank, world = dist.get_rank(), dist.get_world_size()
    box = [make_id() if rank == 0 else None]
    dist.broadcast_object_list(box, src=0)
    return SMCState(n_global, rank=rank, nranks=world, nccl_id=box[0], **kw)


def nparticles(store): return store.nparticles()
def hascol(store, name): return store.hascol(name)
def getcol(store, name): return store.getcol(name)
def colnames(store): return store.colnames()
def resample(store, indices): return store.resample(indices)


# --------------------------------------------------------------------------------------------------
# SMCState
# --------------------------------------------------------------------------------------------------
class SMCState:
    """``SMCState(n; ess_perc_min=0.5)`` (types.jl:48-78).  Weights, flags and depth live in the C
    context; the attributes below read / write them."""

    def __init__(self, n_or_store, *, ess_perc_min=0.5, seed=0, device=0, resampler="stratified", show_progress=False,
                 rank=0, nranks=1, nccl_id=None):
        if isinstance(n_or_store, DeviceColumnStore):
            self.store = n_or_store
            self.store._call("ws_set_ess_perc_min", float(ess_perc_min))
        else:
            self.store = DeviceColumnStore(int(n_or_store), device=device, seed=seed, ess_perc_min=ess_perc_min,
                                           resampler=resampler, rank=rank, nranks=nranks, nccl_id=nccl_id)
        self._root = None
        self._tape_valid = True  # the recorded tape is the score! walk of `root` up to `depth`
        self.record_tape = True
        self.show_progress = show_progress

    # flags ----------------------------------------------------------------------------------------
    def _flags(self):
        r, w, d = C.c_int(), C.c_int(), C.c_int64()
        self.store._call("ws_get_flags", C.byref(r), C.byref(w), C.byref(d))
        return bool(r.value), bool(w.value), d.value

    @property
    def resampled(self): return self._flags()[0]

    @resampled.setter
    def resampled(self, v): self.store._call("ws_set_flags", int(bool(v)), int(self._flags()[1]))

    @property
    def weights_changed(self):
        w = C.c_int()
        self.store._call("ws_get_flags", None, C.byref(w), None)   # (asking for `resampled` would wait for pending Resample steps)
        return bool(w.value)

    @weights_changed.setter
    def weights_changed(self, v): self.store._call("ws_set_flags", int(self._flags()[0]), int(bool(v)))

    @property
    def depth(self):
        d = C.c_int64()
        self.store._call("ws_get_flags", None, None, C.byref(d))
        return d.value

    @depth.setter
    def depth(self, v):
        self.store._call("ws_set_depth", int(v))
        self._tape_valid = False

    @property
    def root(self): return self._root

    @root.setter
    def root(self, t):
        self._root = t
        self._tape_valid = False

    @property
    def ess_perc_min(self):
        v = C.c_double()
        self.store._call("ws_get_ess_perc_min", C.byref(v))
        return v.value

    @ess_perc_min.setter
    def ess_perc_min(self, v): self.store._call("ws_set_ess_perc_min", float(v))

    @property
    def weights(self):
        out = np.empty(self.store.n, dtype=np.float64)
        self.store._call("ws_weights_download", out.ctypes.data_as(C.c_void_p))
        return out

    @weights.setter
    def weights(self, v):
        a = np.ascontiguousarray(v, dtype=np.float64)
        if a.shape != (self.store.n,):
            raise ValueError("weights must have one entry per particle")
        self.store._call("ws_weights_upload", a.ctypes.data_as(C.c_void_p), 0)

    def __getitem__(self, name):
        return self.store.getcol(name)

    def sync(self):
        self.store._call("ws_sync")

    # replay hooks (parity tests) -------------------------------------------------------------------
    def set_replay(self, normals=None, uniforms=None, exponentials=None, variates=None):
        for arr, fn in ((normals, "ws_set_replay_normals"), (uniforms, "ws_set_replay_uniforms"),
                        (exponentials, "ws_set_replay_exponentials"), (variates, "ws_set_replay_variates")):
            if arr is None:
                self.store._call(fn, None, 0)
            else:
                a = np.ascontiguousarray(arr, dtype=np.float64)
                self.store._call(fn, a.ctypes.data_as(C.c_void_p), a.size)

    def stats(self):
        s = L.ws_stats()
        self.store._call("ws_get_stats", C.byref(s))
        return {f: getattr(s, f) for f, _ in L.ws_stats._fields_}

    def ess_ties(self):
        """Resample steps decided on a knife edge (ESS% == ess_perc_min to a few ulp; see ws_get_ess_ties)."""
        v = C.c_int64()
        self.store._call("ws_get_ess_ties", C.byref(v))
        return v.value

    def genealogy(self):
        """Retained per-event ancestor vectors (DESIGN.md: trajectory storage by genealogy)."""
        nv, nb, ev = C.c_int64(), C.c_int64(), C.c_int64()
        self.store._call("ws_genealogy_info", C.byref(nv), C.byref(nb), C.byref(ev))
        return {"vectors": nv.value, "bytes": nb.value, "events": ev.value}

    def set_genealogy(self, on=True, budget_bytes=0):
        self.store._call("ws_set_genealogy", int(bool(on)), int(budget_bytes))

    def kernel_times(self):
        ms = (C.c_double * 8)()
        cnt = (C.c_int64 * 8)()
        self.store._call("ws_kernel_times", ms, cnt, 8)
        return {k: {"ms": ms[i], "launches": cnt[i]} for i, k in enumerate(L.KERNEL_CLASSES)}

    def __repr__(self):
        return f"SMCState(n_particles={self.store.n}, columns={self.store.colnames()})"

    def describe_state(self):
        r, _, d = self._flags()
        return ("SMCState\n  n_particles:  %d\n  columns:      %s\n  ess_perc_min: %s\n  resampled:    %s\n"
                "  depth:        %d" % (self.store.n, self.store.colnames(), self.ess_perc_min, str(r).lower(), d))


# --------------------------------------------------------------------------------------------------
# kernels (the device kernel table; default_kernels.jl)
# --------------------------------------------------------------------------------------------------
def _scalar(tok, what):
    if isinstance(tok, list):
        raise _unsupported(f"{what} must be scalar-valued")
    return tok


def _target(store, lhs, width, create=True):
    """lhs is a column name or (name, j) for an accessor target ``x[j]`` (0-based)."""
    if isinstance(lhs, tuple):
        name, j = lhs
        cid, w = store._lookup(str(name))
        if cid < 0:
            raise KeyError(f"column {name!r} must exist before an accessor write")  # AccessorSample docstring
        if not (0 <= int(j) < w):
            raise IndexError(f"index {j} out of range for column {name!r} of width {w}")
        return cid, int(j)
    cid, w = store._lookup(str(lhs))
    if cid < 0:
        if not create:
            raise KeyError(lhs)
        cid = store._ensure(str(lhs), width)
    elif w != width:
        raise _unsupported(f"column {lhs!r} has width {w}; re-assigning it with width {width} would change its element type")
    return cid, 0


class WeightedKernel:
    """``WeightedKernel(sampler, weighter, logpdf)`` (types.jl:226-230) whose three parts are DEVICE EXPRESSIONS:
    Python callables over particle expressions, traced once per statement and lowered to micro-ops.

    - ``sampler(args...) -> x``: may use fresh variates ``randn()``, ``randu()``, ``randexp()``;
    - ``weighter(args..., x) -> log_weight`` or ``None`` (uniform weights);
    - ``logpdf(args..., x) -> log_density``.
    A callable that cannot be traced (it branches on a particle value, calls NumPy on it, ...) raises
    ``UnsupportedModelError``: nothing ever runs on the host."""

    name = "WeightedKernel"
    has_weighter = False

    def __init__(self, sampler=None, weighter=None, logpdf=None, name=None):
        self.sampler, self.weighter, self.logpdf = sampler, weighter, logpdf
        self.has_weighter = weighter is not None
        if name is not None:
            self.name = name

    def _trace(self, fn, args, what):
        try:
            out = fn(*args)
        except (UnsupportedModelError, NotAProbabilityVector):
            raise
        except Exception as e:  # e.g. math.exp(Expr), float(Expr)
            raise _unsupported(f"{self.name}.{what} is not a device expression ({type(e).__name__}: {e})")
        return out

    def sample(self, state, lhs, args):
        if self.sampler is None:
            raise _unsupported(f"kernel {self.name} has no sampler (it can only be used with `_ ~` / `=>`)")
        st = state.store
        cid, comp = _target(st, lhs, 1)
        x_expr = self._trace(self.sampler, args, "sampler")
        xcol = Col(lhs[0])[lhs[1]] if isinstance(lhs, tuple) else Col(lhs)
        toks = [_scalar(lower(x_expr, st), "sampled value")]
        w_i = l_i = None
        if self.weighter is not None:
            w_i = len(toks)
            toks.append(_scalar(lower(self._trace(self.weighter, tuple(args) + (xcol,), "weighter"), st), "weighter"))
        if self.logpdf is not None:
            l_i = len(toks)
            toks.append(_scalar(lower(self._trace(self.logpdf, tuple(args) + (xcol,), "logpdf"), st), "logpdf"))
        ex = CExprs(toks)
        st._call("ws_sample_expr", cid, comp, ex.ptr(0), ex.ptr(w_i) if w_i is not None else None,
                 ex.ptr(l_i) if l_i is not None else None)

    def observe(self, state, value, args):
        if self.logpdf is None:
            raise _unsupported(f"kernel {self.name} has no logpdf")
        st = state.store
        tok = _scalar(lower(self._trace(self.logpdf, tuple(args) + (value,), "logpdf"), st), "logpdf")
        ex = CExprs([tok])
        st._call("ws_weight_expr", ex.ptr(0))

    def weight(self, state, args):
        """``Weight`` step: kernel.weighter(args...) (sampler must be None; check_weight_kernel, types.jl:243-249)."""
        if self.sampler is not None:
            raise ValueError("Weight kernel must have `sampler === nothing` (a `Weight` step never samples)")
        st = state.store
        tok = _scalar(lower(self._trace(self.weighter or self.logpdf, tuple(args), "weighter"), st), "weighter")
        ex = CExprs([tok])
        st._call("ws_weight_expr", ex.ptr(0))


class _Normal(WeightedKernel):
    name = "Normal"

    def sample(self, state, lhs, args):
        st = state.store
        mu, sigma = (_scalar(lower(a, st), "Normal argument") for a in args)
        cid, comp = _target(st, lhs, 1)
        ex = CExprs([mu, sigma])
        st._call("ws_sample_normal", cid, comp, ex.ptr(0), ex.ptr(1))

    def observe(self, state, value, args):
        st = state.store
        obs = _scalar(lower(value, st), "observed value")
        mu, sigma = (_scalar(lower(a, st), "Normal argument") for a in args)
        ex = CExprs([obs, mu, sigma])
        st._call("ws_observe_normal", ex.ptr(0), ex.ptr(1), ex.ptr(2))


class _Exponential(WeightedKernel):
    name = "Exponential"

    def sample(self, state, lhs, args):
        st = state.store
        (theta,) = (_scalar(lower(a, st), "Exponential argument") for a in args)
        cid, comp = _target(st, lhs, 1)
        ex = CExprs([theta])
        st._call("ws_sample_exponential", cid, comp, ex.ptr(0))

    def observe(self, state, value, args):
        st = state.store
        obs = _scalar(lower(value, st), "observed value")
        (theta,) = (_scalar(lower(a, st), "Exponential argument") for a in args)
        ex = CExprs([obs, theta])
        st._call("ws_observe_exponential", ex.ptr(0), ex.ptr(1))


def _const_matrix(a, d):
    if isinstance(a, Expr) and not isinstance(a, Const):
        raise _unsupported("MvNormal covariance must be a build-time constant (per-particle covariances are outside "
                           "the device-op set)")
    m = np.asarray(a.v if isinstance(a, Expr) else a, dtype=np.float64)
    if m.ndim == 1 and m.shape[0] == d:  # diagonal given as a vector of variances
        m = np.diag(m)
    if m.shape != (d, d):
        raise ValueError(f"covariance must be {d}x{d}, got {m.shape}")
    return np.ascontiguousarray(m)


class _MvNormal(WeightedKernel):
    name = "MvNormal"

    @staticmethod
    def _vec(tok, what):
        if not isinstance(tok, list):
            raise _unsupported(f"{what} must be vector-valued")
        return tok

    def sample(self, state, lhs, args):
        st = state.store
        mu = self._vec(lower(args[0], st), "MvNormal mean")
        d = len(mu)
        cov = _const_matrix(args[1], d)
        if isinstance(lhs, tuple):
            raise _unsupported("MvNormal into an accessor target")
        cid, _ = _target(st, lhs, d)
        ex = CExprs(mu)
        st._call("ws_sample_mvnormal", cid, d, ex.ptr(0), cov.ctypes.data_as(C.c_void_p))

    def observe(self, state, value, args):
        st = state.store
        obs = self._vec(lower(value, st), "observed value")
        mu = self._vec(lower(args[0], st), "MvNormal mean")
        d = len(mu)
        if len(obs) != d:
            raise ValueError("observation and mean dimensions differ")
        cov = _const_matrix(args[1], d)
        eo, em = CExprs(obs), CExprs(mu)
        st._call("ws_observe_mvnormal", d, eo.ptr(0), em.ptr(0), cov.ctypes.data_as(C.c_void_p))


Normal = _Normal()
Exponential = _Exponential()
MvNormal = _MvNormal()


class _ImportanceNormal(WeightedKernel):
    """``importance_kernel(Normal(pm, ps), Normal(tm, ts))`` (default_kernels.jl:69-73)."""
    name = "importance_kernel"
    has_weighter = True

    def __init__(self, pm, ps, tm, ts):
        self.p = (float(pm), float(ps), float(tm), float(ts))

    def sample(self, state, lhs, args):
        if len(args) != 0:
            raise ValueError("importance_kernel takes no arguments")
        st = state.store
        cid, comp = _target(st, lhs, 1)
        st._call("ws_sample_importance_normal", cid, comp, *self.p)


class NormalDist:
    """``Normal(mu, sigma)`` as a distribution VALUE (only as an importance_kernel argument)."""

    def __init__(self, mu, sigma):
        self.mu, self.sigma = float(mu), float(sigma)


def importance_kernel(proposal, target):
    if not (isinstance(proposal, NormalDist) and isinstance(target, NormalDist)):
        raise _unsupported("importance_kernel is built for Normal proposal / Normal target only")
    return _ImportanceNormal(proposal.mu, proposal.sigma, target.mu, target.sigma)


def _beta_sampler(a, b):
    from . import expr as E
    # X / (X + Y) with each variate appearing ONCE (an expression is a tree: a node used twice would be drawn twice);
    # evaluation order, hence replay order: Y ~ Gamma(b) first, then X ~ Gamma(a)
    return 1.0 / (1.0 + E.randgamma(b) / E.randgamma(a))


def _expr_kernels():
    """Distributions whose sampler is a closed-form transform of one standard variate, written as device
    expressions (formulas: Distributions.jl 0.25 `rand` / `logpdf`, un-vendored; pinned by scipy.stats in the tests)."""
    from . import expr as E
    NEG_INF = float("-inf")
    LOG2 = math.log(2.0)
    k = {}
    k["Uniform"] = WeightedKernel(lambda a, b: a + (b - a) * E.randu(), None,
                                  lambda a, b, x: E.where((x >= a) & (x <= b), -E.log(b - a), NEG_INF), "Uniform")
    k["LogNormal"] = WeightedKernel(lambda m, s: E.exp(m + s * E.randn()), None,
                                    lambda m, s, x: E.where(x > 0.0, -(((E.log(x) - m) / s) ** 2 + math.log(2 * math.pi)) / 2.0
                                                            - E.log(s) - E.log(x), NEG_INF), "LogNormal")
    k["Bernoulli"] = WeightedKernel(lambda p: E.randu() < p, None,
                                    lambda p, x: E.where(x, E.log(p), E.log1p(-p)), "Bernoulli")
    k["Laplace"] = WeightedKernel(lambda m, t: m + t * (E.randexp() - E.randexp()), None,
                                  lambda m, t, x: -abs(x - m) / t - E.log(2.0 * t), "Laplace")
    k["Cauchy"] = WeightedKernel(lambda m, s: m + s * E.tan(math.pi * (E.randu() - 0.5)), None,
                                 lambda m, s, x: -math.log(math.pi) - E.log(s) - E.log1p(((x - m) / s) ** 2), "Cauchy")
    k["Logistic"] = WeightedKernel(lambda m, t: m + t * (E.log(E.randexp()) * -1.0 + E.log(E.randexp())), None,
                                   lambda m, t, x: -((x - m) / t) - E.log(t) - 2.0 * E.log1p(E.exp(-((x - m) / t))), "Logistic")
    k["Gumbel"] = WeightedKernel(lambda m, t: m - t * E.log(E.randexp()), None,
                                 lambda m, t, x: -((x - m) / t) - E.exp(-((x - m) / t)) - E.log(t), "Gumbel")
    k["Rayleigh"] = WeightedKernel(lambda s: s * E.sqrt(2.0 * E.randexp()), None,
                                   lambda s, x: E.where(x >= 0.0, E.log(x) - 2.0 * E.log(s) - x * x / (2.0 * s * s), NEG_INF), "Rayleigh")
    k["Weibull"] = WeightedKernel(lambda a, t: t * E.randexp() ** (1.0 / a), None,
                                  lambda a, t, x: E.where(x >= 0.0, E.log(a / t) + (a - 1.0) * E.log(x / t) - (x / t) ** a, NEG_INF),
                                  "Weibull")
    k["Pareto"] = WeightedKernel(lambda a, t: t * E.exp(E.randexp() / a), None,
                                 lambda a, t, x: E.where(x >= t, E.log(a) + a * E.log(t) - (a + 1.0) * E.log(x), NEG_INF), "Pareto")
    # samplers that need a rejection loop: device variates with a parameter (expr.randgamma / randpoisson: Marsaglia-Tsang
    # and inversion / PTRS on Philox sub-counters, csrc/ws_math.cuh); the constructions are Distributions.jl's own
    # (Beta = X / (X + Y) from two Gammas, TDist = Z / sqrt(Chisq(v) / v), Chisq(v) = Gamma(v / 2, 2), InverseGamma = 1 / Gamma)
    k["Gamma"] = WeightedKernel(lambda a, t: t * E.randgamma(a), None, lambda a, t, x: E.where(x >= 0.0, (a - 1.0) * E.log(x) - x / t - E.lgamma(a) - a * E.log(t),
                                                                     NEG_INF), "Gamma")
    k["Beta"] = WeightedKernel(_beta_sampler, None, lambda a, b, x: E.where((x >= 0.0) & (x <= 1.0),
                                                                    (a - 1.0) * E.log(x) + (b - 1.0) * E.log1p(-x)
                                                                    - (E.lgamma(a) + E.lgamma(b) - E.lgamma(a + b)), NEG_INF), "Beta")
    k["TDist"] = WeightedKernel(lambda v: E.randn() / E.sqrt(2.0 * E.randgamma(v / 2.0) / v), None, lambda v, x: E.lgamma((v + 1.0) / 2.0) - E.lgamma(v / 2.0) - 0.5 * E.log(v * math.pi)
                                - (v + 1.0) / 2.0 * E.log1p(x * x / v), "TDist")
    k["Poisson"] = WeightedKernel(lambda lam: E.randpoisson(lam), None,
                                  lambda lam, x: E.where(x >= 0.0, x * E.log(lam) - lam - E.lgamma(x + 1.0), NEG_INF), "Poisson")
    k["Chisq"] = WeightedKernel(lambda v: 2.0 * E.randgamma(v / 2.0), None,
                                lambda v, x: E.where(x >= 0.0, (v / 2.0 - 1.0) * E.log(x) - x / 2.0 - E.lgamma(v / 2.0) - (v / 2.0) * LOG2,
                                                     NEG_INF), "Chisq")
    # Categorical(p), p a constant probability vector or a row P[s, :] of a build-time matrix (expr.Table): the draw
    # inverts the row's sequential partial sums at one uniform, the logpdf reads the row's logarithms (include/wsb200.h)
    k["Categorical"] = WeightedKernel(lambda p: E.randcat(p), None, lambda p, x: E.cat_logpdf(p, x), "Categorical")
    k["InverseGamma"] = WeightedKernel(lambda a, t: t / E.randgamma(a), None,
                                       lambda a, t, x: E.where(x > 0.0, a * E.log(t) - E.lgamma(a) - (a + 1.0) * E.log(x) - t / x, NEG_INF),
                                       "InverseGamma")
    return k


default_kernels = {"Normal": Normal, "MvNormal": MvNormal, "Exponential": Exponential}
default_kernels.update(_expr_kernels())

# the reference's other 52 table entries (default_kernels.jl:83-102) are outside the device-op set
_REFERENCE_ONLY_KERNELS = [k for k in (
    "Beta BernoulliLogit Bernoulli BetaBinomial Binomial Categorical Cauchy Chi Chisq Dirac Dirichlet "
    "DiscreteNonParametric DiscreteUniform FDist Frechet Gamma GeneralizedPareto Geometric Gumbel Hypergeometric "
    "InverseGamma InverseWishart LKJ LKJCholesky Laplace LogNormal Logistic LogitNormal MatrixBeta MatrixFDist "
    "MatrixNormal MatrixTDist MvLogNormal MvLogitNormal MvNormalCanon Multinomial NegativeBinomial NoncentralChisq "
    "NoncentralF NoncentralT NormalCanon Pareto Poisson PoissonBinomial Rayleigh SkewNormal SkewedExponentialPower "
    "TDist Uniform VonMises Weibull Wishart").split() if k not in default_kernels]


def resolve_kernel(f, kernels=None):
    """Kernel resolution by name (rewrites.jl:383-389): user table over default_kernels."""
    if isinstance(f, WeightedKernel):
        return f
    table = dict(default_kernels)
    if kernels:
        table.update(kernels)
    if f in table:
        return table[f]
    if f in _REFERENCE_ONLY_KERNELS:
        raise _unsupported(f"kernel {f} is in the reference's default_kernels but outside the device-op set "
                           "(Normal, MvNormal, Exponential)")
    raise KeyError(f"unknown kernel {f!r}")


# --------------------------------------------------------------------------------------------------
# L3: transformers
# --------------------------------------------------------------------------------------------------
class ParticleTransformer:
    def apply(self, state): raise NotImplementedError
    def score(self, state, ctx): raise NotImplementedError


class ScoreCtx:
    """types.jl:147-152.  ``scores`` are accumulated on the device tape; only depth is tracked here."""

    def __init__(self, targets, target_depth, depth=0):
        self.targets, self.target_depth, self.depth = list(targets), int(target_depth), int(depth)


def _args(argfn, state):
    a = argfn(state) if callable(argfn) else argfn
    return tuple(a) if isinstance(a, (tuple, list)) else (a,)


def _one(fn, state):
    return fn(state) if callable(fn) else fn


class Assign(ParticleTransformer):
    """``x .= expr`` (transformers.jl:18-42).  ``lhs`` may be ``(name, j)`` for ``x[j] .= expr``
    (AccessorAssign on a vector column, transformers.jl:57-80)."""

    def __init__(self, lhs, argfn):
        self.lhs, self.argfn = lhs, argfn

    def apply(self, state):
        st = state.store
        tok = lower(_one(self.argfn, state), st)
        if isinstance(tok, list):
            if isinstance(self.lhs, tuple):
                raise _unsupported("vector value into an accessor target")
            cid, _ = _target(st, self.lhs, len(tok))
            ex = CExprs(tok)
            st._call("ws_assign_vec", cid, len(tok), ex.ptr(0))
        else:
            cid, comp = _target(st, self.lhs, 1)
            ex = CExprs([tok])
            st._call("ws_assign", cid, comp, ex.ptr(0))

    def score(self, state, ctx):
        state.store._call("ws_set_depth", ctx.depth + 1)
        ctx.depth += 1


AccessorAssign = Assign


class Sample(ParticleTransformer):
    """``x ~ f(args)`` (transformers.jl:158-199); ``lhs = (name, j)`` is AccessorSample
    (``x[j] ~ f(args)``, transformers.jl:103-145)."""

    def __init__(self, lhs, kernel, argfn=()):
        self.lhs, self.kernel, self.argfn = lhs, resolve_kernel(kernel), argfn

    def apply(self, state):
        self.kernel.sample(state, self.lhs, _args(self.argfn, state))

    def score(self, state, ctx):
        # record-only mode: the same call appends the statement's log-density to the tape
        self.kernel.sample(state, self.lhs, _args(self.argfn, state))
        ctx.depth += 1


AccessorSample = Sample


class Observe(ParticleTransformer):
    """``expr => f(args)`` (transformers.jl:216-249)."""

    def __init__(self, lhsfn, kernel, argfn):
        self.lhsfn, self.kernel, self.argfn = lhsfn, resolve_kernel(kernel), argfn

    def apply(self, state):
        self.kernel.observe(state, _one(self.lhsfn, state), _args(self.argfn, state))

    def score(self, state, ctx):
        self.apply(state)
        ctx.depth += 1


class Weight(ParticleTransformer):
    """``_ ~ f(args)`` (transformers.jl:270-302).  With a distribution kernel the LAST argument plays
    the role of the value (the reference's NormalWeightKernel: ``(mu, sigma, x) -> logpdf``); with
    ``kernel=None`` the single argument is an arbitrary log-weight expression."""

    def __init__(self, kernel, argfn):
        self.kernel = None if kernel is None else resolve_kernel(kernel)
        self.argfn = argfn

    def apply(self, state):
        a = _args(self.argfn, state)
        if self.kernel is None:
            tok = _scalar(lower(a[0], state.store), "log-weight term")
            ex = CExprs([tok])
            state.store._call("ws_weight_expr", ex.ptr(0))
        elif type(self.kernel) is WeightedKernel:
            self.kernel.weight(state, a)
        else:
            self.kernel.observe(state, a[-1], a[:-1])

    def score(self, state, ctx):
        self.apply(state)
        ctx.depth += 1


class Sequence(ParticleTransformer):
    """transformers.jl:320-349."""

    def __init__(self, *steps):
        if len(steps) == 1 and isinstance(steps[0], (tuple, list)):
            steps = tuple(steps[0])
        self.steps = tuple(steps)

    def apply(self, state):
        for s in self.steps:
            s.apply(state)

    def score(self, state, ctx):
        for s in self.steps:
            if not ctx.depth < ctx.target_depth:
                break
            s.score(state, ctx)


# -- loop bodies described once, replayed per element (include/wsb200.h: ws_exec) ---------------------------------
class _Recorder:
    """Stands in for the store while a loop body built over SYMBOLIC element values is applied: statement calls are
    recorded as ws_cmd entries instead of being issued; anything else a body might do aborts the recording."""

    # (i0, i1 positions among the call's integer arguments come first, then the expression pointers in order)
    def __init__(self, store):
        self.store, self.cmds, self.keep = store, [], []
        self.n = store.n

    def _lookup(self, name):
        return self.store._lookup(name)

    def _table_id(self, tab):
        return self.store._table_id(tab)

    def _ensure(self, name, width):
        cid, w = self.store._lookup(name)
        if cid < 0 or w != width:
            raise _NoTemplate("the body creates a column")      # columns must exist before the body is templated
        return cid

    def colnames(self):
        return self.store.colnames()

    def _call(self, name, *args):
        fn = L.CMD_FN.get(name)
        if fn is None:
            raise _NoTemplate(f"{name} inside a loop body")
        ints = [a for a in args if isinstance(a, int)]
        ptrs = [a for a in args if not isinstance(a, int)]
        d = 1
        if name in ("ws_assign_vec", "ws_sample_mvnormal"):
            d = ints[1]
        elif name == "ws_observe_mvnormal":
            d = ints[0]
        mat = None
        if name in ("ws_sample_mvnormal", "ws_observe_mvnormal"):
            mat = ptrs.pop()
        self.cmds.append((fn, ints, ptrs, d, mat))
        self.keep.append(args)


class _NoTemplate(Exception):
    pass


class _RecState:
    """what a statement's ``apply`` touches of an SMCState, over a recorder"""

    def __init__(self, store):
        self.store = store


def _symbolic_like(x):
    """(symbolic stand-in for the loop element x with Param leaves, flatten(x') -> list of floats or None)"""
    from .expr import Param
    counter = [0]

    def sym(v):
        if isinstance(v, (bool, np.bool_)):
            raise _NoTemplate("a Bool loop element")
        if isinstance(v, (int, np.integer)):
            raise _NoTemplate("an integer loop element (it may index or name something at build time)")
        if isinstance(v, (float, np.floating)):
            counter[0] += 1
            return Param(counter[0] - 1)
        if isinstance(v, np.ndarray):
            if v.ndim != 1 or v.dtype.kind != "f":
                raise _NoTemplate("a non-vector array loop element")
            return [sym(float(t)) for t in v]
        if isinstance(v, (tuple, list)):
            out = [sym(t) for t in v]
            return tuple(out) if isinstance(v, tuple) else out
        raise _NoTemplate(f"a loop element of type {type(v).__name__}")

    def shape(v):
        if isinstance(v, (float, np.floating)) and not isinstance(v, (bool, np.bool_)):
            return "f"
        if isinstance(v, np.ndarray) and v.ndim == 1 and v.dtype.kind == "f":
            return ("a", v.shape[0])
        if isinstance(v, (tuple, list)):
            return (type(v).__name__, tuple(shape(t) for t in v))
        return None

    s = sym(x)
    want = shape(x)

    def flatten(v):
        if shape(v) != want:
            return None
        out = []

        def walk(t):
            if isinstance(t, (tuple, list)):
                for u in t:
                    walk(u)
            elif isinstance(t, np.ndarray):
                out.extend(float(u) for u in t)
            else:
                out.append(float(t))
        walk(v)
        return out
    return s, flatten, counter[0]


_TEMPLATE_OK = ("Sequence", "Assign", "Sample", "Observe", "Weight", "Resample")


def _only_statements(t):
    k = type(t).__name__
    if k not in _TEMPLATE_OK:
        return False
    return all(_only_statements(s) for s in t.steps) if k == "Sequence" else True


class _LoopTemplate:
    """The body of a loop as one ws_cmd array with WS_TOK_PARAM holes for the element's values."""

    def __init__(self, bodyfn, x, store):
        sym, self.flatten, self.n_params = _symbolic_like(x)
        try:
            body = bodyfn(sym)
        except (UnsupportedModelError, _NoTemplate):
            raise
        except Exception as e:          # the body uses the element at build time (indexing, names, arithmetic on it, ...)
            raise _NoTemplate(f"{type(e).__name__}: {e}")
        # "weighting statements, Resample(), if resampled ... end" (examples/linear_regression.jl:20-26): the statements
        # are templated and run in speculative blocks (ws_exec_spec); the `if` body is built for the element that fires
        self.spec = False
        if not _only_statements(body):
            steps = getattr(body, "steps", ())
            if (SPEC_BLOCKS and type(body).__name__ == "Sequence" and len(steps) >= 3 and type(steps[-1]).__name__ == "Cond"
                    and getattr(steps[-1].predfn, "only_resampled", False) and type(steps[-2]).__name__ == "Resample"
                    and all(type(t).__name__ in ("Observe", "Weight") for t in steps[:-2])):
                body = Sequence(*steps[:-1])
                self.spec = True
            else:
                raise _NoTemplate("the body contains control flow or moves")
        rec = _Recorder(store)
        try:
            body.apply(_RecState(rec))
        except (UnsupportedModelError, _NoTemplate):
            raise
        except Exception as e:
            raise _NoTemplate(f"{type(e).__name__}: {e}")
        if not rec.cmds:
            raise _NoTemplate("empty body")
        self.keep = rec.keep
        self.arr = (L.ws_cmd * len(rec.cmds))()
        for c, (fn, ints, ptrs, d, mat) in zip(self.arr, rec.cmds):
            c.fn = fn
            c.i0 = ints[0] if len(ints) > 0 else 0
            c.i1 = ints[1] if len(ints) > 1 else 0
            for k, p in enumerate(ptrs):
                if p is None:
                    c.n_e[k] = 0
                else:
                    c.n_e[k] = d
                    c.e[k] = p
            if mat is not None:
                c.mat = C.cast(mat, C.POINTER(C.c_double))
        self.n = len(rec.cmds)
        self.store = store
        self._params = (C.c_double * max(1, self.n_params))()

    def run(self, x):
        vals = self.flatten(x)
        if vals is None:
            return False
        self._params[:len(vals)] = vals
        self.store._call("ws_exec", self.arr, self.n, self._params, self.n_params)
        return True

    def run_many(self, coll, i, limit=512):
        """elements coll[i], coll[i + 1], ... (up to `limit`, up to the first one of another shape) with one C call
        -> number of elements done"""
        flat, j, n = [], i, len(coll)
        while j < n and j - i < limit:
            vals = self.flatten(coll[j])
            if vals is None:
                break
            flat.extend(vals)
            j += 1
        if j > i:
            buf = (C.c_double * max(1, len(flat)))(*flat)
            self.store._call("ws_exec_n", self.arr, self.n, buf, self.n_params, j - i)
        return j - i

    def run_block(self, xs):
        """up to len(xs) consecutive elements as one speculative block -> (elements done, the last of them resampled);
        None if an element does not have the template's shape"""
        flat = []
        for x in xs:
            vals = self.flatten(x)
            if vals is None:
                return None
            flat.extend(vals)
        buf = (C.c_double * max(1, len(flat)))(*flat)
        n_done, fired = C.c_int32(), C.c_int32()
        self.store._call("ws_exec_spec", self.arr, self.n, buf, self.n_params, len(xs), C.byref(n_done), C.byref(fired))
        return n_done.value, bool(fired.value)


LOOP_TEMPLATES = os.environ.get("WSB200_LOOP_TEMPLATE", "1") != "0"
SPEC_BLOCKS = os.environ.get("WSB200_SPEC_BLOCKS", "1") != "0"
SPEC_BLOCK_STEPS = int(os.environ.get("WSB200_SPEC_BLOCK_STEPS", "8"))   # what the register-resident block kernel holds (WS_SLCK_N)


class Loop(ParticleTransformer):
    """``for x in coll ... end`` (transformers.jl:367-398); the body is rebuilt per iteration.

    When the elements are plain numbers / vectors and the body is a straight list of statements that uses them only
    as constants (a filter step: ``o => Normal(x, r)``), rebuilding it per element would produce the same statement
    calls with different constants.  From the second element on such a body is described ONCE (built over symbolic
    element values, recorded instead of issued) and replayed per element with one C call (``ws_exec``): the
    statements issued, their order and their results are those of the per-element rebuild; a body that does anything
    else with its element (an index, a column name ``x{t}``, ``if``, ``<<``) is rebuilt per element as before."""

    def __init__(self, collfn, bodyfn):
        self.collfn, self.bodyfn = collfn, bodyfn

    def _coll(self, state):
        return self.collfn(state) if callable(self.collfn) else self.collfn

    def apply(self, state):
        coll = self._coll(state)
        if not LOOP_TEMPLATES or not isinstance(state.store, DeviceColumnStore) or not hasattr(coll, "__len__") or len(coll) < 4:
            for x in coll:
                self.bodyfn(x).apply(state)
            return
        if not hasattr(coll, "__getitem__"):
            coll = list(coll)
        self.bodyfn(coll[0]).apply(state)           # the first element runs as written (it may create the columns)
        tmpl = None
        i, n = 1, len(coll)
        k_cur = SPEC_BLOCK_STEPS        # steps per speculative block: halved when blocks end early, doubled when they run through
        while i < n:
            x = coll[i]
            if tmpl is None:
                try:
                    tmpl = _LoopTemplate(self.bodyfn, x, state.store)
                except _NoTemplate:
                    tmpl = False
            if tmpl is not False and tmpl.spec:
                # blocks of steps in one pass; a step that resamples ends its block and runs its `if resampled` body.
                # A block that ends early has computed the steps behind the firing one for nothing, so where steps
                # resample often (a high threshold, the first observations of a diffuse prior) the blocks shrink, down
                # to plain element-by-element execution, and grow again once steps stop firing.
                if k_cur <= 1:
                    self.bodyfn(x).apply(state)
                    i += 1
                    if not state.resampled:
                        k_cur = 2
                    continue
                try:
                    r = tmpl.run_block([coll[k] for k in range(i, min(n, i + k_cur))])
                except UnsupportedModelError:
                    r = None
                if r is None:
                    tmpl = False        # (sharded / replayed state, an element of another shape): element by element
                    continue
                done, fired = r
                if fired:
                    self.bodyfn(coll[i + done - 1]).steps[-1].body.apply(state)
                    if done <= k_cur // 2:
                        k_cur = max(1, k_cur // 2)
                else:
                    k_cur = min(SPEC_BLOCK_STEPS, k_cur * 2)
                i += done
                continue
            if tmpl is not False:
                done = tmpl.run_many(coll, i)
                if done > 0:
                    i += done
                    continue
            self.bodyfn(x).apply(state)
            i += 1

    def score(self, state, ctx):
        for x in self._coll(state):
            if not ctx.depth < ctx.target_depth:
                break
            self.bodyfn(x).score(state, ctx)


class Cond(ParticleTransformer):
    """``if cond ... end`` (transformers.jl:413-444); ``predfn(state) -> bool`` on the host."""

    def __init__(self, predfn, body=None, lazy_body=None):
        # ``lazy_body``: zero-argument builder of the body, used by the @model front-end when constructing the body
        # has no build-time side effects: a loop that rebuilds `if resampled ... end` per iteration (the reference
        # does, rewrites.jl:671-682) then pays for the body only in the iterations that take the branch
        self.predfn, self._body, self._lazy = predfn, body, lazy_body

    @property
    def body(self):
        if self._body is None:
            self._body = self._lazy()
        return self._body

    def apply(self, state):
        if self.predfn(state):
            self.body.apply(state)

    def score(self, state, ctx):
        if self.predfn(state):
            self.body.score(state, ctx)


class Resample(ParticleTransformer):
    """transformers.jl:461-507 — the whole state machine runs inside ``ws_resample``."""

    def __init__(self):
        self._store = None

    def apply(self, state):
        # queued, not awaited: the decision stays on the device until somebody asks (`state.resampled`, `.last`, ...)
        state.store._call("ws_resample_async")
        self._store = state.store

    @property
    def last(self):
        """outcome of the most recent application (fired, resampled, ess_perc, log_mean_w); waits for it if needed"""
        if self._store is None:
            return None
        info = L.ws_resample_info()
        self._store._call("ws_last_resample", C.byref(info))
        return info

    def score(self, state, ctx):
        return None


# -- proposals (move_kernels.jl:189-265) ------------------------------------------------------------
class _Proposal:
    def __init__(self, code, name):
        self.code, self.name = code, name

    def __repr__(self):
        return self.name


RW = _Proposal(0, "RW")
autoRW = _Proposal(1, "autoRW")
default_proposals = {"RW": RW, "autoRW": autoRW}


def _normalize_bounds(bounds, d):
    """move_kernels.jl:23-28."""
    if bounds is None:
        return None
    if isinstance(bounds, tuple) and len(bounds) == 2 and not isinstance(bounds[0], (tuple, list)):
        return [tuple(map(float, bounds))] * d
    b = [tuple(map(float, x)) for x in bounds]
    if len(b) != d:
        raise ValueError(f"bounds must have length {d} (one (lo, hi) tuple per target), got {len(b)}")
    return b


def _target_planes(store, targets):
    cols, comps = [], []
    for t in targets:
        if isinstance(t, tuple):
            raise _unsupported("accessor targets (x[e] / x.p) cannot be moved; a move rewrites a whole column")
        cid, w = store._lookup(str(t))
        if cid < 0:
            raise KeyError(f"move target {t!r} does not exist")
        for k in range(w):  # a vector-valued target moves all its components jointly
            cols.append(cid)
            comps.append(k)
    return cols, comps


def marginal_diversity(store, targets):
    """transformers.jl:560-565: min over targets of |unique(col)| / N."""
    cols, comps = _target_planes(store, list(targets))
    c = (C.c_int32 * len(cols))(*cols)
    k = (C.c_int32 * len(cols))(*comps)
    out = C.c_double()
    store._call("ws_marginal_diversity", len(cols), c, k, C.byref(out))
    return out.value


class Move(ParticleTransformer):
    """``x << q(args)`` (transformers.jl:543-633)."""

    def __init__(self, targets, proposal, argfn=(), diversity_threshold=None):
        if isinstance(targets, str):
            targets = [targets]
        self.targets = list(targets)
        self.proposal = default_proposals[proposal] if isinstance(proposal, str) else proposal
        if not isinstance(self.proposal, _Proposal):
            raise _unsupported("custom host proposal functions are outside the device-op set (RW, autoRW)")
        self.argfn = argfn
        self.diversity_threshold = diversity_threshold
        self.last = None

    def apply(self, state):
        st = state.store
        args = _args(self.argfn, state)
        cols, comps = _target_planes(st, self.targets)
        d = len(cols)
        if self.proposal is RW:
            if len(args) < 1:
                raise TypeError("RW(step_size, bounds=nothing) needs a step size")
            step = float(np.asarray(args[0]).ravel()[0])
            bounds = args[1] if len(args) > 1 else None
        else:
            step = float(np.asarray(args[0]).ravel()[0]) if len(args) > 0 else 1e-3  # min_step
            bounds = args[1] if len(args) > 1 else None
        bnds = _normalize_bounds(bounds, d)
        if not state._tape_valid:
            _rebuild_tape(state)
        spec = L.ws_move_spec()
        spec.n_targets = d
        c_arr = (C.c_int32 * d)(*cols)
        k_arr = (C.c_int32 * d)(*comps)
        spec.col, spec.comp = c_arr, k_arr
        spec.proposal = self.proposal.code
        if bnds is None:
            spec.has_bounds = 0
        else:
            spec.has_bounds = 1
            lo = (C.c_double * d)(*[b[0] for b in bnds])
            hi = (C.c_double * d)(*[b[1] for b in bnds])
            spec.lo, spec.hi = lo, hi
        spec.step = step
        spec.diversity = float("nan") if self.diversity_threshold is None else float(self.diversity_threshold)
        spec.target_depth = -1
        info = L.ws_move_info()
        st._call("ws_move", C.byref(spec), C.byref(info))
        self.last = info

    def score(self, state, ctx):
        return None


# --------------------------------------------------------------------------------------------------
# run! / score_logpdf
# --------------------------------------------------------------------------------------------------
def apply(t, state):
    """``apply!(t, state)``."""
    t.apply(state)


def score(t, state, ctx):
    """``score!(t, state, ctx)`` (record-only walk; see :func:`score_logpdf`)."""
    t.score(state, ctx)


def run(root, state):
    """``run!(root, state)`` (types.jl:120-126)."""
    st = state.store
    record = bool(state.record_tape) and getattr(root, "_has_moves", True)
    st._call("ws_tape_enable", int(record))
    st._call("ws_begin_run")
    state._root = root
    state._tape_valid = record
    root.apply(state)
    faults = st._new_index_faults()
    if faults:
        raise IndexError(f"{faults} table reads had an index that is not an integer in range (Julia would throw a "
                         "BoundsError); those values are NaN")
    return state


def _rebuild_tape(state, target_depth=None):
    """Re-walk ``state.root`` with score! semantics, recording (not executing) every scored
    statement with depth < target_depth onto the device tape."""
    if state._root is None:
        raise RuntimeError("state.root is not set: a Move / score_logpdf needs run!(root, state) or state.root = root")
    st = state.store
    depth = state._flags()[2]
    td = depth if target_depth is None else int(target_depth)
    st._call("ws_tape_enable", 1)
    st._call("ws_tape_clear")
    st._call("ws_tape_record_only", 1)
    try:
        st._call("ws_set_depth", 0)
        ctx = ScoreCtx([], td, 0)
        if ctx.depth < ctx.target_depth:
            state._root.score(state, ctx)
    finally:
        st._call("ws_tape_record_only", 0)
        st._call("ws_set_depth", depth)
    state._tape_valid = target_depth is None


def score_logpdf(state, targets, target_depth):
    """``score_logpdf(state, targets, target_depth)`` (types.jl:183-206) -> host vector."""
    _rebuild_tape(state, target_depth)
    out = np.empty(state.store.n, dtype=np.float64)
    state.store._call("ws_score_logpdf", int(target_depth), out.ctypes.data_as(C.c_void_p))
    state._tape_valid = False
    return out
