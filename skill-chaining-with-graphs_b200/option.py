"""Per-option Sarsa(lambda) over an order-n Fourier basis and logistic initiation classifiers on
B200 (K2, K3, K4), behind the interface of the CPU oracle (oracle/option.py OptionSet / Option and
oracle/fourier.py FourierBasis - the stand-in for the reference, which has no code:
/root/reference/README.md:1-2).

All tensors are CUDA tensors; weights W (K, A, F), classifiers theta (K, 6), per-env traces
(B, A, F), window accumulators dW (K, A, F) / cnt (K,).  States are passed as (B, 4) tensors (they
are transposed to structure-of-arrays for the kernels) or directly as a (4, B) SoA tensor via the
`soa=` keyword.
"""
import ctypes as C

import numpy as np

from . import _lib
from ._lib import check, ptr, N_ACTIONS, N_PSI


class FourierBasis:
    """Feature definition only (multi-index table, per-feature step-size scale); the kernels
    regenerate features in registers.  `features()` runs the debug operator scg_features."""

    def __init__(self, order):
        if not 1 <= int(order) <= _lib.MAX_ORDER:
            raise ValueError(f"order must be in 1..{_lib.MAX_ORDER}")
        self.order = int(order)
        n1 = self.order + 1
        self.n_features = n1 ** 4
        f = np.arange(self.n_features)
        self.C = np.stack([(f // n1 ** 3) % n1, (f // n1 ** 2) % n1, (f // n1) % n1, f % n1], axis=1).astype(np.int32)
        norm = np.sqrt((self.C.astype(np.float64) ** 2).sum(axis=1))
        norm[norm == 0] = 1.0
        self.alpha_scale = (1.0 / norm).astype(np.float32)

    def features(self, state):
        import torch
        soa = _as_soa(state)
        B = soa.shape[1]
        phi = torch.empty((B, self.n_features), dtype=torch.float32, device=soa.device)
        check(_lib.load().scg_features(self.order, B, ptr(soa[0]), ptr(soa[1]), ptr(soa[2]), ptr(soa[3]), ptr(phi),
                                       _lib.current_stream()))
        return phi


def _as_soa(state):
    """(B, 4) CUDA tensor / numpy -> contiguous (4, B) fp32 CUDA tensor."""
    import torch
    if not hasattr(state, "is_cuda"):
        state = torch.as_tensor(np.asarray(state, dtype=np.float32))
    if not state.is_cuda:
        state = state.cuda()
    state = state.to(torch.float32)
    if state.dim() != 2 or state.shape[1] != 4:
        raise ValueError("state must have shape (B, 4)")
    return state.t().contiguous()


def _dev(t, dtype):
    import torch
    if not hasattr(t, "is_cuda"):
        t = torch.as_tensor(np.asarray(t))
    if not t.is_cuda:
        t = t.cuda()
    return t.to(dtype).contiguous()


class OptionSet:
    def __init__(self, n_options, order, batch, gamma=0.99, lam=0.9, alpha=1e-3, epsilon=0.05, seed=0,
                 env_offset=0, device=None, deterministic=False, top_slots=0, alpha_top=1e-3):
        import torch
        if not torch.cuda.is_available():
            raise _lib.ScgError("OptionSet needs a CUDA device: there is no CPU fallback")
        self.torch = torch
        self.lib = _lib.load()
        self.K = int(n_options)
        # top-level learner (oracle/option.py OptionSet(top_slots=...)): Q_top(s, j) is row j % 5 of slot K + j // 5
        self.top_slots = int(top_slots)
        self.K_all = self.K + self.top_slots
        self.alpha_top = float(alpha_top)
        if not 1 <= self.K or not self.K_all <= _lib.MAX_OPTIONS or self.top_slots < 0:
            raise ValueError(f"n_options (+ top-level slots) must be in 1..{_lib.MAX_OPTIONS}")
        self.basis = FourierBasis(order)
        self.order = self.basis.order
        self.F = self.basis.n_features
        self.B = int(batch)
        self.gamma, self.lam, self.alpha, self.epsilon = float(gamma), float(lam), float(alpha), float(epsilon)
        self.seed = int(seed)
        self.env_offset = int(env_offset)
        self.device = torch.device("cuda", torch.cuda.current_device()) if device is None else torch.device(device)
        z = dict(dtype=torch.float32, device=self.device)
        self.W = torch.zeros((self.K_all, N_ACTIONS, self.F), **z)
        self.Wt = torch.zeros((self.K_all, self.lib.scg_packed_slot_floats(self.order)), **z)   # packed pair layout
        self.theta = torch.zeros((self.K, N_PSI), **z)
        self._trace = torch.zeros((self.B, N_ACTIONS, self.F), **z)
        self._dW = torch.zeros((self.K_all, N_ACTIONS, self.F), **z)
        self._pre_read = None        # set by SkillChainAgent: folds its open window in before a read
        self._on_weights_changed = None   # set by SkillChainAgent: its carried Q_o(s, a) goes stale
        self._cnt = torch.zeros(self.K_all, dtype=torch.int32, device=self.device)
        self.window_steps = 0
        self._ctx = C.c_void_p()
        check(self.lib.scg_ctx_create(self.order, self.K_all, C.byref(self._ctx)))
        if deterministic:       # fixed-order dW reduction: bit-reproducible runs, ~1 us per step slower at 65,536 envs
            check(self.lib.scg_ctx_set_deterministic(self._ctx, 1))

    def __del__(self):
        try:
            if getattr(self, "_ctx", None):
                self.lib.scg_ctx_destroy(self._ctx)
                self._ctx = None
        except Exception:
            pass

    @property
    def ctx(self):
        return self._ctx

    @property
    def trace(self):
        """Per-env eligibility traces (B, A, F)."""
        if self._pre_read is not None:
            self._pre_read()
        return self._trace

    @property
    def cnt(self):
        """Updates per weight slot accumulated since the last apply (K_all,)."""
        if self._pre_read is not None:
            self._pre_read()
        return self._cnt

    @property
    def dW(self):
        """Weight deltas accumulated since the last apply (K, A, F)."""
        if self._pre_read is not None:
            self._pre_read()
        return self._dW

    # -- weights ---------------------------------------------------------------------------------
    def set_weights(self, W):
        self.W.copy_(_dev(W, self.torch.float32).reshape(self.K_all, N_ACTIONS, self.F))
        self.pack()
        if self._on_weights_changed is not None:
            self._on_weights_changed()

    def pack(self):
        check(self.lib.scg_pack_weights(self.order, self.K_all, ptr(self.W), ptr(self.Wt), _lib.current_stream()))

    # -- K2 --------------------------------------------------------------------------------------
    def q(self, state, option_ids, soa=None):
        torch = self.torch
        s = _as_soa(state) if soa is None else soa
        B = s.shape[1]
        o = _dev(option_ids, torch.int32)
        Q = torch.empty((B, N_ACTIONS), dtype=torch.float32, device=self.device)
        check(self.lib.scg_q_eval(self.order, self.K_all, B, ptr(s[0]), ptr(s[1]), ptr(s[2]), ptr(s[3]), ptr(o),
                                  ptr(self.Wt), ptr(Q), _lib.current_stream()))
        return Q

    def q_top(self, state, soa=None):
        """Q_top(s, j) for every option slot j: (B, K) (rows of the top-level slots of W)."""
        torch = self.torch
        s = _as_soa(state) if soa is None else soa
        B = s.shape[1]
        cols = []
        for sl in range(self.top_slots):
            ids = torch.full((B,), self.K + sl, dtype=torch.int32, device=self.device)
            cols.append(self.q(None, ids, soa=s))
        return torch.cat(cols, dim=1)[:, :self.K] if cols else torch.zeros((B, 0), device=self.device)

    def select(self, Q, step, stream=_lib.STREAM_ACTION):
        torch = self.torch
        B = Q.shape[0]
        a = torch.empty(B, dtype=torch.int32, device=self.device)
        check(self.lib.scg_select(B, ptr(Q), self.epsilon, self.seed, int(step) & 0xFFFFFFFF, int(stream),
                                  self.env_offset, ptr(a), _lib.current_stream()))
        return a

    def act(self, state, option_ids, step, stream=_lib.STREAM_ACTION, soa=None):
        return self.select(self.q(state, option_ids, soa=soa), step, stream)

    def td_error(self, s, a, r, s2, a2, done, option_ids):
        torch = self.torch
        s, s2 = _as_soa(s), _as_soa(s2)
        B = s.shape[1]
        a, a2, o = _dev(a, torch.int32), _dev(a2, torch.int32), _dev(option_ids, torch.int32)
        r = _dev(r, torch.float32)
        d = _dev(done, torch.uint8)
        delta = torch.empty(B, dtype=torch.float32, device=self.device)
        check(self.lib.scg_td_error(self.order, self.K_all, B, ptr(s[0]), ptr(s[1]), ptr(s[2]), ptr(s[3]), ptr(a), ptr(r),
                                    ptr(s2[0]), ptr(s2[1]), ptr(s2[2]), ptr(s2[3]), ptr(a2), ptr(d), ptr(o),
                                    ptr(self.Wt), self.gamma, ptr(delta), _lib.current_stream()))
        return delta

    # -- K3 --------------------------------------------------------------------------------------
    def update(self, s, a, r, s2, a2, done, option_ids, mask=None):
        """One Sarsa(lambda) update for every env (or those in `mask`); returns delta (B,)."""
        torch = self.torch
        delta = self.td_error(s, a, r, s2, a2, done, option_ids)
        soa = _as_soa(s)
        a, o = _dev(a, torch.int32), _dev(option_ids, torch.int32)
        d = _dev(done, torch.uint8)
        m = None if mask is None else _dev(mask, torch.uint8)
        if m is not None:
            delta = torch.where(m.bool(), delta, torch.zeros_like(delta))
        gl = float(np.float32(self.gamma) * np.float32(self.lam))
        check(self.lib.scg_sarsa_update(self._ctx, self.B, ptr(soa[0]), ptr(soa[1]), ptr(soa[2]), ptr(soa[3]), ptr(a),
                                        ptr(o), ptr(delta), ptr(d), ptr(m), gl, ptr(self._trace), ptr(self._dW),
                                        ptr(self._cnt), _lib.current_stream()))
        return delta

    def tick(self):
        self.window_steps += 1

    def apply(self):
        """Fold the window's dW into W (call after any cross-rank allreduce of dW / cnt)."""
        if self._pre_read is not None:
            self._pre_read()
        check(self.lib.scg_apply(self._ctx, self.K, ptr(self.W), ptr(self.Wt), ptr(self._dW), ptr(self._cnt), self.alpha,
                                 self.alpha_top, max(self.window_steps, 1), _lib.current_stream()))
        self.window_steps = 0
        if self._on_weights_changed is not None:
            self._on_weights_changed(applied=True)

    # -- K4 --------------------------------------------------------------------------------------
    def initiation_prob(self, state):
        torch = self.torch
        s = _as_soa(state)
        B = s.shape[1]
        p = torch.empty((B, self.K), dtype=torch.float32, device=self.device)
        check(self.lib.scg_clf_eval(B, ptr(s[0]), ptr(s[1]), ptr(self.theta), self.K, ptr(p), _lib.current_stream()))
        return p

    def initiation(self, state):
        """I_k(s) for every option: bool (B, K), decided on the fp32 logit exactly as the oracle does (bit-identical)."""
        torch = self.torch
        s = _as_soa(state)
        B = s.shape[1]
        out = torch.empty((B, self.K), dtype=torch.uint8, device=self.device)
        check(self.lib.scg_clf_decide(B, ptr(s[0]), ptr(s[1]), ptr(self.theta), self.K, ptr(out), _lib.current_stream()))
        return out.bool()

    def clf_grad(self, k, X, y):
        torch = self.torch
        X = _dev(X, torch.float32).reshape(-1, 2)
        y = _dev(y, torch.uint8)
        g = torch.empty(N_PSI, dtype=torch.float32, device=self.device)
        check(self.lib.scg_clf_grad(X.shape[0], ptr(X), ptr(y), ptr(self.theta[k]), ptr(g), _lib.current_stream()))
        return g

    def fit_initiation(self, k, X, y, steps=200, lr=1.0):
        torch = self.torch
        X = _dev(X, torch.float32).reshape(-1, 2)
        y = _dev(y, torch.uint8)
        if X.shape[0] == 0:
            raise ValueError("no examples")
        check(self.lib.scg_clf_fit(X.shape[0], ptr(X), ptr(y), ptr(self.theta[k]), int(steps), float(lr),
                                   _lib.current_stream()))
        return self.theta[k].clone()


class Option:
    """One option's (initiation, act, update) triple over an OptionSet - the paper's option."""

    def __init__(self, option_set, k):
        self.set = option_set
        self.k = int(k)

    def _ids(self, B):
        t = self.set.torch
        return t.full((B,), self.k, dtype=t.int32, device=self.set.device)

    def q(self, state):
        return self.set.q(state, self._ids(len(state)))

    def initiation(self, state):
        return self.set.initiation(state)[:, self.k]

    def act(self, state, step=0):
        return self.set.act(state, self._ids(len(state)), step)

    def update(self, s, a, r, s2, a2, done):
        return self.set.update(s, a, r, s2, a2, done, self._ids(len(s)))

    def fit_initiation(self, X, y, steps=200, lr=1.0):
        return self.set.fit_initiation(self.k, X, y, steps, lr)
