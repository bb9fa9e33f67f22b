"""Host mirror of `twisterl.twisterl.nn` (rust/src/python_interface/{layers,modules,policy}.rs).

The classes keep the constructor signatures `BasicPolicy.to_rust()` calls
(src/twisterl/nn/utils.py:17-79, src/twisterl/nn/policy.py:191-199); the arithmetic runs on the
device (kernel K2).  Weights stay in the layouts the reference hands over: `Linear` gets
`W.T.flatten()`, `EmbeddingBag` gets `vec_vectors[obs_idx][E]`.
"""
from __future__ import annotations

import ctypes as C

import numpy as np

from . import _lib


def _f32(a) -> np.ndarray:
    return np.ascontiguousarray(a, dtype=np.float32)


class Linear:
    """`nn.Linear(weights_vector, bias_vector, apply_relu)` (python_interface/layers.rs:19-33)."""

    def __init__(self, weights_vector, bias_vector, apply_relu: bool):
        self.bias = _f32(bias_vector).ravel()
        self.weights = _f32(weights_vector).ravel()
        self.out = int(self.bias.size)
        if self.out == 0 or self.weights.size % self.out:
            raise ValueError("weights_vector length must be a multiple of len(bias_vector)")
        self.in_ = self.weights.size // self.out              # layers.rs:26
        self.apply_relu = bool(apply_relu)


class EmbeddingBag:
    """`nn.EmbeddingBag(vec_vectors, bias_vector, apply_relu, obs_shape, conv_dim)` (layers.rs:36-49)."""

    def __init__(self, vec_vectors, bias_vector, apply_relu: bool, obs_shape, conv_dim: int):
        self.vectors = _f32(vec_vectors)
        if self.vectors.ndim != 2:
            raise ValueError("vec_vectors must be a list of equal-length vectors")
        self.bias = _f32(bias_vector).ravel()
        self.apply_relu = bool(apply_relu)
        self.obs_shape = [int(x) for x in obs_shape]
        self.conv_dim = int(conv_dim)


class Sequential:
    """`nn.Sequential(layers)` (python_interface/modules.rs:19-33)."""

    def __init__(self, layers):
        self.layers = list(layers)
        for l in self.layers:
            if not isinstance(l, Linear):
                raise TypeError("Sequential takes a list of nn.Linear")


class Policy:
    """`nn.Policy(embeddings, common, action_net, value_net, obs_perms, act_perms)`
    (python_interface/policy.rs:20-46, rust/src/nn/policy.rs:20-128)."""

    def __init__(self, embeddings: EmbeddingBag, common: Sequential, action_net: Sequential, value_net: Sequential,
                 obs_perms, act_perms):
        self.embeddings, self.common, self.action_net, self.value_net = embeddings, common, action_net, value_net
        as2d = lambda p: (np.ascontiguousarray(p, dtype=np.int32).reshape(len(p), -1) if len(p)
                          else np.zeros((0, 0), dtype=np.int32))
        self.obs_perms, self.act_perms = as2d(obs_perms), as2d(act_perms)
        if len(self.obs_perms) != len(self.act_perms):
            raise ValueError("obs_perms and act_perms must have the same length")
        self._dev = None          # (engine, handle)
        self._keep = None

    # -- C ABI descriptor -----------------------------------------------------------
    def desc(self) -> _lib.PolicyDesc:
        keep = []

        def lin_array(seq: Sequential):
            arr = (_lib.LinearDesc * max(len(seq.layers), 1))()
            for i, l in enumerate(seq.layers):
                arr[i] = _lib.LinearDesc(l.weights.ctypes.data_as(_lib.f32p), l.bias.ctypes.data_as(_lib.f32p),
                                         l.in_, l.out, int(l.apply_relu))
            keep.append(arr)
            return arr

        e = self.embeddings
        d = _lib.PolicyDesc()
        d.emb_vectors = e.vectors.ctypes.data_as(_lib.f32p)
        d.emb_bias = e.bias.ctypes.data_as(_lib.f32p)
        d.obs_size, d.emb_size = int(e.vectors.shape[0]), int(e.bias.size)
        d.emb_apply_relu = int(e.apply_relu)
        d.obs_shape_len = len(e.obs_shape)
        for i, v in enumerate(e.obs_shape[:2]):
            d.obs_shape[i] = v
        d.conv_dim = e.conv_dim
        d.common, d.n_common = lin_array(self.common), len(self.common.layers)
        d.action_net, d.n_action = lin_array(self.action_net), len(self.action_net.layers)
        d.value_net, d.n_value = lin_array(self.value_net), len(self.value_net.layers)
        d.n_perms = int(len(self.obs_perms))
        if d.n_perms:
            d.obs_perms = self.obs_perms.ctypes.data_as(_lib.i32p)
            d.act_perms = self.act_perms.ctypes.data_as(_lib.i32p)
        self._keep = keep
        return d

    @property
    def num_actions(self) -> int:
        if getattr(self, "_native", False):
            return self._native_actions
        return int(self.action_net.layers[-1].out)

    def device_handle(self, engine: _lib.Engine | None = None):
        engine = engine or _lib.default_engine()
        if getattr(self, "_native", False):
            if self._dev is None or self._dev[0] is not engine:
                raise RuntimeError("a policy loaded with from_safetensors lives on the engine it was loaded on")
            return self._dev[1]
        if self._dev is None or self._dev[0] is not engine:
            self.release()
            h = C.c_void_p()
            d = self.desc()
            _lib.check(_lib.load().twr_policy_create(engine._h, C.byref(d), C.byref(h)))
            self._dev = (engine, h)
        return self._dev[1]

    def update_from_torch(self, module, engine: _lib.Engine | None = None) -> None:
        """In-place weight refresh from the LIVE parameters of a torch policy (SURVEY.md 8f row f3): what the reference
        does every iteration through `policy.to_rust()` -- `.cpu().numpy().T.flatten().tolist()` per layer
        (src/twisterl/nn/utils.py:17-59, rl/algorithm.py:91-93) -- becomes device-to-device copies into the engine's
        parameter blob (each Linear as W.T, the layout twr_policy_desc documents) and one operand re-pack
        (twr_policy_update_from_device).  `module` is a BasicPolicy-shaped torch module on the engine's GPU: `embeddings`
        (Linear), `common` / `action` / `value` (Sequentials of Linear and ReLU); this policy must have been built from
        the same architecture (e.g. by `module.to_rust()`).  Raises NotImplementedError for other embedding kinds."""
        import torch
        engine = engine or (self._dev[0] if self._dev is not None else _lib.default_engine())
        h = self.device_handle(engine)
        emb = module.embeddings
        if type(emb).__name__ != "Linear" or len(self.embeddings.obs_shape) != 1:
            raise NotImplementedError("update_from_torch covers the Linear embedding of BasicPolicy; rebuild with to_rust() instead")
        lins = [l for seq in (module.common, module.action, module.value) for l in seq if type(l).__name__ == "Linear"]
        mine = self.common.layers + self.action_net.layers + self.value_net.layers
        if len(lins) != len(mine) or any((l.in_features, l.out_features) != (m.in_, m.out) for l, m in zip(lins, mine)) or \
                tuple(emb.weight.shape) != (self.embeddings.bias.size, self.embeddings.vectors.shape[0]):
            raise ValueError("torch module and engine policy have different architectures")
        L = _lib.load()
        n = int(L.twr_policy_blob_floats(h))
        dptr = C.c_void_p()
        _lib.check(L.twr_policy_blob_device_ptr(h, C.byref(dptr)))
        dev = torch.device("cuda", engine.device)
        if emb.weight.device != dev:
            raise ValueError(f"torch module lives on {emb.weight.device}, the engine on {dev}")

        class _Blob:
            __cuda_array_interface__ = {"shape": (n,), "typestr": "<f4", "data": (int(dptr.value), False), "version": 2}
        blob = torch.as_tensor(_Blob(), device=dev)
        off = 0

        def put(t, shape):
            nonlocal off
            k = int(np.prod(shape))
            blob[off:off + k].view(*shape).copy_(t.detach())
            off += k
        with torch.no_grad():
            E, O = emb.weight.shape
            put(emb.weight.T, (O, E))                              # vec_vectors[obs][E]
            put(emb.bias if getattr(emb, "bias", None) is not None else torch.zeros(E, device=dev), (E,))
            for l in lins:
                put(l.weight.T, (l.in_features, l.out_features))   # W.T.flatten(): w[i*out + o] == W[o][i]
                put(l.bias, (l.out_features,))
        assert off == n
        torch.cuda.current_stream(dev).synchronize()               # the engine refreshes its operand tiles on its own stream
        _lib.check(L.twr_policy_update_from_device(h, dptr))

    def release(self):
        if self._dev is not None:
            eng, h = self._dev
            if getattr(eng, "_h", None):
                _lib.load().twr_policy_destroy(h)
            self._dev = None

    @classmethod
    def from_safetensors(cls, path, obs_shape=None, conv_dim: int = 0, obs_perms=(), act_perms=(), engine: _lib.Engine | None = None):
        """Device policy built by the library's native safetensors reader (twr_policy_create_from_safetensors) from a
        checkpoint of the reference's BasicPolicy / Conv1dPolicy state dict -- no torch, no to_rust() round trip.
        The result only lives on `engine` (no host copy of the weights; `predict` / `desc` are not available)."""
        engine = engine or _lib.default_engine()
        self = cls.__new__(cls)
        two_d = lambda a: (np.ascontiguousarray(a, dtype=np.int32).reshape(len(a), -1) if len(a) else np.zeros((0, 0), np.int32))
        self.obs_perms, self.act_perms = two_d(obs_perms), two_d(act_perms)
        self._keep = None
        self._native_actions = int(self.act_perms.shape[1]) if len(act_perms) else 4
        shape = np.ascontiguousarray(obs_shape if obs_shape is not None else [], dtype=np.int32)
        h = C.c_void_p()
        n_perms = int(len(obs_perms))
        _lib.check(_lib.load().twr_policy_create_from_safetensors(
            engine._h, str(path).encode(), shape.ctypes.data_as(_lib.i32p) if shape.size else None, int(shape.size), int(conv_dim),
            self.obs_perms.ctypes.data_as(_lib.i32p) if n_perms else None, self.act_perms.ctypes.data_as(_lib.i32p) if n_perms else None,
            n_perms, C.byref(h)))
        self._dev = (engine, h)
        self._native = True
        return self

    def __del__(self):
        try:
            self.release()
        except Exception:
            pass

    # -- scalar API of the reference ---------------------------------------------------
    def _raw(self, obs, perm_idx: int, engine=None):
        """_raw_predict (nn/policy.rs:79-100) of one sparse observation, on the device."""
        engine = engine or _lib.default_engine()
        return forward_obs(engine, self, [list(obs)], None if perm_idx < 0 else [perm_idx])

    def _pick_perm(self) -> int:
        # get_perm_id (nn/policy.rs:67-77): uniform over the twists; the reference is unseeded here too
        return int(np.random.randint(len(self.obs_perms))) if len(self.obs_perms) else -1

    def forward(self, obs, masks):
        logits, value = self._raw(obs, self._pick_perm())
        l = np.where(np.asarray(masks, dtype=bool), logits[0], np.float32(-1e10)).astype(np.float32)   # policy.rs:62
        return [float(x) for x in l], float(value[0])

    def predict(self, obs, masks):
        logits, value = self._raw(obs, self._pick_perm())
        return _masked_exp_normalise(logits[0], masks), float(value[0])

    def full_predict(self, obs, masks):
        if len(self.obs_perms) == 0:
            return self.predict(obs, masks)
        n = np.float32(len(self.obs_perms))
        acc = np.zeros(self.num_actions, dtype=np.float32)
        val = np.float32(0)
        for pi in range(len(self.obs_perms)):                  # policy.rs:109-115
            l, v = self._raw(obs, pi)
            val = np.float32(val + v[0] / n)
            acc = (acc + l[0] / n).astype(np.float32)
        return _masked_exp_normalise(acc, masks), float(val)


def _masked_exp_normalise(logits, masks):
    m = np.asarray(masks, dtype=bool)
    e = np.where(m, np.exp(logits.astype(np.float32)), np.float32(0)).astype(np.float32)   # policy.rs:43-47
    s = np.float32(e.sum(dtype=np.float32) + np.float32(1e-6))
    return [float(x) for x in (e / s)]


def forward_batch(engine: _lib.Engine, policy: Policy, batch, perm_idx=None, apply_masks: bool = False):
    """Batched _raw_predict / forward_with_perm (twr_policy_forward): (logits [n][A], values [n])."""
    n, A = batch.n, policy.num_actions
    logits = np.zeros((n, A), dtype=np.float32)
    values = np.zeros(n, dtype=np.float32)
    pi = None
    if perm_idx is not None:
        pi = np.ascontiguousarray(perm_idx, dtype=np.int32).reshape(n)
    _lib.check(_lib.load().twr_policy_forward(engine._h, policy.device_handle(engine), batch._h,
                                              _lib.ptr(pi) if pi is not None else None, int(apply_masks),
                                              _lib.ptr(logits), _lib.ptr(values)))
    return logits, values


def full_predict_batch(engine: _lib.Engine, policy: Policy, batch):
    """Batched Policy::full_predict (twr_policy_full_predict), the leaf evaluation of the MCTS searches:
    (probs [n][A], values [n])."""
    n, A = batch.n, policy.num_actions
    probs = np.zeros((n, A), dtype=np.float32)
    values = np.zeros(n, dtype=np.float32)
    _lib.check(_lib.load().twr_policy_full_predict(engine._h, policy.device_handle(engine), batch._h,
                                                   _lib.ptr(probs), _lib.ptr(values)))
    return probs, values


def forward_obs(engine: _lib.Engine, policy: Policy, obs, perm_idx=None):
    """Batched _raw_predict on sparse observations given directly (twr_policy_forward_obs)."""
    o = np.ascontiguousarray(obs, dtype=np.int32)
    n, n_obs = o.shape
    logits = np.zeros((n, policy.num_actions), dtype=np.float32)
    values = np.zeros(n, dtype=np.float32)
    pi = None if perm_idx is None else np.ascontiguousarray(perm_idx, dtype=np.int32).reshape(n)
    _lib.check(_lib.load().twr_policy_forward_obs(engine._h, policy.device_handle(engine), _lib.ptr(o), n, n_obs,
                                                  _lib.ptr(pi) if pi is not None else None, _lib.ptr(logits),
                                                  _lib.ptr(values)))
    return logits, values
