"""The DLRM operators either side of the cache, behind the reference's own names
(dlrm_s_pytorch_C1_C2_C3.py): ``apply_emb_evstore`` (:226-267), ``apply_emb_ori_dlrm`` (:191-223),
``interact_features`` (:625-658, op "dot").  All of them run hand-written CUDA kernels through the
C-ABI; inputs and outputs are CUDA tensors.

Differences from the reference, on purpose:
* the reference's apply_emb_evstore serves batch element 0 only (``sparse_index[0]``, :236-239;
  its drivers force --test-mini-batch-size=1); here the whole ``lS_i [n_tables, B]`` batch is
  served in one call and every returned tensor is ``[B, dim]`` (a view of one ``[B, n_tables, dim]``
  buffer) instead of ``[1, dim]``;
* ``cache_algo`` names the policy of the GPU cache: "cpp_algo", "evlfu" and "lfu" (the reference's
  EvLFU_C1 branch is keyed "lfu", :249) need an EvStore built with ``policy="evlfu"``, "lru" (:251,
  cache_algo/LRU.py) one built with ``policy="lru"``; the policy is a property of the cache, so a mismatch
  raises instead of silently serving another policy.  The plain LFU of cache_algo/LFU.py (unreachable in
  the reference too: its ``elif cache_algo == "lfu"`` at :253 is shadowed by :249) is not available.
"""
from __future__ import annotations

import ctypes as C

from . import _native
from .cache_manager import EvStore, _stream_handle

cache_algo = "cpp_algo"        # --cache-algo (dlrm_s_pytorch_C1_C2_C3.py:1229)
evstore_gpu_id = 0             # --evstore-gpu-id
_store: EvStore | None = None  # the cache the module-level operator uses (set_store)
last_hit = None                # aggHitMissRecord of the last call: uint8 [B, n_tables]


def set_store(store: EvStore):
    global _store
    _store = store


def apply_emb_evstore(lS_o, lS_i, emb_l=None, v_W_l=None, use_gpu=True, use_emb_cache=True, approx_emb_threshold=-1,
                      store: EvStore | None = None, out=None):
    """lS_i: int64 CUDA tensor [n_tables, B] (or a list of n_tables [B] tensors); lS_o is ignored, as
    in the reference (pooling factor 1).  Returns ly: list of n_tables tensors [B, dim]."""
    global last_hit
    import torch
    st = store or _store
    if st is None:
        raise RuntimeError("apply_emb_evstore: no EvStore (call dlrm_ops.set_store)")
    if isinstance(lS_i, (list, tuple)):
        lS_i = torch.stack(list(lS_i))
    if not lS_i.is_cuda:
        raise RuntimeError("apply_emb_evstore runs on the GPU cache: pass CUDA indices (there is no CPU fallback)")
    lS_i = lS_i.contiguous()
    if use_emb_cache:
        if cache_algo not in ("cpp_algo", "evlfu", "lfu", "lru"):
            raise ValueError("ERROR: This algorithm is not yet supported! " + str(cache_algo))
        want = "lru" if cache_algo == "lru" else "evlfu"
        if st.cfg.policy != want:
            raise ValueError(f"cache_algo {cache_algo!r} needs an EvStore with policy={want!r}; this one has policy={st.cfg.policy!r}")
        if approx_emb_threshold > 0 and st.cfg.approx_emb_thres != approx_emb_threshold:
            raise ValueError("approx_emb_threshold is a property of the cache: set CacheConfig.approx_emb_thres")
        buf, last_hit = st.lookup(lS_i, out=out)
    else:
        buf = st.storage_lookup(lS_i, out=out)          # storage_manager.request_to_emb_storage (:264)
    return [buf[:, k, :] for k in range(buf.shape[1])]


def embedding_bag(table, indices, offsets, per_sample_weights=None, precision=32, dim=None, out=None, stream=None):
    """nn.EmbeddingBag(mode="sum") on one table.  table: CUDA tensor [rows, dim] fp32, or raw rows
    (uint16 / uint8) at `precision` bits with `dim` given."""
    import torch
    lib = _native.load_library()
    rows = table.shape[0]
    d = dim or table.shape[1]
    B = offsets.numel()
    if out is None:
        out = torch.empty((B, d), dtype=torch.float32, device=indices.device)
    st = _stream_handle(stream, indices.device)
    rc = lib.evs_embedding_bag(table.data_ptr(), rows, d, precision, indices.data_ptr(), offsets.data_ptr(),
                               indices.numel(), B, per_sample_weights.data_ptr() if per_sample_weights is not None else None,
                               out.data_ptr(), out.stride(0), st)
    _native.check(rc, "evs_embedding_bag")
    return out


def apply_emb_ori_dlrm(lS_o, lS_i, emb_l, v_W_l=None):
    """emb_l: list of fp32 CUDA weight tensors [rows_k, dim] (nn.EmbeddingBag.weight).  Returns ly."""
    ly = []
    for k, idx in enumerate(lS_i):
        w = None
        if v_W_l is not None and v_W_l[k] is not None:
            w = v_W_l[k].gather(0, idx)                 # dlrm_s_pytorch_C1_C2_C3.py:208
        E = emb_l[k].weight if hasattr(emb_l[k], "weight") else emb_l[k]
        ly.append(embedding_bag(E, idx, lS_o[k], w))
    return ly


def _check_fp32_cuda(name, t, dims, device=None):
    import torch
    if not isinstance(t, torch.Tensor):
        raise ValueError(f"interact_features: {name} must be a tensor, not {type(t).__name__}")
    if t.dtype != torch.float32:
        raise ValueError(f"interact_features: {name} must be float32, not {t.dtype}")
    if not t.is_cuda or (device is not None and t.device != device):
        raise ValueError(f"interact_features: {name} is on {t.device}, the interaction runs on {device or 'a CUDA device'}")
    if t.dim() != dims:
        raise ValueError(f"interact_features: {name} must have {dims} dimensions, not shape {tuple(t.shape)}")


def interact_features(x, ly, out=None, stream=None):
    """x [B, d], ly: list of n_f tensors [B, d] (or one [B, n_f, d] tensor) -> [B, d + (n_f+1) n_f / 2].
    Everything is float32 on one CUDA device; `out`, when given, must be a contiguous [B, d + (n_f+1) n_f / 2] tensor.
    A list of views ``buf[:, k, :]`` of one contiguous [B, n_f, d] buffer (what apply_emb_evstore returns) is read in
    place; any other list is stacked into one first."""
    import torch
    lib = _native.load_library()
    _check_fp32_cuda("x", x, 2)
    B, d = x.shape
    if isinstance(ly, (list, tuple)):
        if not ly:
            raise ValueError("interact_features: ly is an empty list")
        for k, t in enumerate(ly):
            _check_fp32_cuda(f"ly[{k}]", t, 2, x.device)
            if tuple(t.shape) != (B, d):
                raise ValueError(f"interact_features: ly[{k}] has shape {tuple(t.shape)}, x has {(B, d)}")
        n_f = len(ly)
        base = ly[0]._base
        same = base is not None and tuple(base.shape) == (B, n_f, d) and base.is_contiguous() and all(
            t._base is base and t.stride() == (n_f * d, 1) and t.data_ptr() == base.data_ptr() + k * d * 4
            for k, t in enumerate(ly))
        lyt = base if same else torch.stack(list(ly), dim=1).contiguous()
    else:
        _check_fp32_cuda("ly", ly, 3, x.device)
        if ly.shape[0] != B or ly.shape[2] != d:
            raise ValueError(f"interact_features: ly has shape {tuple(ly.shape)}, x has {(B, d)}: want [{B}, n_f, {d}]")
        lyt = ly.contiguous()
    n_f = lyt.shape[1]
    want = (B, d + (n_f + 1) * n_f // 2)
    if out is None:
        out = torch.empty(want, dtype=torch.float32, device=x.device)
    else:
        _check_fp32_cuda("out", out, 2, x.device)
        if tuple(out.shape) != want or not out.is_contiguous():
            raise ValueError(f"interact_features: out must be a contiguous {want} tensor, not shape {tuple(out.shape)} "
                             f"with strides {out.stride()}")
    st = _stream_handle(stream, x.device)
    _native.check(lib.evs_interact(x.contiguous().data_ptr(), lyt.data_ptr(), out.data_ptr(), B, n_f, d, st), "evs_interact")
    return out


class DLRMInference:
    """The inference half of ``DLRM_Net`` around the cache: ``sequential_forward``
    (dlrm_s_pytorch_C1_C2_C3.py:742-768) = bottom MLP -> apply_emb -> interact_features -> top MLP ->
    optional clamp, with ``apply_mlp`` / ``create_mlp`` semantics (:117-119, 207-245: Linear + ReLU, a
    Sigmoid after layer ``sigmoid_layer``).  The MLPs are plain library GEMMs (``F.linear`` -> cuBLAS, fp32,
    TF32 off); the lookup and the interaction are this package's kernels.  The bottom MLP does not depend
    on the lookup, so it runs on a side stream next to it.

    bot / top: lists of (weight [out, in], bias [out]) -- ``nn.Linear`` parameters as numpy arrays or tensors.
    """

    def __init__(self, bot, top, store: EvStore, sigmoid_bot: int = -1, sigmoid_top: int | None = None,
                 loss_threshold: float = 0.0, use_emb_cache: bool = True):
        import torch
        self.store = store
        self.device = torch.device("cuda", store.cfg.device)
        as_t = lambda a: torch.as_tensor(a, dtype=torch.float32).to(self.device).contiguous()
        self.bot = [(as_t(w), as_t(b)) for w, b in bot]
        self.top = [(as_t(w), as_t(b)) for w, b in top]
        self.sigmoid_bot = sigmoid_bot
        self.sigmoid_top = len(self.top) - 1 if sigmoid_top is None else sigmoid_top
        self.loss_threshold = loss_threshold
        self.use_emb_cache = use_emb_cache
        self._side = torch.cuda.Stream(device=self.device)
        d = self.bot[-1][0].shape[0]
        if d != store.dim:
            raise ValueError(f"bottom MLP ends in {d} features, the embedding dimension is {store.dim}")
        n_f = store.n_tables
        want = d + (n_f + 1) * n_f // 2
        if self.top[0][0].shape[1] != want:
            raise ValueError(f"top MLP takes {self.top[0][0].shape[1]} features, the dot interaction produces {want}")

    @staticmethod
    def apply_mlp(x, layers, sigmoid_layer: int):
        import torch
        import torch.nn.functional as F
        for i, (w, b) in enumerate(layers):
            x = F.linear(x, w, b)
            x = torch.sigmoid(x) if i == sigmoid_layer else torch.relu(x)
        return x

    def sequential_forward(self, dense_x, lS_o, lS_i):
        """dense_x [B, 13] fp32, lS_i int64 [n_tables, B] (CUDA); lS_o is ignored like in apply_emb_evstore.
        Returns the click probabilities [B, 1]."""
        import torch
        prev = torch.backends.cuda.matmul.allow_tf32
        torch.backends.cuda.matmul.allow_tf32 = False
        try:
            cur = torch.cuda.current_stream(self.device)
            self._side.wait_stream(cur)
            with torch.cuda.stream(self._side):
                x = self.apply_mlp(dense_x, self.bot, self.sigmoid_bot)
            ly = apply_emb_evstore(lS_o, lS_i, use_emb_cache=self.use_emb_cache, store=self.store)
            cur.wait_stream(self._side)
            x.record_stream(cur)
            z = interact_features(x, ly)
            p = self.apply_mlp(z, self.top, self.sigmoid_top)
        finally:
            torch.backends.cuda.matmul.allow_tf32 = prev
        if 0.0 < self.loss_threshold < 1.0:
            p = torch.clamp(p, min=self.loss_threshold, max=1.0 - self.loss_threshold)
        return p

    # ---- the whole forward as one CUDA graph -----------------------------------------------------------------------
    def capture(self, batch: int, n_dense: int | None = None):
        """Capture ``sequential_forward`` for batches of ``batch`` samples into ONE CUDA graph: the bottom MLP branch, the
        cache's serve / update / evict kernels, the interaction and the top MLP, with their dependencies -- a forward is then
        a single graph launch instead of a dozen kernel launches and two stream joins.  Call ``replay(dense_x, lS_i)``."""
        import torch
        n_dense = n_dense or self.bot[0][0].shape[1]
        self._g_dense = torch.zeros((batch, n_dense), dtype=torch.float32, device=self.device)
        self._g_idx = torch.zeros((self.store.n_tables, batch), dtype=torch.int64, device=self.device)
        # one eager pass on a side stream first (library handles, workspaces), as torch's capture rules ask
        warm = torch.cuda.Stream(device=self.device)
        warm.wait_stream(torch.cuda.current_stream(self.device))
        with torch.cuda.stream(warm):
            self.sequential_forward(self._g_dense, None, self._g_idx)
        torch.cuda.current_stream(self.device).wait_stream(warm)
        torch.cuda.synchronize(self.device)
        self._graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(self._graph):
            self._g_out = self.sequential_forward(self._g_dense, None, self._g_idx)
        return self

    def replay(self, dense_x, lS_i):
        """One captured forward: fills the static inputs, launches the graph, returns the (static) probabilities [B, 1]."""
        self._g_dense.copy_(dense_x, non_blocking=True)
        self._g_idx.copy_(lS_i, non_blocking=True)
        self._graph.replay()
        self.store.note_replays(1)
        return self._g_out
