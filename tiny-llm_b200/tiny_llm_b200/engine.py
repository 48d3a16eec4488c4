"""CUDA-graph decode engine for the Week-3 paged model (B200 host runtime).

The reference issues ~500 operator calls per generated token from a Python loop
(SURVEY.md section 3.1); at B200 speeds one W4A16 projection lasts about a
microsecond, so per-call dispatch would leave the GPU idle >90 % of the time.
The engine keeps the operator semantics and removes the dispatch:

* one decode step (embedding -> 36 blocks -> norm -> tied head -> greedy
  argmax) for a fixed number of slots ``B`` is captured once into a CUDA graph
  over static buffers and replayed per step;
* everything the step needs from the scheduler is DATA, not kernel arguments:
  token ids, RoPE offsets, post-append context lengths and the per-layer block
  tables live in one device buffer that is refreshed with a single pinned
  host->device copy; K/V appends and attention read page ids from it;
* the integer page bookkeeping stays on the host in the very same
  ``TinyKvPagedCache`` / ``TinyKvPagedPool`` objects the per-operator path uses
  (``append_token_slot``), so block tables, page ids and counters are identical;
* ``decode_on_device`` runs N greedy steps with no host involvement at all
  (token feedback + position advance by ``tl_decode_advance``, pages allocated
  ahead) - the device-resident number of bench.py.

Page slabs must not move while a graph is alive: pools are ``reserve()``d up
front and the engine re-captures if a slab pointer changes.
"""

from __future__ import annotations

import contextlib
import gc
import os

from types import SimpleNamespace

import numpy as np
import torch

from extensions_b200 import tiny_llm_ext_b200 as ext

from .kv_cache import BatchingKvCache
from .paged_kv_cache import TinyKvPagedCache


@contextlib.contextmanager
def _gc_paused():
    """No cyclic garbage collection during a graph capture.  An engine and its model reference each other, so a
    dropped model is freed by the collector; destroying its CUDA graphs while a stream captures is a CUDA call
    that capture forbids, and it invalidates the capture in progress."""
    enabled = gc.isenabled()
    gc.disable()
    try:
        yield
    finally:
        if enabled:
            gc.enable()


def _concat_weights(parts):
    """Stack packed projections along the output dimension (one launch instead of
    len(parts)): rows of codes, scales and biases are simply concatenated."""
    first = parts[0]
    return SimpleNamespace(
        weight=torch.cat([p.weight.view(torch.int32) if p.weight.dtype == torch.uint32 else p.weight for p in parts], dim=0).contiguous(),
        scales=torch.cat([p.scales for p in parts], dim=0).contiguous(),
        biases=torch.cat([p.biases for p in parts], dim=0).contiguous(),
        group_size=first.group_size,
        bits=first.bits,
    )


def _interleave_gate_up(gate, up):
    """gate|up rows in blocks of 8 (``ext.interleave_gate_up``): the streaming kernel's
    EPI_SWIGLU_PAIRS epilogue then emits swiglu(gate, up) directly, so the MLP activation never
    makes a round trip through memory as two separate vectors."""
    as_i32 = lambda w: w.view(torch.int32) if w.dtype == torch.uint32 else w
    return SimpleNamespace(
        weight=ext.interleave_gate_up(as_i32(gate.weight), as_i32(up.weight)),
        scales=ext.interleave_gate_up(gate.scales, up.scales),
        biases=ext.interleave_gate_up(gate.biases, up.biases),
        group_size=gate.group_size,
        bits=gate.bits,
    )


class _LockstepGroup:
    """The per-layer cache objects of ONE request plus the number of one-token appends the engine
    has accounted for but not yet written into them (see ``TinyKvPagedCache._lazy``)."""

    __slots__ = ("caches", "pending")

    def __init__(self, caches):
        self.caches = caches
        self.pending = 0

    def settle(self) -> None:
        n = self.pending
        if n:
            self.pending = 0
            for c in self.caches:
                c._page_lens[-1] += n
                c._offset += n


class _SlotRecord:
    """What the engine knows about the request in one decode slot."""

    __slots__ = ("c0", "group", "lockstep", "epoch", "offset", "pages")

    def __init__(self, c0, group, lockstep):
        self.c0, self.group, self.lockstep = c0, group, lockstep
        self.epoch = c0.epoch
        self.offset = c0._offset      # logical context length (settled offset + pending)
        self.pages = len(c0.page_ids)


class DecodeEngine:
    def __init__(self, model, batch_size: int, max_seq_len: int, device, log_capacity: int = 4096, fused: bool = True):
        self.model = model
        self.B = batch_size
        self.device = torch.device(device)
        self.page_size = model.page_size
        self.max_pages = (max_seq_len + self.page_size - 1) // self.page_size
        self.max_seq_len = self.max_pages * self.page_size
        self.n_layers = model.num_hidden_layers
        attn = model.layers_inner[0].self_attn
        self.Hq, self.Hkv, self.D = attn.num_heads, attn.num_kv_heads, attn.head_dim
        self.V = model.vocab_size
        self.log_capacity = log_capacity

        B, Ly, MP = self.B, self.n_layers, self.max_pages
        # one int32 block: tokens | offsets | context_lens | block tables [Ly, B, MP]
        self._meta_len = 3 * B + Ly * B * MP
        self.meta_host = torch.empty(self._meta_len, dtype=torch.int32, pin_memory=True)
        self.meta_np = self.meta_host.numpy()
        self.meta_np[: 3 * B] = 0
        self.meta_np[3 * B :] = -1
        self.meta_dev = torch.zeros(self._meta_len, dtype=torch.int32, device=self.device)
        self._meta_dev_head, self._meta_host_head = self.meta_dev[: 3 * B], self.meta_host[: 3 * B]  # the per-step upload
        self.tokens = self.meta_dev[0:B]
        self.offsets = self.meta_dev[B : 2 * B]
        self.context_lens = self.meta_dev[2 * B : 3 * B]
        self.tables = self.meta_dev[3 * B :].view(Ly, B, MP)
        self.tables_np = self.meta_np[3 * B :].reshape(Ly, B, MP)
        self.next_tokens = torch.zeros(B, dtype=torch.int32, device=self.device)
        self.out_log = torch.full((log_capacity * B,), -1, dtype=torch.int32, device=self.device)
        self.step_counter = torch.zeros(1, dtype=torch.int32, device=self.device)
        self.logits = None
        # per slot: the request group (its per-layer cache objects) the table rows reflect
        self._recs: list[_SlotRecord | None] = [None] * B
        self._tables_dirty = True
        self._upload_event = torch.cuda.Event()
        self._upload_pending = False
        self.h2d_bytes = 0  # bytes copied host -> device by step() / decode_on_device() so far
        self._graph = None
        self._graph_loop = None
        self._slab_ptrs = None
        self._stream = torch.cuda.Stream(device=self.device)
        self.graph_replays = 0
        self.captures = 0  # graph (re-)captures: 1 + one per move of the page slabs
        self.kernels_per_step = 0
        rope = attn.rope
        self.fused = bool(fused) and not rope.traditional and rope.dims == self.D and self.D % 2 == 0
        self._packed = None
        if self.fused:
            # q|k|v and gate|up share their input, so they stream as one launch each.
            self._packed = [
                SimpleNamespace(
                    qkv=_concat_weights([b.self_attn.wq, b.self_attn.wk, b.self_attn.wv]),
                    gate_up=_interleave_gate_up(b.mlp.w_gate, b.mlp.w_up),
                )
                for b in model.layers_inner
            ]
        # one-launch attention (q/k norm + rope + append + paged GQA) when the head layout allows it
        attn0 = model.layers_inner[0].self_attn
        # The one-launch attention is a latency design (few CTAs, K/V rows staged per lane): it wins while the
        # step is launch-bound.  With many slots or long contexts the K/V stream dominates and the step uses
        # q/k norm + rope + append as one small launch followed by tl_paged_attention, whose long-context path
        # is the TMA + tcgen05 streaming kernel (attention_prefill_tc.cu).  TL_ATTENTION_FUSED=0/1 forces either.
        fused_env = os.environ.get("TL_ATTENTION_FUSED")
        fused_pays = self.B * self.max_seq_len <= int(os.environ.get("TL_ATTENTION_FUSED_MAX_TOKENS", "16384"))
        self._attention_fused = (self.fused and self.D == 128 and self.Hq // self.Hkv <= 4
                                 and model.embedding.weight.scales.dtype == torch.bfloat16
                                 and not getattr(attn0.rope, "traditional", False)
                                 and (fused_env == "1" or (fused_env != "0" and fused_pays)))
        if self._attention_fused:
            self._rope_inv_freq = ext.rope_inv_freq_table(self.D, attn0.rope.base, self.device)
            self._attn_ws = torch.empty(ext.decode_attention_fused_workspace(self.B, self.Hq, self.Hkv), dtype=torch.float32, device=self.device)
        # Row variants: the scheduler fills slots from index 0 (batch.py:220-226), so while few requests are live the
        # occupied slots are a prefix of the table.  A step graph over the first 16 / 32 rows is captured beside the
        # full one and step() replays the smallest that covers the highest occupied slot: every kernel of the wide
        # path costs by rows (swap-AB column count, attention CTAs, reduction planes).  All variants stay on the
        # >= 9-row kernels and the split counts do not depend on the row count, so a row's result is bit-identical
        # whichever variant computed it.  (Config 4 runs 64 slots with ~20 live: decode step p50 3.31 -> 3.02 ms.)
        rows_env = os.environ.get("TL_ROW_VARIANTS", "1")
        self._variants = sorted({r for r in (16, 32, 64) if r < self.B} | {self.B}) if (self.fused and self.B > 16 and rows_env != "0") else [self.B]
        self._graphs: dict = {}
        self.variant_replays = {r: 0 for r in self._variants}

    # ------------------------------------------------------------------ pools --
    def reserve_pools(self, pages_per_layer: int | None = None) -> None:
        pages = pages_per_layer if pages_per_layer is not None else self.B * self.max_pages + 1
        for pool in self.model.page_pools:
            pool.reserve(pages, self.Hkv, self.D, dtype=torch.bfloat16, device=self.device)

    def _slabs(self):
        return tuple(p.slab_version for p in self.model.page_pools)  # changes whenever a pool's slabs are (re)allocated

    # ------------------------------------------------------------ graph body --
    def _forward_unfused(self) -> None:
        """One decode step over the static buffers, operator by operator (the
        call sequence of qwen3_week3.py:55-121,139-146,196-207,320-338 at L == 1)."""
        m = self.model
        B, Hq, Hkv, D = self.B, self.Hq, self.Hkv, self.D
        emb = m.embedding.weight
        x = ext.quantized_embedding(self.tokens, emb.scales, emb.biases, emb.weight, emb.group_size, emb.bits)  # [B, H]

        def proj(h, w):
            return ext.quantized_matmul(w.scales, w.biases, w.group_size, w.bits, h, w.weight, True)

        for i, block in enumerate(m.layers_inner):
            at = block.self_attn
            pool = m.page_pools[i]
            h = ext.rms_norm(x, block.input_layernorm._weight_as(x.dtype, x.device), block.input_layernorm.eps)
            q = proj(h, at.wq).view(B, 1, Hq, D)
            k = proj(h, at.wk).view(B, 1, Hkv, D)
            v = proj(h, at.wv).view(B, Hkv, 1, D)
            q = ext.rms_norm(q, at.q_norm._weight_as(x.dtype, x.device), at.q_norm.eps)
            k = ext.rms_norm(k, at.k_norm._weight_as(x.dtype, x.device), at.k_norm.eps)
            q = ext.rope(q, self.offsets, at.rope.dims, at.rope.base, at.rope.traditional)
            k = ext.rope(k, self.offsets, at.rope.dims, at.rope.base, at.rope.traditional)
            ext.paged_cache_append_decode(pool._key_pages, pool._value_pages, k.view(B, Hkv, 1, D), v, self.tables[i], self.context_lens)
            y = ext.paged_attention(q.view(B * Hq, 1, D), pool._key_pages, pool._value_pages, self.tables[i], self.context_lens,
                                    at.scale, is_causal=True, num_kv_heads=Hkv, num_heads=Hq)
            x = ext.add(x, proj(y.view(B, Hq * D), at.wo))
            h = ext.rms_norm(x, block.post_attention_layernorm._weight_as(x.dtype, x.device), block.post_attention_layernorm.eps)
            mlp = block.mlp
            x = ext.add(x, proj(ext.swiglu(proj(h, mlp.w_gate), proj(h, mlp.w_up)), mlp.w_down))
        x = ext.rms_norm(x, m.norm._weight_as(x.dtype, x.device), m.norm.eps)
        head = m.w_lm_head if m.w_lm_head is not None else m.embedding.weight
        logits = proj(x, head)
        self.next_tokens.copy_(ext.argmax(logits))
        if self.logits is None:
            self.logits = torch.empty_like(logits)
        self.logits.copy_(logits)

    def _forward_fused(self, rows: int | None = None) -> None:
        """Same step in ~7 launches per layer: norm / SwiGLU / residual folded into
        the streaming projections, q/k norm + RoPE + K/V append in one kernel.
        Every rounding point of the operator-by-operator sequence is kept.
        ``rows``: only the first ``rows`` slots (a row variant, see __init__)."""
        m = self.model
        R = self.B if rows is None else rows
        emb = m.embedding.weight
        x = ext.quantized_embedding(self.tokens[:R], emb.scales, emb.biases, emb.weight, emb.group_size, emb.bits)
        logits = self._forward_fused_layers(x, R)
        self.next_tokens[:R].copy_(ext.argmax(logits))
        if self.logits is None:
            self.logits = torch.zeros((self.B, logits.shape[-1]), dtype=logits.dtype, device=logits.device)
        self.logits[:R].copy_(logits)

    def _forward_fused_layers(self, x, R: int | None = None):
        m = self.model
        B, Hq, Hkv, D = (self.B if R is None else R), self.Hq, self.Hkv, self.D
        offsets, context_lens = self.offsets[:B], self.context_lens[:B]
        # More than 8 rows: the projections run on the swap-AB tcgen05 kernel (w4a16_skinny.cu: weights streamed once
        # for all rows), which has no prologue, so RMSNorm is its own (tiny) launch; the rounding points are the same.
        wide = self.B > 8

        def normed(h, norm):
            return ext.rms_norm(h, norm._weight_as(h.dtype, h.device), norm.eps)

        layers = list(m.layers_inner)
        # wide path: the residual projections (o, down) hand the NEXT RMSNorm's output back together with the residual
        # stream (one launch: the kernel that adds the split-reduction planes has the whole row in registers)
        h = normed(x, layers[0].input_layernorm) if wide else None
        for i, block in enumerate(layers):
            at, pk, pool = block.self_attn, self._packed[i], m.page_pools[i]
            ln1, ln2 = block.input_layernorm, block.post_attention_layernorm
            qkv = None
            if wide and self._attention_fused:
                qkv = ext.quantized_matmul_fused(pk.qkv.scales, pk.qkv.biases, pk.qkv.weight, h)
            elif not wide:
                qkv = ext.quantized_matmul_fused(pk.qkv.scales, pk.qkv.biases, pk.qkv.weight, x, ln1._weight_as(x.dtype, x.device),
                                                 prologue=ext.PRO_RMSNORM, eps=ln1.eps)
            if self._attention_fused:
                y = ext.decode_attention_fused(qkv, at.q_norm._weight_as(x.dtype, x.device), at.k_norm._weight_as(x.dtype, x.device),
                                               offsets, self.tables[i][:B], context_lens, self._rope_inv_freq,
                                               pool._key_pages, pool._value_pages, Hq, Hkv, at.q_norm.eps, at.scale,
                                               self.max_seq_len, workspace=self._attn_ws)
            else:
                if wide:  # projection + q/k norm + RoPE + append: the split-reduction planes feed the second kernel, q|k|v is never written
                    q = ext.qkv_project_rope_append(pk.qkv.scales, pk.qkv.biases, pk.qkv.weight, h, at.q_norm._weight_as(x.dtype, x.device),
                                                    at.k_norm._weight_as(x.dtype, x.device), offsets, self.tables[i][:B], context_lens,
                                                    pool._key_pages, pool._value_pages, Hq, Hkv, at.rope.base, at.q_norm.eps)
                else:
                    q = ext.decode_qk_norm_rope_append(qkv, at.q_norm._weight_as(x.dtype, x.device), at.k_norm._weight_as(x.dtype, x.device),
                                                       offsets, self.tables[i][:B], context_lens, pool._key_pages, pool._value_pages,
                                                       Hq, Hkv, at.rope.base, at.q_norm.eps)
                y = ext.paged_attention(q.view(B * Hq, 1, D), pool._key_pages, pool._value_pages, self.tables[i][:B], context_lens,
                                        at.scale, is_causal=True, num_kv_heads=Hkv, num_heads=Hq)
            wd = block.mlp.w_down
            if wide:
                x, h = ext.quantized_matmul_residual_norm(at.wo.scales, at.wo.biases, at.wo.weight, y.view(B, Hq * D), x,
                                                          ln2._weight_as(x.dtype, x.device), ln2.eps)
                act = ext.quantized_matmul_fused(pk.gate_up.scales, pk.gate_up.biases, pk.gate_up.weight, h, epilogue=ext.EPI_SWIGLU_PAIRS)
                nxt = layers[i + 1].input_layernorm if i + 1 < len(layers) else m.norm
                x, h = ext.quantized_matmul_residual_norm(wd.scales, wd.biases, wd.weight, act, x, nxt._weight_as(x.dtype, x.device), nxt.eps)
                continue
            x = ext.quantized_matmul_fused(at.wo.scales, at.wo.biases, at.wo.weight, y.view(B, Hq * D), residual=x, epilogue=ext.EPI_RESIDUAL)
            act = ext.quantized_matmul_fused(pk.gate_up.scales, pk.gate_up.biases, pk.gate_up.weight, x, ln2._weight_as(x.dtype, x.device),
                                             prologue=ext.PRO_RMSNORM, eps=ln2.eps, epilogue=ext.EPI_SWIGLU_PAIRS)  # [B, inter]
            x = ext.quantized_matmul_fused(wd.scales, wd.biases, wd.weight, act, residual=x, epilogue=ext.EPI_RESIDUAL)
        head = m.w_lm_head if m.w_lm_head is not None else m.embedding.weight
        if wide:
            return ext.quantized_matmul_fused(head.scales, head.biases, head.weight, h)
        return ext.quantized_matmul_fused(head.scales, head.biases, head.weight, x, m.norm._weight_as(x.dtype, x.device),
                                          prologue=ext.PRO_RMSNORM, eps=m.norm.eps)

    def _capture(self) -> None:
        self.captures += 1
        self._slab_ptrs = self._slabs()
        forward = self._forward_fused if self.fused else self._forward_unfused
        with torch.cuda.stream(self._stream), _gc_paused():
            self._stream.wait_stream(torch.cuda.current_stream(self.device))
            # The warm-up passes really run: with the previous step's metadata still on the device they
            # would append a stale token's K/V through a stale block table - possibly into a page that
            # has been released and handed to another request since (slabs move when a second engine
            # reserves more pages).  All slots idle: appends are skipped and attention returns zeros;
            # step() / decode_on_device() upload the real block before they replay.
            self.meta_dev[2 * self.B : 3 * self.B].zero_()
            self.meta_dev[3 * self.B :].fill_(-1)
            self._tables_dirty = True
            for _ in range(2):  # warm-up: lazy kernel attribute setup must not happen under capture
                forward()
            self._stream.synchronize()
            self._graph = torch.cuda.CUDAGraph()
            with torch.cuda.graph(self._graph, stream=self._stream):
                forward()
            self._graph_loop = torch.cuda.CUDAGraph()
            launched = ext.launch_count()
            with torch.cuda.graph(self._graph_loop, stream=self._stream, pool=self._graph.pool()):
                forward()
                ext.decode_advance(self.tokens, self.next_tokens, self.offsets, self.context_lens, self.out_log, self.step_counter)
            # kernels of libtiny_llm_b200.so recorded into one self-advancing step
            self.kernels_per_step = ext.launch_count() - launched
            self._graphs = {self.B: self._graph}
            for rows in self._variants:
                if rows == self.B:
                    continue
                for _ in range(2):  # warm-up (metadata still all-idle): the narrower kernels set their attributes lazily
                    forward(rows)
                self._stream.synchronize()
                g = torch.cuda.CUDAGraph()
                with torch.cuda.graph(g, stream=self._stream, pool=self._graph.pool()):
                    forward(rows)
                self._graphs[rows] = g
        torch.cuda.current_stream(self.device).wait_stream(self._stream)

    def _ensure_graph(self) -> None:
        if self._graph is None or self._slab_ptrs != self._slabs():
            self._capture()

    # ------------------------------------------------------- host bookkeeping --
    def _slot_caches(self, caches, layer: int):
        """The per-slot request caches of one layer: a BatchingKvCache table, or a
        single request's cache list (B == 1)."""
        entry = caches[layer]
        if isinstance(entry, BatchingKvCache):
            return entry.kv_caches
        return [entry]

    def _drop(self, b: int) -> None:
        rec = self._recs[b]
        if rec is not None:
            rec.group.settle()
            for c in rec.group.caches:
                if c._lazy is rec.group:
                    c._lazy = None
            self.tables_np[:, b, :] = -1
            self._tables_dirty = True
            self._recs[b] = None

    def _register(self, b: int, caches) -> "_SlotRecord":
        """Slow path, once per request admission: take the request's per-layer cache objects as a
        group, check that they really are in lockstep (same page ids / fill / offset in every layer,
        which is what the schedulers of batch.py / generate.py produce: SURVEY section 7) and mirror
        their page ids into the table rows."""
        self._drop(b)
        group_caches = [self._slot_caches(caches, layer)[b] for layer in range(self.n_layers)]
        c0 = group_caches[0]
        for c in group_caches:
            if not isinstance(c, TinyKvPagedCache):
                raise ValueError("the decode engine needs paged request caches")
            if c._lazy is not None:
                c._lazy.settle()
        n = len(c0.page_ids)
        if n > self.max_pages:
            raise ValueError("request exceeds the engine's max_seq_len")
        lockstep = all(type(c) is TinyKvPagedCache and c.page_ids == c0.page_ids and c._page_lens == c0._page_lens and c._offset == c0._offset
                       for c in group_caches)
        if lockstep:
            self.tables_np[:, b, :n] = c0.page_ids
            self.tables_np[:, b, n:] = -1
        else:
            for layer, c in enumerate(group_caches):
                k = len(c.page_ids)
                if k > self.max_pages:
                    raise ValueError("request exceeds the engine's max_seq_len")
                self.tables_np[layer, b, :k] = c.page_ids
                self.tables_np[layer, b, k:] = -1
        self._tables_dirty = True
        group = _LockstepGroup(group_caches)
        if lockstep:
            for c in group_caches:
                c._lazy = group
        rec = _SlotRecord(c0, group, lockstep)
        self._recs[b] = rec
        return rec

    def _advance_host(self, caches, steps: int = 1) -> list[int]:
        """Account for ``steps`` one-token appends of every active request (host integers only) and
        bring the table rows up to date.  Returns the context length each slot will have after the
        FIRST of those steps.

        Cost per step at B = 64: one identity check per slot; the 36 per-layer cache objects of a
        request are touched only when its tail page overflows (once per ``page_size`` tokens) - the
        one-token appends in between are deferred (``TinyKvPagedCache._lazy``) and settled when
        somebody reads ``page_lens`` / ``offset``.  Round 1 walked 36 x B objects every step
        (0.4-1 ms of Python at B = 64, VERDICT weak #10)."""
        first_ctx = [0] * self.B
        slots0 = self._slot_caches(caches, 0)
        page = self.page_size
        for b, c0 in enumerate(slots0):
            rec = self._recs[b]
            if c0 is None:
                if rec is not None:
                    self._drop(b)
                continue
            if (rec is None or rec.c0 is not c0 or rec.epoch != c0.epoch
                    or (rec.lockstep and (c0._lazy is not rec.group or c0._offset + rec.group.pending != rec.offset or len(c0.page_ids) != rec.pages))):
                rec = self._register(b, caches)
            if not rec.lockstep:  # layers disagree: walk them (always correct, never taken by the in-tree schedulers)
                self._advance_slow(b, rec, caches, steps)
                first_ctx[b] = rec.offset - steps + 1
                continue
            tail = rec.offset - (rec.pages - 1) * page if rec.pages else page
            if tail + steps <= page:
                rec.group.pending += steps
                rec.offset += steps
            else:
                self._advance_pages(b, rec, steps)
            first_ctx[b] = rec.offset - steps + 1
        return first_ctx

    def _check_headroom(self, group_caches, steps: int) -> None:
        """All layers must be able to take the new pages BEFORE any of them is touched (a shortage
        used to surface at layer k with layers < k already advanced: ADVICE round 1)."""
        for c in group_caches:
            tail = c._page_lens[-1] if c.page_ids else self.page_size
            need = max(0, -(-(tail + steps - self.page_size) // self.page_size))
            if len(c.page_ids) + need > self.max_pages:
                raise ValueError("request exceeds the engine's max_seq_len")
            if need > len(c.pool.free_page_ids) + (c.pool.capacity - c.pool.num_pages):
                raise RuntimeError("page pool slab exhausted: reserve() more pages before decoding")

    def _advance_pages(self, b: int, rec: "_SlotRecord", steps: int) -> None:
        rec.group.settle()
        self._check_headroom(rec.group.caches, steps)
        old = rec.pages
        for layer, c in enumerate(rec.group.caches):
            for _ in range(steps):
                c.append_token_slot()
            self.tables_np[layer, b, old:len(c.page_ids)] = c.page_ids[old:]
        c0 = rec.c0
        rec.pages, rec.offset = len(c0.page_ids), c0._offset
        self._tables_dirty = True

    def _advance_slow(self, b: int, rec: "_SlotRecord", caches, steps: int) -> None:
        group_caches = [self._slot_caches(caches, layer)[b] for layer in range(self.n_layers)]
        self._check_headroom(group_caches, steps)
        for layer, c in enumerate(group_caches):
            for _ in range(steps):
                c.append_token_slot()
            k = len(c.page_ids)
            self.tables_np[layer, b, :k] = c.page_ids
            self.tables_np[layer, b, k:] = -1
        rec.group.caches = group_caches
        rec.offset = group_caches[0]._offset
        rec.pages = len(group_caches[0].page_ids)
        self._tables_dirty = True

    def _host_write_begin(self) -> None:
        """The pinned block is about to be rewritten: the previous upload must have been consumed
        (a caller that keeps sampling on the device never synchronises between steps)."""
        if self._upload_pending:
            self._upload_event.synchronize()
            self._upload_pending = False

    def _upload(self) -> None:
        B = self.B
        if self._tables_dirty:
            self.meta_dev.copy_(self.meta_host, non_blocking=True)
            self.h2d_bytes += self._meta_len * 4
            self._tables_dirty = False
        else:  # tokens | offsets | context_lens only: the block tables on the device are current
            self._meta_dev_head.copy_(self._meta_host_head, non_blocking=True)
            self.h2d_bytes += 3 * B * 4
        self._upload_event.record()
        self._upload_pending = True

    def upload_bytes_per_step(self) -> int:
        """Host -> device bytes of a steady-state step (block tables travel only when a page was added)."""
        return 3 * self.B * 4

    # ------------------------------------------------------------------ steps --
    def step(self, tokens, offsets, caches):
        """One decode step.  ``tokens``: B ids (list or tensor), ``offsets``: B
        RoPE positions; returns (logits [B, 1, V] static buffer, next_tokens [B])."""
        B = self.B
        self._host_write_begin()
        ctx = self._advance_host(caches, 1)
        self._ensure_graph()
        if isinstance(tokens, torch.Tensor):
            tok_host = None
        else:
            tok_host = tokens
            self.meta_np[0:B] = tok_host
        self.meta_np[B : 2 * B] = offsets
        self.meta_np[2 * B : 3 * B] = ctx
        # upload and replay on the CALLER's stream (the side stream is only needed for capture): two stream waits and a
        # stream-context switch less per step - host time here is serial with the GPU step when the caller reads every token
        self._upload()
        if tok_host is None:
            self.tokens.copy_(tokens.reshape(-1) if tokens.dtype == torch.int32 else tokens.reshape(-1).to(torch.int32), non_blocking=True)
        rows = B
        if len(self._variants) > 1:
            hi = 0
            for b, rec in enumerate(self._recs):
                if rec is not None:
                    hi = b + 1
            rows = next(r for r in self._variants if r >= hi)
            self.variant_replays[rows] += 1
        self._graphs[rows].replay()
        self.graph_replays += 1
        return self.logits.view(B, 1, self.V), self.next_tokens

    def decode_on_device(self, tokens, offsets, caches, steps: int) -> torch.Tensor:
        """``steps`` greedy decode steps with no host round trip: pages for all
        steps are allocated ahead, then the self-advancing graph is replayed
        back to back.  Returns the sampled tokens ``[steps, B]`` (device)."""
        if steps > self.log_capacity:
            raise ValueError("steps exceed the engine's token log capacity")
        B = self.B
        self._host_write_begin()
        ctx = self._advance_host(caches, steps)
        self._ensure_graph()
        self.meta_np[0:B] = tokens
        self.meta_np[B : 2 * B] = offsets
        self.meta_np[2 * B : 3 * B] = ctx
        cur = torch.cuda.current_stream(self.device)
        self._stream.wait_stream(cur)
        with torch.cuda.stream(self._stream):
            self._upload()
            self.step_counter.zero_()
            for i in range(steps):
                self._graph_loop.replay()
        cur.wait_stream(self._stream)
        self.graph_replays += steps
        return self.out_log[: steps * B].view(steps, B)


class PrefillEngine:
    """CUDA-graph replay of ONE chunked-prefill step (``Request.try_prefill``: B = 1, up to ``chunk`` prompt tokens,
    ``/root/reference/src/tiny_llm_ref/batch.py:48-76``) for the Week-3 paged model.

    The reference (and the operator path of this backend) issues ~20 operator calls per layer per chunk from
    Python: ~700 launches, 10-25 ms of host time for a 128-token chunk whose GPU work is ~1.5 ms.  Here the
    chunk's whole forward pass is captured once over static buffers; what changes between chunks is DATA in one
    pinned block: the token ids, per-token RoPE positions and post-append lengths, the request's block-table
    row per layer and the final context length.  A short (tail) chunk is RIGHT-aligned in the ``chunk`` rows:
    the padding rows in front carry context length 0 (nothing is appended for them) and the bottom-right causal
    rule of paged attention (``key <= row + ctx - L``) then gives every real row exactly its own prefix.

    Per layer: rms_norm -> q|k|v projection (one launch) -> q/k norm + RoPE + K/V append for all rows (one
    launch, ``tl_chunk_qk_norm_rope_append``) -> paged FlashAttention (tcgen05) -> o projection + residual ->
    rms_norm -> gate|up (+ SwiGLU) -> down + residual.  Rounding points are those of the operator sequence.
    Integer page bookkeeping stays in the request's ``TinyKvPagedCache`` objects (``append_slots``)."""

    def __init__(self, model, chunk: int, max_seq_len: int, device):
        self.model, self.L, self.device = model, int(chunk), torch.device(device)
        self.page_size = model.page_size
        self.max_pages = (max_seq_len + self.page_size - 1) // self.page_size
        self.max_seq_len = self.max_pages * self.page_size
        attn = model.layers_inner[0].self_attn
        self.Hq, self.Hkv, self.D = attn.num_heads, attn.num_kv_heads, attn.head_dim
        self.n_layers = model.num_hidden_layers
        L, Ly, MP = self.L, self.n_layers, self.max_pages
        # one int32 block: tokens [L] | offsets [L] | context_lens [L] | ctx_after [1] | tables [Ly, MP]
        self._meta_len = 3 * L + 1 + Ly * MP
        self.meta_host = torch.empty(self._meta_len, dtype=torch.int32, pin_memory=True)
        self.meta_np = self.meta_host.numpy()
        self.meta_np[:] = 0
        self.meta_np[3 * L + 1:] = -1
        self.meta_dev = torch.zeros(self._meta_len, dtype=torch.int32, device=self.device)
        self.meta_dev[3 * L + 1:] = -1
        self.tokens = self.meta_dev[0:L].view(1, L)
        self.offsets = self.meta_dev[L:2 * L]
        self.ctxs = self.meta_dev[2 * L:3 * L]
        self.ctx_after = self.meta_dev[3 * L:3 * L + 1]
        self.tables = self.meta_dev[3 * L + 1:].view(Ly, MP)
        self.tables_np = self.meta_np[3 * L + 1:].reshape(Ly, MP)
        self.logits = None
        self.next_token = torch.zeros(1, dtype=torch.int32, device=self.device)
        self._graph = None
        self._slab_ptrs = None
        self._stream = torch.cuda.Stream(device=self.device)
        self._upload_event = torch.cuda.Event()
        self._upload_pending = False
        self.replays = 0
        self.captures = 0
        self.kernels_per_chunk = 0
        self._packed = [
            SimpleNamespace(qkv=_concat_weights([b.self_attn.wq, b.self_attn.wk, b.self_attn.wv]),
                            gate_up=_interleave_gate_up(b.mlp.w_gate, b.mlp.w_up))
            for b in model.layers_inner
        ]

    @staticmethod
    def supported(model, device) -> bool:
        attn = model.layers_inner[0].self_attn
        rope = attn.rope
        return (torch.device(device).type == "cuda" and attn.head_dim == 128 and not rope.traditional and rope.dims == attn.head_dim
                and model.embedding.weight.scales.dtype == torch.bfloat16 and model.page_size % 64 == 0
                and 128 % (attn.num_heads // attn.num_kv_heads) == 0)

    def _slabs(self):
        return tuple(p.slab_version for p in self.model.page_pools)  # changes whenever a pool's slabs are (re)allocated

    def _forward(self) -> None:
        m, L = self.model, self.L
        Hq, Hkv, D = self.Hq, self.Hkv, self.D
        emb = m.embedding.weight
        x = ext.quantized_embedding(self.tokens, emb.scales, emb.biases, emb.weight, emb.group_size, emb.bits).view(L, -1)
        skinny = L <= 128  # the fused epilogues live in the <= 128-row tensor-core kernel; longer chunks use the 128 x 128-tile GEMM

        def normed(h, norm):
            return ext.rms_norm(h, norm._weight_as(h.dtype, h.device), norm.eps)

        def proj(h, w):
            return ext.quantized_matmul(w.scales, w.biases, w.group_size, w.bits, h, w.weight, True)

        layers = list(m.layers_inner)
        h = normed(x, layers[0].input_layernorm) if skinny else None
        for i, block in enumerate(layers):
            at, pk, pool = block.self_attn, self._packed[i], m.page_pools[i]
            if not skinny:
                h = normed(x, block.input_layernorm)
            if skinny:  # q|k|v projection + q/k norm + RoPE + append: the split-reduction planes feed the second kernel
                q = ext.qkv_project_rope_append(pk.qkv.scales, pk.qkv.biases, pk.qkv.weight, h, at.q_norm._weight_as(x.dtype, x.device),
                                                at.k_norm._weight_as(x.dtype, x.device), self.offsets, self.tables[i], self.ctxs,
                                                pool._key_pages, pool._value_pages, Hq, Hkv, at.rope.base, at.q_norm.eps, chunk=True)  # [Hq, L, D]
            else:
                q = ext.chunk_qk_norm_rope_append(proj(h, pk.qkv), at.q_norm._weight_as(x.dtype, x.device), at.k_norm._weight_as(x.dtype, x.device),
                                                  self.offsets, self.tables[i], self.ctxs, pool._key_pages, pool._value_pages,
                                                  Hq, Hkv, at.rope.base, at.q_norm.eps)  # [Hq, L, D]
            # [L, Hq * D]: the tcgen05 kernel writes the o-projection's layout itself (else: attention + one transpose copy)
            y = ext.paged_attention_token_major(q, pool._key_pages, pool._value_pages, self.tables[i:i + 1], self.ctx_after, at.scale,
                                                True, Hkv, Hq)
            if skinny:  # the residual projections return the next RMSNorm's output too (DecodeEngine._forward_fused_layers)
                ln2, wd = block.post_attention_layernorm, block.mlp.w_down
                x, h = ext.quantized_matmul_residual_norm(at.wo.scales, at.wo.biases, at.wo.weight, y, x, ln2._weight_as(x.dtype, x.device), ln2.eps)
                act = ext.quantized_matmul_fused(pk.gate_up.scales, pk.gate_up.biases, pk.gate_up.weight, h, epilogue=ext.EPI_SWIGLU_PAIRS)
                nxt = layers[i + 1].input_layernorm if i + 1 < len(layers) else m.norm
                x, h = ext.quantized_matmul_residual_norm(wd.scales, wd.biases, wd.weight, act, x, nxt._weight_as(x.dtype, x.device), nxt.eps)
            else:
                x = ext.add(x, proj(y, at.wo))
                h = normed(x, block.post_attention_layernorm)
                x = ext.add(x, proj(ext.swiglu(proj(h, block.mlp.w_gate), proj(h, block.mlp.w_up)), block.mlp.w_down))
        # logits_to_keep = 1: the hidden state is sliced before the final norm (qwen3_week3.py:330-338); RMSNorm is row-wise,
        # so the last row of the already normalised chunk is the same thing
        last = h[L - 1:L] if skinny else normed(x[L - 1:L], m.norm)
        head = m.w_lm_head if m.w_lm_head is not None else m.embedding.weight
        logits = proj(last, head)
        self.next_token.copy_(ext.argmax(logits))
        if self.logits is None:
            self.logits = torch.empty_like(logits)
        self.logits.copy_(logits)

    def _capture(self) -> None:
        self.captures += 1
        self._slab_ptrs = self._slabs()
        with torch.cuda.stream(self._stream), _gc_paused():
            self._stream.wait_stream(torch.cuda.current_stream(self.device))
            # warm-up passes run for real: all rows padding (context 0 -> no append), no visible keys
            self.meta_dev[2 * self.L:3 * self.L + 1].zero_()
            self.meta_dev[3 * self.L + 1:].fill_(-1)
            for _ in range(2):
                self._forward()
            self._stream.synchronize()
            self._graph = torch.cuda.CUDAGraph()
            launched = ext.launch_count()
            with torch.cuda.graph(self._graph, stream=self._stream):
                self._forward()
            self.kernels_per_chunk = ext.launch_count() - launched
        torch.cuda.current_stream(self.device).wait_stream(self._stream)

    def reserve_pools(self, pages_per_layer: int) -> None:
        for pool in self.model.page_pools:
            pool.reserve(pages_per_layer, self.Hkv, self.D, dtype=torch.bfloat16, device=self.device)

    def applies(self, tokens: int, offset: int, cache) -> bool:
        if not (0 < tokens <= self.L) or offset + tokens > self.max_seq_len:
            return False
        for layer_cache, pool in zip(cache, self.model.page_pools):
            if type(layer_cache) is not TinyKvPagedCache or layer_cache.pool is not pool or layer_cache.offset != offset:
                return False
            if pool._key_pages is None or pool._key_pages.dtype != torch.bfloat16:
                return False
            fresh = -(-(offset + tokens) // self.page_size) - len(layer_cache.page_ids)
            if fresh > len(pool.free_page_ids) + (pool.capacity - pool.num_pages):
                return False
        return True

    def prefill_chunk(self, token_ids, offset: int, cache):
        """Append ``token_ids`` (1..chunk ids at positions offset.., a list or an int32 device tensor) to the request's
        caches and return (logits [1, 1, V] of the last token - a static buffer -, greedy next token [1])."""
        on_device = isinstance(token_ids, torch.Tensor)
        r, L = (int(token_ids.numel()) if on_device else len(token_ids)), self.L
        if self._upload_pending:
            self._upload_event.synchronize()
            self._upload_pending = False
        for layer, layer_cache in enumerate(cache):
            layer_cache.append_slots(r)
            n = len(layer_cache.page_ids)
            self.tables_np[layer, :n] = layer_cache.page_ids
            self.tables_np[layer, n:] = -1
        if self._graph is None or self._slab_ptrs != self._slabs():
            self._capture()
        pad = L - r
        meta = self.meta_np
        meta[0:L] = 0
        if not on_device:
            meta[pad:L] = token_ids
        pos = np.arange(L, dtype=np.int32) - pad + offset
        meta[L:2 * L] = pos
        meta[2 * L:3 * L] = np.where(np.arange(L) >= pad, pos + 1, 0)
        meta[3 * L] = offset + r
        cur = torch.cuda.current_stream(self.device)
        self._stream.wait_stream(cur)
        with torch.cuda.stream(self._stream):
            self.meta_dev.copy_(self.meta_host, non_blocking=True)
            self._upload_event.record()
            self._upload_pending = True
            if on_device:  # ids stay on the device: no host round trip for the prompt
                self.meta_dev[pad:L].copy_(token_ids.reshape(-1).to(torch.int32), non_blocking=True)
            self._graph.replay()
        cur.wait_stream(self._stream)
        self.replays += 1
        return self.logits.view(1, 1, -1), self.next_token
