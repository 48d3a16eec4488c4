"""B200 decode runtime: fused decode kernels and the CUDA-graph engine must
reproduce the operator-by-operator path (same rounding points), and the
device-resident greedy loop must emit the tokens of the host-driven loop."""

import gc

import pytest
import torch

from extensions_b200 import tiny_llm_ext_b200 as ext
from tiny_llm_b200 import BatchingKvCache, ContinuousBatcher, Qwen3ModelWeek3
from tiny_llm_b200.engine import DecodeEngine
from tiny_llm_b200.synthetic import synthetic_qwen3

pytestmark = pytest.mark.gpu
BF16 = torch.bfloat16


@pytest.fixture(scope="module")
def dev(cuda_device):
    return cuda_device


def packed(K, N, g, dev):
    sigma = 1.0 / (4.717 * N**0.5)
    words = torch.randint(-(2**31), 2**31, (K, N // 8), dtype=torch.int64, generator=g).to(torch.int32)
    scales = (torch.randn(K, N // 128, generator=g) * sigma).to(BF16)
    biases = (-7.5 * scales.float() + torch.randn(K, N // 128, generator=g) * sigma).to(BF16)
    return words.to(dev), scales.to(dev), biases.to(dev)


@pytest.mark.parametrize("M", [1, 3, 8, 16])
@pytest.mark.parametrize("N,K", [(2560, 6144), (256, 96), (9728, 2560), (1024, 40)])
def test_fused_projection_equals_the_unfused_operator_sequence(dev, M, N, K):
    g = torch.Generator().manual_seed(M * 100 + N + K)
    w, s, b = packed(K, N, g, dev)
    x = (torch.randn(M, N, generator=g) * 2).to(BF16).to(dev)
    nw = (1 + 0.1 * torch.randn(N, generator=g)).to(BF16).to(dev)
    res = torch.randn(M, K, generator=g).to(BF16).to(dev)
    plain = ext.quantized_matmul(s, b, 128, 4, x, w, True)
    assert torch.equal(ext.quantized_matmul_fused(s, b, w, x), plain)
    # residual epilogue: add(residual, matmul) with the intermediate rounded exactly as the two-op sequence
    assert torch.equal(ext.quantized_matmul_fused(s, b, w, x, residual=res, epilogue=ext.EPI_RESIDUAL), ext.add(res, plain))
    # rms_norm prologue: the sum of squares is reduced in a different order than the standalone
    # kernel, so the normalised activations may differ by one bf16 ulp in rare elements
    want = ext.quantized_matmul(s, b, 128, 4, ext.rms_norm(x, nw, 1e-6), w, True)
    got = ext.quantized_matmul_fused(s, b, w, x, nw, prologue=ext.PRO_RMSNORM, eps=1e-6)
    torch.testing.assert_close(got.float(), want.float(), rtol=2**-7, atol=2e-3 * float(want.float().abs().max()))
    # swiglu prologue over the two halves of one [M, 2N] buffer (how gate|up is laid out)
    gu = (torch.randn(M, 2 * N, generator=g) * 2).to(BF16).to(dev)
    want = ext.quantized_matmul(s, b, 128, 4, ext.swiglu(gu[:, :N].contiguous(), gu[:, N:].contiguous()), w, True)
    got = ext.quantized_matmul_fused(s, b, w, gu[:, :N], gu[:, N:], residual=res, prologue=ext.PRO_SWIGLU, epilogue=ext.EPI_RESIDUAL)
    if M <= 8:
        assert torch.equal(got, ext.add(res, want))
    else:  # more than 8 rows: the unfused product runs on the tensor-core kernel (weights rounded to bf16), the prologue form on the streaming kernel
        torch.testing.assert_close(got.float(), ext.add(res, want).float(), rtol=2**-7, atol=2e-3 * float(want.float().abs().max()) + 2**-7)


@pytest.mark.parametrize("M", [3, 16, 64, 128])
@pytest.mark.parametrize("N,K", [(4096, 2560), (9728, 2560), (256, 96), (2560, 6144)])
def test_residual_projection_with_the_next_rmsnorm_equals_the_two_operators(dev, M, N, K):
    """o / down projection + residual, handing back the next block's RMSNorm output too: the residual stream is the
    two-operator result bit for bit; the normalised row may differ by one bf16 ulp in rare elements (the sum of squares
    is reduced in another order than the standalone kernel's).  K = 6144 exceeds the in-kernel row limit and K = 96 /
    M = 3 take the unsplit / streaming paths: the call falls back to rms_norm itself."""
    g = torch.Generator().manual_seed(M * 7 + N + K)
    w, s, b = packed(K, N, g, dev)
    x = (torch.randn(M, N, generator=g) * 2).to(BF16).to(dev)
    nw = (1 + 0.1 * torch.randn(K, generator=g)).to(BF16).to(dev)
    res = torch.randn(M, K, generator=g).to(BF16).to(dev)
    want_x = ext.quantized_matmul_fused(s, b, w, x, residual=res, epilogue=ext.EPI_RESIDUAL)
    want_h = ext.rms_norm(want_x, nw, 1e-6)
    got_x, got_h = ext.quantized_matmul_residual_norm(s, b, w, x, res, nw, 1e-6)
    assert torch.equal(got_x, want_x)
    torch.testing.assert_close(got_h.float(), want_h.float(), rtol=2**-7, atol=2**-8 * float(want_h.float().abs().max()))
    again_x, again_h = ext.quantized_matmul_residual_norm(s, b, w, x, res, nw, 1e-6)
    assert torch.equal(again_h, got_h) and torch.equal(again_x, got_x)  # same bits on every run


@pytest.mark.parametrize("M", [1, 5, 8, 16, 64])
@pytest.mark.parametrize("N,inter", [(2560, 9728), (256, 384), (1024, 40)])
def test_swiglu_pairs_epilogue_equals_projection_then_swiglu(dev, M, N, inter):
    """gate|up rows interleaved in blocks of 8: the projection emits swiglu(gate, up) itself."""
    g = torch.Generator().manual_seed(M + N + inter)
    wg, sg, bg = packed(inter, N, g, dev)
    wu, su, bu = packed(inter, N, g, dev)
    x = (torch.randn(M, N, generator=g) * 2).to(BF16).to(dev)
    want = ext.swiglu(ext.quantized_matmul(sg, bg, 128, 4, x, wg, True), ext.quantized_matmul(su, bu, 128, 4, x, wu, True))
    w, s, b = ext.interleave_gate_up(wg, wu), ext.interleave_gate_up(sg, su), ext.interleave_gate_up(bg, bu)
    got = ext.quantized_matmul_fused(s, b, w, x, epilogue=ext.EPI_SWIGLU_PAIRS)
    assert got.shape == (M, inter)
    # the 2*inter-row projection deals its rows to CTAs and warps differently from the two
    # inter-row projections, so the fp32 partial sums meet in a different order: one bf16 ulp
    torch.testing.assert_close(got.float(), want.float(), rtol=2**-7, atol=2e-3 * float(want.float().abs().max()))


def test_fused_qk_norm_rope_append_equals_the_unfused_sequence(dev):
    g = torch.Generator().manual_seed(3)
    B, Hq, Hkv, D, page, P = 3, 32, 8, 128, 16, 7
    qkv = torch.randn(B, (Hq + 2 * Hkv) * D, generator=g).to(BF16).to(dev)
    qw = (1 + 0.1 * torch.randn(D, generator=g)).to(BF16).to(dev)
    kw = (1 + 0.1 * torch.randn(D, generator=g)).to(BF16).to(dev)
    offsets = torch.tensor([16, 0, 4095], dtype=torch.int32, device=dev)
    ctx = torch.tensor([17, 0, 33], dtype=torch.int32, device=dev)
    bt = torch.tensor([[5, 2, -1], [-1, -1, -1], [0, 6, 3]], dtype=torch.int32, device=dev)
    kp = torch.randn(P, Hkv, page, D, generator=g).to(BF16).to(dev)
    vp = torch.randn(P, Hkv, page, D, generator=g).to(BF16).to(dev)
    kp_ref, vp_ref = kp.clone(), vp.clone()
    q_in = qkv[:, : Hq * D].reshape(B, 1, Hq, D).contiguous()
    k_in = qkv[:, Hq * D : (Hq + Hkv) * D].reshape(B, 1, Hkv, D).contiguous()
    v_in = qkv[:, (Hq + Hkv) * D :].reshape(B, Hkv, 1, D).contiguous()
    q_ref = ext.rope(ext.rms_norm(q_in, qw, 1e-6), offsets, D, 1e6)
    k_ref = ext.rope(ext.rms_norm(k_in, kw, 1e-6), offsets, D, 1e6)
    ext.paged_cache_append_decode(kp_ref, vp_ref, k_ref.reshape(B, Hkv, 1, D), v_in, bt, ctx)
    q = ext.decode_qk_norm_rope_append(qkv, qw, kw, offsets, bt, ctx, kp, vp, Hq, Hkv, 1e6, 1e-6)
    # the per-head sum of squares is reduced in a different order: allow one bf16 ulp
    torch.testing.assert_close(q.float(), q_ref.reshape(B, Hq, D).float(), rtol=2**-7, atol=1e-3)
    torch.testing.assert_close(kp.float(), kp_ref.float(), rtol=2**-7, atol=1e-3)
    assert torch.equal(vp, vp_ref), "V rows are copied, bit for bit"
    untouched = torch.ones(P, dtype=torch.bool)
    untouched[[2, 3]] = False
    assert torch.equal(kp[untouched.to(dev)], kp_ref[untouched.to(dev)])


@pytest.mark.parametrize("contexts,page", [([17, 1, 33], 16), ([131, 256, 257], 128), ([700, 5, 1030], 64), ([4100], 128)])
@pytest.mark.parametrize("Hq,Hkv", [(32, 8), (4, 2), (2, 2)])
def test_fused_decode_attention_equals_the_operator_sequence(dev, contexts, page, Hq, Hkv):
    """q/k norm + rope + append + paged attention in one launch (and its split/merge form for long
    contexts) against the per-operator kernels on the same cache."""
    g = torch.Generator().manual_seed(sum(contexts) + Hq)
    B, D = len(contexts), 128
    max_pages = (max(contexts) + page - 1) // page + 1
    P = B * max_pages + 2
    qkv = torch.randn(B, (Hq + 2 * Hkv) * D, generator=g).to(BF16).to(dev)
    qw = (1 + 0.1 * torch.randn(D, generator=g)).to(BF16).to(dev)
    kw = (1 + 0.1 * torch.randn(D, generator=g)).to(BF16).to(dev)
    ctx = torch.tensor(contexts, dtype=torch.int32, device=dev)
    offsets = (ctx - 1).clamp_min(0).to(torch.int32)
    perm = torch.randperm(P, generator=g)
    bt = torch.full((B, max_pages), -1, dtype=torch.int32)
    for b, c in enumerate(contexts):
        n = (c + page - 1) // page
        bt[b, :n] = perm[b * max_pages : b * max_pages + n].to(torch.int32)
    bt = bt.to(dev)
    kp = torch.randn(P, Hkv, page, D, generator=g).to(BF16).to(dev)
    vp = torch.randn(P, Hkv, page, D, generator=g).to(BF16).to(dev)
    kp_ref, vp_ref = kp.clone(), vp.clone()
    scale = D**-0.5
    q = ext.decode_qk_norm_rope_append(qkv, qw, kw, offsets, bt, ctx, kp_ref, vp_ref, Hq, Hkv, 1e6, 1e-6)
    want = ext.paged_attention(q.view(B * Hq, 1, D), kp_ref, vp_ref, bt, ctx, scale, is_causal=True, num_kv_heads=Hkv, num_heads=Hq)
    freq = ext.rope_inv_freq_table(D, 1e6, dev)
    got = ext.decode_attention_fused(qkv, qw, kw, offsets, bt, ctx, freq, kp, vp, Hq, Hkv, 1e-6, scale, max(contexts) + 7)
    assert torch.equal(kp, kp_ref) and torch.equal(vp, vp_ref), "the appended rows are the same bits"
    # probabilities stay fp32 in both; the summation order over tokens differs
    torch.testing.assert_close(got.float().view(B * Hq, D), want.float().view(B * Hq, D), rtol=2**-7, atol=4e-3)


def test_fused_decode_attention_and_swiglu_epilogue_against_the_cpu_oracle(dev):
    """The two fused decode launches against the CPU restatement of the reference operators
    (oracle/ops.py), not against other GPU kernels: q/k rms_norm -> rope -> paged_cache_update ->
    paged_attention, and quantized_matmul x2 -> swiglu."""
    from oracle import ops as oracle

    g = torch.Generator().manual_seed(11)
    B, Hq, Hkv, D, page = 2, 8, 2, 128, 16
    contexts = [37, 70]
    max_pages = 6
    P = B * max_pages
    qkv = torch.randn(B, (Hq + 2 * Hkv) * D, generator=g).to(BF16)
    qw = (1 + 0.1 * torch.randn(D, generator=g)).to(BF16)
    kw = (1 + 0.1 * torch.randn(D, generator=g)).to(BF16)
    ctx = torch.tensor(contexts, dtype=torch.int32)
    offsets = ctx - 1
    bt = torch.full((B, max_pages), -1, dtype=torch.int32)
    perm = torch.randperm(P, generator=g)
    for b, c in enumerate(contexts):
        n = (c + page - 1) // page
        bt[b, :n] = perm[b * max_pages : b * max_pages + n].to(torch.int32)
    kp = torch.randn(P, Hkv, page, D, generator=g).to(BF16)
    vp = torch.randn(P, Hkv, page, D, generator=g).to(BF16)
    scale = D**-0.5
    # oracle: the reference operator sequence, request by request
    kp_ref, vp_ref = kp.clone(), vp.clone()
    q_in = qkv[:, : Hq * D].reshape(B, 1, Hq, D)
    k_in = qkv[:, Hq * D : (Hq + Hkv) * D].reshape(B, 1, Hkv, D)
    v_in = qkv[:, (Hq + Hkv) * D :].reshape(B, 1, Hkv, D)
    q_ref = oracle.rope(oracle.rms_norm(q_in, qw, 1e-6), offsets, D, 1e6)
    k_ref = oracle.rope(oracle.rms_norm(k_in, kw, 1e-6), offsets, D, 1e6)
    for b, c in enumerate(contexts):
        tok = c - 1
        pid = int(bt[b, tok // page])
        oracle.paged_cache_update(kp_ref, k_ref[b : b + 1].transpose(1, 2).contiguous(), pid, tok % page)
        oracle.paged_cache_update(vp_ref, v_in[b : b + 1].transpose(1, 2).contiguous(), pid, tok % page)
    want = oracle.paged_attention(q_ref.transpose(1, 2).reshape(B * Hq, 1, D).contiguous(), kp_ref, vp_ref, bt, ctx, scale, True, Hkv, Hq)
    kd, vd = kp.to(dev), vp.to(dev)
    got = ext.decode_attention_fused(qkv.to(dev), qw.to(dev), kw.to(dev), offsets.to(dev), bt.to(dev), ctx.to(dev),
                                     ext.rope_inv_freq_table(D, 1e6, dev), kd, vd, Hq, Hkv, 1e-6, scale, max(contexts))
    torch.testing.assert_close(kd.cpu().float(), kp_ref.float(), rtol=2**-7, atol=4e-3)
    assert torch.equal(vd.cpu(), vp_ref)
    torch.testing.assert_close(got.cpu().float().view(B * Hq, D), want.float().view(B * Hq, D), rtol=2e-2, atol=5e-3)  # 2e-2: test_week_3_day_5.py:61

    # gate|up projection with the SwiGLU epilogue
    N, inter, M = 512, 256, 3
    wg, sg, bg = packed(inter, N, g, torch.device("cpu"))
    wu, su, bu = packed(inter, N, g, torch.device("cpu"))
    x = (torch.randn(M, N, generator=g) * 2).to(BF16)
    want = oracle.swiglu(oracle.quantized_matmul(sg, bg, 128, 4, x, wg, True), oracle.quantized_matmul(su, bu, 128, 4, x, wu, True))
    w, s_, b_ = ext.interleave_gate_up(wg, wu), ext.interleave_gate_up(sg, su), ext.interleave_gate_up(bg, bu)
    got = ext.quantized_matmul_fused(s_.to(dev), b_.to(dev), w.to(dev), x.to(dev), epilogue=ext.EPI_SWIGLU_PAIRS)
    torch.testing.assert_close(got.cpu().float(), want.float(), rtol=2e-2, atol=2e-2 * float(want.float().abs().max()))


@pytest.fixture(scope="module")
def tiny_gpu(dev):
    return synthetic_qwen3("tiny-d128", seed=0, realistic=True, max_position_embeddings=512, device=dev)


def prefill(model, dev, prompt):
    cache = model.create_kv_cache()
    was = model.use_decode_graph
    model.use_decode_graph = False
    logits = model(torch.tensor([prompt], dtype=torch.int32, device=dev), 0, cache, logits_to_keep=1)
    model.use_decode_graph = was
    return cache, int(torch.argmax(logits[0, -1].float()))


@pytest.mark.parametrize("mode", ["graph-unfused", "graph-fused"])
def test_engine_step_matches_the_operator_path(dev, tiny_gpu, mode):
    fused = mode != "graph-unfused"
    prompt = [5, 17, 3, 250, 99, 42, 7, 300, 11, 8, 1]
    ref_model = Qwen3ModelWeek3(tiny_gpu, page_size=8)
    ref_model.use_decode_graph = False
    model = Qwen3ModelWeek3(tiny_gpu, page_size=8)
    engine = DecodeEngine(model, 1, 256, dev, fused=fused)
    engine.reserve_pools()
    ref_cache, tok = prefill(ref_model, dev, prompt)
    cache, tok2 = prefill(model, dev, prompt)
    assert tok == tok2
    offset = len(prompt)
    for step in range(20):  # crosses page boundaries (page size 8)
        want = ref_model(torch.tensor([[tok]], dtype=torch.int32, device=dev), offset, ref_cache, logits_to_keep=1)
        got, nxt = engine.step([tok], [offset], cache)
        if fused:
            torch.testing.assert_close(got.float(), want.float(), rtol=0, atol=0.06)
        else:
            assert torch.equal(got.view_as(want), want), f"step {step}: graph replay of the same operators must be bit-identical"
        assert cache[0].page_ids == ref_cache[0].page_ids and cache[0].page_lens == ref_cache[0].page_lens
        assert int(nxt[0]) == int(torch.argmax(got.float().reshape(-1)))
        tok = int(torch.argmax(want[0, -1].float()))
        offset += 1
    assert engine.graph_replays == 20
    for c in (*cache, *ref_cache):
        c.release()


def test_graph_step_with_split_kv_attention_matches_operator_path(dev, tiny_gpu):
    """Context long enough that the fused attention launch splits the KV range over several
    CTAs and runs its merge launch (601 tokens of a 1024-token engine)."""
    g = torch.Generator().manual_seed(5)
    prompt = torch.randint(1, 500, (600,), generator=g).tolist()
    ref_model = Qwen3ModelWeek3(tiny_gpu, page_size=128)
    ref_model.use_decode_graph = False
    model = Qwen3ModelWeek3(tiny_gpu, page_size=128)
    engine = DecodeEngine(model, 1, 1024, dev)
    engine.reserve_pools()
    ref_cache, tok = prefill(ref_model, dev, prompt)
    cache, _ = prefill(model, dev, prompt)
    offset = len(prompt)
    for step in range(4):
        want = ref_model(torch.tensor([[tok]], dtype=torch.int32, device=dev), offset, ref_cache, logits_to_keep=1)
        got, nxt = engine.step([tok], [offset], cache)
        torch.testing.assert_close(got.float(), want.float(), rtol=0, atol=0.06)
        # the appended K/V rows must be the ones the operator path wrote
        pool, ref_pool = model.page_pools[1], ref_model.page_pools[1]
        pid, slot = cache[1].page_ids[-1], cache[1].page_lens[-1] - 1
        rid = ref_cache[1].page_ids[-1]
        # (layer 1's rows have been through a full layer of two different kernel families: the hidden
        # state may differ by an ulp, which rms_norm + rope can turn into a few ulps of a K element; a misplaced row would be off by O(1))
        torch.testing.assert_close(pool._key_pages[pid, :, slot].float(), ref_pool._key_pages[rid, :, slot].float(), rtol=2**-6, atol=5e-2)
        torch.testing.assert_close(pool._value_pages[pid, :, slot].float(), ref_pool._value_pages[rid, :, slot].float(), rtol=2**-6, atol=5e-2)
        tok = int(torch.argmax(want[0, -1].float()))
        offset += 1


def test_device_resident_greedy_loop_equals_host_driven_loop(dev, tiny_gpu):
    prompt = [9, 2, 4, 6, 8, 10, 12]
    steps = 24

    def run(on_device: bool):
        model = Qwen3ModelWeek3(tiny_gpu, page_size=8)
        engine = DecodeEngine(model, 1, 256, dev)
        engine.reserve_pools()
        cache, tok = prefill(model, dev, prompt)
        if on_device:
            out = engine.decode_on_device([tok], [len(prompt)], cache, steps).cpu().reshape(-1).tolist()
        else:
            out, offset = [], len(prompt)
            for _ in range(steps):
                _, nxt = engine.step([tok], [offset], cache)
                tok = int(nxt[0])
                out.append(tok)
                offset += 1
        state = (list(cache[0].page_ids), list(cache[0].page_lens), cache[0].offset)
        for c in cache:
            c.release()
        return out, state

    host_tokens, host_state = run(False)
    dev_tokens, dev_state = run(True)
    assert dev_tokens == host_tokens
    assert dev_state == host_state == ([0, 1, 2, 3], [8, 8, 8, 7], 31)


def test_no_garbage_collection_starts_while_an_engine_captures(dev, tiny_gpu):
    """An engine and its model reference each other, so a dropped model's CUDA graphs are freed by the cyclic
    collector, and destroying a graph while a stream captures invalidates that capture.  With a collection due at
    almost every allocation, none may start inside the decode or the prefill engine's capture."""
    capturing = []

    def watch(phase, info):
        if phase == "start":
            capturing.append(torch.cuda.is_current_stream_capturing())

    model = Qwen3ModelWeek3(tiny_gpu, page_size=64)  # 64-token pages: prefill chunks run on the prefill engine
    cache, tok = prefill(model, dev, [9, 2, 4, 6, 8])
    gc.collect()  # engines dropped by earlier tests go now, outside any capture
    threshold = gc.get_threshold()
    gc.callbacks.append(watch)
    gc.set_threshold(1)
    try:
        model(torch.tensor([[tok]], dtype=torch.int32, device=dev), 5, cache, logits_to_keep=1)  # decode engine capture
        second = model.create_kv_cache()
        model(torch.tensor([[1, 5, 7]], dtype=torch.int32, device=dev), 0, second, logits_to_keep=1)  # prefill engine capture
    finally:
        gc.set_threshold(*threshold)
        gc.callbacks.remove(watch)
    for c in (*cache, *second):
        c.release()
    assert model._decode_engines and model._prefill_engines
    assert capturing and not any(capturing)


def test_public_model_call_uses_the_graph_and_matches_operator_path(dev, tiny_gpu):
    auto = Qwen3ModelWeek3(tiny_gpu, page_size=8)
    plain = Qwen3ModelWeek3(tiny_gpu, page_size=8)
    plain.use_decode_graph = False
    prompts = {0: [1, 5, 7], 2: [9, 2, 4, 6, 8, 10, 12, 14, 16, 18, 20]}
    outs = []
    for model in (auto, plain):
        tables = [BatchingKvCache(3, max_seq_len=64) for _ in range(model.num_hidden_layers)]
        for slot, ids in prompts.items():
            cache = model.create_kv_cache()
            model(torch.tensor([ids], dtype=torch.int32, device=dev), 0, cache, logits_to_keep=1)
            for layer_cache, table in zip(cache, tables):
                table.add_request(layer_cache, slot)
        seq = []
        for step in range(7):
            seq.append(model(torch.tensor([[11], [0], [13]], dtype=torch.int32, device=dev), [3 + step, 0, 11 + step], tables, logits_to_keep=1))
        outs.append((seq, [tables[0].kv_caches[s].page_ids[:] for s in (0, 2)], tables[0].HD))
    assert auto._decode_engines and not plain._decode_engines
    assert outs[0][1] == outs[1][1] and outs[0][2] == outs[1][2] == (2, 128)
    for a, b in zip(outs[0][0], outs[1][0]):
        assert tuple(a.shape) == (3, 1, 512)
        torch.testing.assert_close(a[[0, 2]].float(), b[[0, 2]].float(), rtol=0, atol=0.06)


def test_scheduler_runs_on_the_graph_path_and_releases_everything(dev, tiny_gpu):
    model = Qwen3ModelWeek3(tiny_gpu, page_size=8)
    g = torch.Generator().manual_seed(11)
    prompts = [torch.randint(1, 500, (n,), generator=g).tolist() for n in (5, 19, 3, 12, 8, 27, 9)]
    budgets = [6, 3, 5, 2, 4, 3, 7]
    batcher = ContinuousBatcher(model, None, prompts, max_seq_len=64, batch_size=3, prefill_step=8, verbose=False, device=dev, max_new_tokens=budgets)
    results = dict(batcher.run())
    assert [len(results[i].split()) for i in range(7)] == budgets
    assert all(pool.used_page_ids == set() and pool.num_free_pages == pool.num_pages for pool in model.page_pools)
    assert model._decode_engines, "decode steps should have gone through the CUDA graph"
    with pytest.raises(ValueError, match="exceeds max_seq_len"):
        ContinuousBatcher(model, None, [[1] * 70], max_seq_len=64, batch_size=3, verbose=False, device=dev).run()
