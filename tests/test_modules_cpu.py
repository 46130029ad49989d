"""CPU: host-side mirror of the reference interface -- names, state_dict keys, fp32/CPU semantics == oracle ==
reference fixtures, differentiable everywhere (the reference's autograd wrappers were not)."""
import pytest
import torch
import torch.nn as nn

import llama32_b200 as L
from conftest import load_golden
from oracle import ffn_oracle as O


def test_rmsnorm_module_matches_reference_fixture():
    g = load_golden("rmsnorm_cfg1.npz")
    n = L.LLAMARMSNorm(256, eps=g["eps"])
    with torch.no_grad():
        n.weight.copy_(g["weight"])
    assert torch.equal(n(g["x"]), g["y_nores"])
    assert torch.equal(n(g["x"], residual=g["residual"]), g["y_res"])
    assert list(n.state_dict().keys()) == ["weight"]


def test_ffn_module_matches_reference_fixture_and_is_differentiable():
    g = load_golden("ffn_small.npz")
    ff = L.FusedFeedforward(64, 176)
    assert sorted(ff.state_dict().keys()) == ["swiglu.w_gate", "swiglu.w_up", "w_down.weight"]
    with torch.no_grad():
        ff.swiglu.w_gate.copy_(g["w_gate"]); ff.swiglu.w_up.copy_(g["w_up"]); ff.w_down.weight.copy_(g["w_down"])
    x = g["x"].clone().requires_grad_(True)
    y = ff(x)
    assert torch.equal(y, g["y"])
    y.backward(g["grad_out"])    # the reference raises here (SURVEY.md 0.4)
    assert O.rel_l2(x.grad, g["dx"]) < 1e-5
    assert O.rel_l2(ff.swiglu.w_gate.grad, g["dw_gate"]) < 1e-5
    assert O.rel_l2(ff.swiglu.w_up.grad, g["dw_up"]) < 1e-5
    assert O.rel_l2(ff.w_down.weight.grad, g["dw_down"]) < 1e-5


def test_ffn_bias_variant():
    g = load_golden("ffn_bias.npz")
    ff = L.FusedFeedForward(64, 104, bias=True)
    assert sorted(ff.state_dict().keys()) == ["swiglu.b_gate", "swiglu.b_up", "swiglu.w_gate", "swiglu.w_up",
                                              "w_down.bias", "w_down.weight"]
    with torch.no_grad():
        ff.swiglu.w_gate.copy_(g["w_gate"]); ff.swiglu.w_up.copy_(g["w_up"]); ff.w_down.weight.copy_(g["w_down"])
        ff.swiglu.b_gate.copy_(g["b_gate"]); ff.swiglu.b_up.copy_(g["b_up"]); ff.w_down.bias.copy_(g["b_down"])
    x = g["x"].clone().requires_grad_(True)
    y = ff(x)
    assert torch.equal(y, g["y"])
    y.backward(g["grad_out"])
    assert ff.swiglu.b_gate.grad is not None and O.rel_l2(x.grad, g["dx"]) < 1e-5


def test_swiglu_function_none_biases_and_needs_input_grad():
    x = torch.randn(3, 16)
    wg, wu = torch.randn(24, 16, requires_grad=True), torch.randn(24, 16)
    out = L.SwiGLUFunction.apply(x, wg, wu, None, None)
    out.sum().backward()
    assert wg.grad is not None and wu.grad is None and x.grad is None


def test_rmsnorm_function_no_grad_for_none_residual():
    n = L.LLAMARMSNorm(16)
    x = torch.randn(2, 16, requires_grad=True)
    n(x).sum().backward()          # residual=None: must not raise / return a tensor grad for None
    assert x.grad is not None and n.weight.grad is not None


def test_lora_surgery_like_reference_readme():
    g = load_golden("lora_small.npz")
    lin = L.Linear_LORA(176, 64, rank=16, alpha=32.0, dropout=0.0)
    assert sorted(lin.state_dict().keys()) == g["state_dict_keys"]
    with torch.no_grad():
        lin.linear.weight.copy_(g["w"]); lin.lora_a.weight.copy_(g["lora_a"]); lin.lora_b.weight.copy_(g["lora_b"])
    assert torch.equal(lin(g["x"]), g["y"])
    assert not lin.linear.weight.requires_grad and lin.lora_a.weight.requires_grad
    # README recipe: replace w_down by Linear_LORA; w_gate / w_up are bare Parameters and stay trainable
    ff = L.FusedFeedforward(64, 176)
    lo = L.Linear_LORA(176, 64, rank=16, alpha=32.0, dropout=0.0)
    with torch.no_grad():
        lo.linear.weight.copy_(ff.w_down.weight)
        lo.lora_b.weight.zero_()
    ref = ff(g["x"][:, :64].contiguous())
    ff.w_down = lo
    x = g["x"][:, :64].contiguous().requires_grad_(True)
    out = ff(x)
    assert torch.allclose(out, ref, atol=1e-6)
    out.sum().backward()
    assert lo.linear.weight.grad is None and lo.lora_b.weight.grad is not None and ff.swiglu.w_gate.grad is not None


def test_block_hot_path_with_modules():
    g = load_golden("block_cfg1.npz")
    norm2 = L.LLAMARMSNorm(256, eps=g["eps"])
    ff = L.FusedFeedforward(256, 688)
    with torch.no_grad():
        norm2.weight.copy_(g["norm2_weight"])
        ff.swiglu.w_gate.copy_(g["w_gate"]); ff.swiglu.w_up.copy_(g["w_up"]); ff.w_down.weight.copy_(g["w_down"])
    normed = norm2(g["attn_out"], residual=g["hidden"])
    out = g["attn_out"] + ff(normed)
    assert torch.equal(normed, g["normed"]) and torch.equal(out, g["block_out"])


def test_convert_feedforward_to_fused():
    class FeedForward(nn.Module):
        def __init__(self):
            super().__init__()
            self.w1 = nn.Linear(16, 40, bias=False)
            self.w3 = nn.Linear(16, 40, bias=False)
            self.w2 = nn.Linear(40, 16, bias=False)

        def forward(self, x):
            return self.w2(torch.nn.functional.silu(self.w1(x)) * self.w3(x))

    m = FeedForward()
    f = L.convert_feedforward_to_fused(m)
    x = torch.randn(5, 16)
    assert torch.allclose(f(x), m(x), atol=1e-6)


def test_mixed_dtype_weight_is_rejected_by_cuda_ops_but_module_gates():
    # fp32 module, bf16 CPU input: reference semantics = PyTorch expression (no CUDA path on CPU tensors)
    n = L.LLAMARMSNorm(16)
    y = n(torch.randn(2, 16, dtype=torch.bfloat16))
    assert y.dtype == torch.float32   # promotion, as the reference fallback does (SURVEY.md 8a)


def test_kv_cache_preallocated_semantics():
    """KVCache (drop-in for reference Model/model.py:12-29): update() returns what the reference's torch.cat version would,
    capacity grows by doubling without losing content, num_items() follows layer 0."""
    import llama32_b200 as L
    torch.manual_seed(0)
    cache = L.KVCache(capacity=4)
    ks, vs = [], []
    for step, t in enumerate((3, 1, 1, 70, 1)):
        for layer in range(2):
            k, v = torch.randn(2, 2, t, 8), torch.randn(2, 2, t, 8)
            if layer == 0:
                ks.append(k); vs.append(v)
            kk, vv = cache.update(k, v, layer)
            if layer == 0:
                assert torch.equal(kk, torch.cat(ks, dim=-2)) and torch.equal(vv, torch.cat(vs, dim=-2))
        assert cache.num_items() == sum(x.shape[-2] for x in ks)
    assert cache._k[0].shape[2] >= 76 and cache._k[0].shape[2] % 64 == 0
    assert torch.equal(cache.key_cache[0], torch.cat(ks, dim=-2))


@pytest.mark.parametrize("tag", ["d64", "d128"])
def test_gqa_module_cpu_path_matches_the_reference_fixture(tag, golden):
    """GroupQueryAttention on CPU fp32 evaluates the reference's expressions: the reference's own outputs (prefill with a
    padded batch + a KV-cached decode step) up to fp32 rounding, with OUR preallocated KVCache underneath."""
    import llama32_b200 as L
    from oracle import ffn_oracle as O
    g = golden(f"attention_{tag}.npz")
    heads, kv = int(g["n_heads"]), int(g["n_kv"])
    b, t, hidden = g["x"].shape

    class Cfg:
        hidden_size, n_heads, n_kv_groups, rope_base = hidden, heads, kv, float(g["rope_base"])
    att = L.GroupQueryAttention(Cfg, layer_idx=0).eval()
    with torch.no_grad():
        att.W_query.weight.copy_(g["wq"]); att.W_key.weight.copy_(g["wk"]); att.W_value.weight.copy_(g["wv"]); att.out_proj.weight.copy_(g["wo"])
    cache = L.KVCache()
    with torch.no_grad():
        y = att(g["x"], attention_mask=O.causal_padding_mask(g["mask2d"], t), position_ids=g["position_ids"], kv_cache=cache)
        y1 = att(g["x_decode"], attention_mask=torch.zeros(b, 1, 1, 1), position_ids=g["position_ids_decode"], kv_cache=cache)

    # The fixture was computed on another host.  fp32 GEMMs on the CPU round differently with the instruction set and the
    # thread split the BLAS picks there (MKL's AVX2 path moves cache_v by ~5e-7), so exact equality would test the host.
    # The bound: reductions over `hidden` products, each ordering within ~sqrt(hidden) ulps of its operands' scale.  The
    # outputs are reduced from K / V, which are an order of magnitude larger than y_decode, so every tensor is held to the
    # scale of the largest of them, and never to less than 2e-6.  A real defect shows as ~1e-2.
    scale = max(float(g[k].abs().max()) for k in ("y_prefill", "y_decode", "cache_k", "cache_v"))
    atol = max(2e-6, 2 * hidden ** 0.5 * torch.finfo(torch.float32).eps * scale)
    close = lambda got, ref: torch.allclose(got, ref, rtol=0, atol=atol)
    assert close(y, g["y_prefill"]) and close(y1, g["y_decode"])
    assert close(cache.key_cache[0], g["cache_k"]) and close(cache.value_cache[0], g["cache_v"])
