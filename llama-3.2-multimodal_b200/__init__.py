"""B200-native (sm_100a) Add-RMSNorm + SwiGLU feed-forward hot path of LLaMA-3.2-Multimodal.

The directory name is not a Python identifier; import it as `llama32_b200` (alias package at the repo root).
"""
from .modules import (  # noqa: F401
    BlockTailFunction,
    FFNFunction,
    FFNLoRAFunction,
    FusedFeedForward,
    FusedFeedforward,
    FusedSwiGLU,
    GQAAttentionFunction,
    GroupQueryAttention,
    KVCache,
    PagedKVCache,
    LLAMARMSNorm,
    LMHeadCEFunction,
    Linear_LORA,
    LinearFunction,
    LinearLoRAFunction,
    RMSNormFunction,
    SpeculativeDecoder,
    SwiGLUFunction,
    TokenSampler,
    block_tail,
    chain_block_norms,
    convert_feedforward_to_fused,
    convert_instances,
    last_token_logits,
    lm_head_loss,
    patch_reference,
    shift_labels,
)

__all__ = [
    "FFNFunction", "FFNLoRAFunction", "FusedFeedForward", "FusedFeedforward", "FusedSwiGLU", "LLAMARMSNorm", "Linear_LORA",
    "LinearFunction", "RMSNormFunction", "SwiGLUFunction", "block_tail", "convert_feedforward_to_fused", "convert_instances",
    "patch_reference", "BlockTailFunction", "LinearLoRAFunction", "chain_block_norms", "LMHeadCEFunction", "lm_head_loss", "shift_labels", "GroupQueryAttention", "KVCache",
    "GQAAttentionFunction", "PagedKVCache", "TokenSampler", "last_token_logits",
    "SpeculativeDecoder",
]
