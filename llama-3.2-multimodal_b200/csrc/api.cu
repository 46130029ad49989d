// C-ABI layer (include/l32_ffn.h): argument validation and composition of the kernels.  No torch types, no
// allocation, no synchronisation: everything is enqueued on the caller's stream and scratch is caller-provided.
#include "../../include/l32_ffn.h"
#include "l32_internal.cuh"

#include <atomic>
#include <cstdlib>

using namespace l32;

namespace l32 {
static std::atomic<unsigned long long> g_launches{0};
void count_launch(int n) { g_launches.fetch_add(static_cast<unsigned long long>(n), std::memory_order_relaxed); }
unsigned long long launch_count() { return g_launches.load(std::memory_order_relaxed); }
uint64_t spin_timeout_ns() {
    static const uint64_t ns = [] {
        const char* v = getenv("L32_TP_TIMEOUT_S");
        double sec = (v != nullptr && *v != '\0') ? atof(v) : 120.0;
        if (!(sec >= 1.0)) sec = 1.0;
        if (sec > 86400.0) sec = 86400.0;
        return static_cast<uint64_t>(sec * 1e9);
    }();
    return ns;
}
}  // namespace l32

namespace {

inline cudaStream_t as_stream(void* s) { return static_cast<cudaStream_t>(s); }
inline bool dtype_ok(int dtype) { return dtype == L32_BF16 || dtype == L32_FP16; }
inline size_t align256(size_t v) { return (v + 255) & ~static_cast<size_t>(255); }

// Largest token count routed to the weight-streaming small-M kernels (ffn_decode.cu); above it the tiled
// tcgen05 GEMM is used.  L32_DECODE_MAX_TOKENS overrides it for experiments (0 disables the small-M path).
int decode_max_tokens() {
    const char* v = getenv("L32_DECODE_MAX_TOKENS");
    if (v != nullptr && *v != '\0') return atoi(v);
    return 128;
}

GemmOperand op(const void* p, int64_t ld, int mn_major) {
    GemmOperand o;
    o.ptr = p;
    o.ld = ld;
    o.mn_major = mn_major;
    return o;
}

GemmProblem blank(int m, int n, int dtype) {
    GemmProblem g;
    memset(&g, 0, sizeof(g));
    g.m = m;
    g.n = n;
    g.num_phases = 1;
    g.dtype = dtype;
    return g;
}

// dx[T,H] = d_gate[T,I] * w_gate[I,H] + d_up[T,I] * w_up[I,H]   (weights consumed as MN-major B operands)
int dgrad_x(const void* d_gate, const void* d_up, const void* w_gate, const void* w_up, void* dx, int tokens, int hidden,
            int inter, int dtype, cudaStream_t s) {
    GemmProblem g = blank(tokens, hidden, dtype);
    g.num_phases = 2;
    g.k[0] = g.k[1] = inter;
    g.a[0] = op(d_gate, inter, 0);
    g.a[1] = op(d_up, inter, 0);
    g.b[0] = op(w_gate, hidden, 1);
    g.b[1] = op(w_up, hidden, 1);
    g.epilogue = EPI_STORE;
    g.d[0] = dx;
    g.ldd = hidden;
    return gemm_sm100(g, s);
}

// dw[R,C] = lhs[T,R]^T * rhs[T,C]   (both operands consumed as MN-major, reduction over tokens)
int wgrad(const void* lhs, int r, const void* rhs, int c, void* dw, int tokens, int dtype, cudaStream_t s) {
    GemmProblem g = blank(r, c, dtype);
    g.k[0] = tokens;
    g.a[0] = op(lhs, r, 1);
    g.b[0] = op(rhs, c, 1);
    g.epilogue = EPI_STORE;
    g.d[0] = dw;
    g.ldd = c;
    return gemm_sm100(g, s);
}

// Several weight gradients dw_i[R_i, C_i] = lhs_i[T, R_i]^T rhs_i[T, C_i] as ONE grouped launch: their tiles share the
// persistent loop, so the machine sees e.g. 3 x 896 tiles = 36.3 waves instead of 3 x (12.1 run as 13).
struct WgradItem {
    const void* lhs; int r; const void* rhs; int c; void* dw;
};
int wgrad_group(const WgradItem* items, int count, int tokens, int dtype, cudaStream_t s) {
    if (count == 1 || tokens <= 128) {
        for (int i = 0; i < count; ++i) {
            const int rc = wgrad(items[i].lhs, items[i].r, items[i].rhs, items[i].c, items[i].dw, tokens, dtype, s);
            if (rc != L32_OK) return rc;
        }
        return L32_OK;
    }
    GemmProblem g = blank(items[0].r, items[0].c, dtype);
    g.k[0] = tokens;
    g.a[0] = op(items[0].lhs, items[0].r, 1);
    g.b[0] = op(items[0].rhs, items[0].c, 1);
    g.epilogue = EPI_STORE;
    g.d[0] = items[0].dw;
    g.ldd = items[0].c;
    g.cta_group = 2;
    g.group_count = count;
    for (int i = 0; i < count; ++i) {
        GroupMember& q = g.group[i];
        q.a = items[i].lhs; q.lda = items[i].r; q.m = items[i].r;
        q.b = items[i].rhs; q.ldb = items[i].c; q.n = items[i].c;
        q.d = items[i].dw; q.ldd = items[i].c;
    }
    return gemm_sm100(g, s);
}

bool shapes_ok(int64_t tokens, int hidden, int inter) {
    return tokens >= 0 && tokens <= 0x7fffffff && hidden > 0 && inter > 0 && (hidden % 8) == 0 && (inter % 8) == 0;
}

}  // namespace

extern "C" {

int l32_abi_version(void) { return 3; }

unsigned long long l32_kernel_launch_count(void) { return launch_count(); }

const char* l32_error_string(int code) {
    switch (code) {
        case L32_OK: return "success";
        case L32_ERR_BAD_DTYPE: return "unsupported dtype (expected L32_DTYPE_BF16 or L32_DTYPE_FP16)";
        case L32_ERR_BAD_SHAPE: return "unsupported shape (sizes must be positive; hidden/inter multiples of 8)";
        case L32_ERR_BAD_ALIGN: return "pointer not 16-byte aligned or row pitch not a multiple of 8 elements";
        case L32_ERR_NULL: return "required pointer is null";
        case L32_ERR_DRIVER: return "CUDA driver entry point unavailable (cuTensorMapEncodeTiled)";
        case L32_ERR_WORKSPACE: return "workspace too small or misaligned";
        case L32_ERR_NOT_RESIDENT: return "tensor-parallel kernel: the persistent grid cannot be co-resident on this context's SMs";
        default: return code > 0 ? cudaGetErrorString(static_cast<cudaError_t>(code)) : "unknown error";
    }
}

int l32_add_rmsnorm_forward(const void* x, const void* residual, const void* weight, void* y, void* h_out, float* rms,
                            int64_t rows, int hidden, float eps, int dtype, void* stream) {
    if (!dtype_ok(dtype)) return L32_ERR_BAD_DTYPE;
    if (rows < 0 || hidden <= 0) return L32_ERR_BAD_SHAPE;
    if (rows == 0) return L32_OK;
    if (x == nullptr || weight == nullptr || y == nullptr) return L32_ERR_NULL;
    return static_cast<int>(add_rmsnorm_fwd(x, residual, weight, y, h_out, rms, rows, hidden, eps, dtype, as_stream(stream)));
}

size_t l32_rmsnorm_backward_workspace_bytes(int64_t rows, int hidden) {
    if (rows < 0 || hidden <= 0) return 0;
    return rmsnorm_bwd_workspace_bytes(rows, hidden);
}

int l32_rmsnorm_backward(const void* dy, const void* h, const void* weight, const float* rms, void* dx, void* dweight,
                         void* workspace, size_t workspace_bytes, int64_t rows, int hidden, int dtype, void* stream) {
    return l32_rmsnorm_backward_add(dy, h, weight, rms, nullptr, dx, nullptr, dweight, workspace, workspace_bytes, rows, hidden,
                                    dtype, stream);
}

int l32_rmsnorm_backward_add(const void* dy, const void* h, const void* weight, const float* rms, const void* addend, void* dx,
                             void* dx_plain, void* dweight, void* workspace, size_t workspace_bytes, int64_t rows, int hidden,
                             int dtype, void* stream) {
    if (!dtype_ok(dtype)) return L32_ERR_BAD_DTYPE;
    if (rows < 0 || hidden <= 0) return L32_ERR_BAD_SHAPE;
    if (dy == nullptr || h == nullptr || weight == nullptr || rms == nullptr || dx == nullptr) {
        if (rows != 0) return L32_ERR_NULL;
    }
    if (rows > 0 && (workspace == nullptr || workspace_bytes < rmsnorm_bwd_workspace_bytes(rows, hidden) ||
                     !is_aligned16(workspace)))
        return L32_ERR_WORKSPACE;
    return static_cast<int>(rmsnorm_bwd(dy, h, weight, rms, addend, dx, dx_plain, dweight, static_cast<float*>(workspace), rows,
                                        hidden, dtype, as_stream(stream)));
}

int l32_swiglu_forward(const void* x, const void* w_gate, const void* w_up, const void* b_gate, const void* b_up,
                       void* act, void* gate_cache, void* up_cache, int64_t tokens, int hidden, int inter, int dtype,
                       void* stream) {
    if (!dtype_ok(dtype)) return L32_ERR_BAD_DTYPE;
    if (!shapes_ok(tokens, hidden, inter)) return L32_ERR_BAD_SHAPE;
    if (tokens == 0) return L32_OK;
    if (x == nullptr || w_gate == nullptr || w_up == nullptr || act == nullptr) return L32_ERR_NULL;
    if ((gate_cache == nullptr) != (up_cache == nullptr)) return L32_ERR_NULL;
    if (tokens <= decode_max_tokens()) {
        const int rc = ffn_decode_swiglu(x, w_gate, w_up, b_gate, b_up, act, gate_cache, up_cache, static_cast<int>(tokens),
                                         hidden, inter, dtype, as_stream(stream));
        if (rc != L32_ERR_BAD_SHAPE) return rc;   // shape outside the small-M kernel's envelope: use the tiled kernel
    }
    GemmProblem g = blank(static_cast<int>(tokens), inter, dtype);
    g.k[0] = hidden;
    g.a[0] = op(x, hidden, 0);
    g.b[0] = op(w_gate, hidden, 0);
    g.b[1] = op(w_up, hidden, 0);
    g.epilogue = EPI_SWIGLU;
    g.d[0] = act;
    g.d[1] = gate_cache;
    g.d[2] = up_cache;
    g.bias[0] = b_gate;
    g.bias[1] = b_up;
    g.ldd = inter;
    return gemm_sm100(g, as_stream(stream));
}

namespace {
int linear_forward_add(const void* a, const void* w, const void* bias, const void* addend, void* y, int64_t tokens,
                       int in_features, int out_features, int dtype, void* stream);
}

int l32_linear_group_forward(const void* a, const void* const* w, void* const* y, const int* out_features, int count, int64_t tokens,
                             int in_features, int dtype, void* stream) {
    if (!dtype_ok(dtype)) return L32_ERR_BAD_DTYPE;
    if (count < 1 || count > 3 || w == nullptr || y == nullptr || out_features == nullptr) return L32_ERR_BAD_SHAPE;
    for (int i = 0; i < count; ++i) {
        if (!shapes_ok(tokens, in_features, out_features[i])) return L32_ERR_BAD_SHAPE;
        if (w[i] == nullptr || y[i] == nullptr) return L32_ERR_NULL;
    }
    if (tokens == 0) return L32_OK;
    if (a == nullptr) return L32_ERR_NULL;
    cudaStream_t s = as_stream(stream);
    if (tokens <= decode_max_tokens()) {
        const int rc = ffn_decode_linear_group(a, w, y, out_features, count, static_cast<int>(tokens), in_features, dtype, s);
        if (rc != L32_ERR_BAD_SHAPE) return rc;
    }
    if (count == 1 || tokens <= 128) {          // (the grouped tile loop wants 2-CTA tiles of 256 rows)
        for (int i = 0; i < count; ++i) {
            const int rc = linear_forward_add(a, w[i], nullptr, nullptr, y[i], tokens, in_features, out_features[i], dtype, stream);
            if (rc != L32_OK) return rc;
        }
        return L32_OK;
    }
    // tiled GEMMs: one grouped launch -- the problems' tiles share the persistent loop (no wave tail per projection)
    GemmProblem g = blank(static_cast<int>(tokens), out_features[0], dtype);
    g.k[0] = in_features;
    g.a[0] = op(a, in_features, 0);
    g.b[0] = op(w[0], in_features, 0);
    g.epilogue = EPI_STORE;
    g.d[0] = y[0];
    g.ldd = out_features[0];
    g.cta_group = 2;
    g.group_count = count;
    for (int i = 0; i < count; ++i) {
        GroupMember& q = g.group[i];
        q.a = a; q.lda = in_features; q.m = static_cast<int>(tokens);
        q.b = w[i]; q.ldb = in_features; q.n = out_features[i];
        q.d = y[i]; q.ldd = out_features[i];
    }
    return gemm_sm100(g, s);
}

int l32_linear_forward(const void* a, const void* w, const void* bias, void* y, int64_t tokens, int in_features,
                       int out_features, int dtype, void* stream) {
    return linear_forward_add(a, w, bias, nullptr, y, tokens, in_features, out_features, dtype, stream);
}

int l32_block_tail_forward(const void* attn_out, const void* residual, const void* norm_weight, float eps, const void* w_gate,
                           const void* w_up, const void* w_down, void* out, void* normed_ws, void* act_ws, int64_t tokens,
                           int hidden, int inter, int dtype, void* stream) {
    return l32_block_tail_forward_ex(attn_out, residual, norm_weight, eps, w_gate, w_up, w_down, out, normed_ws, act_ws, nullptr,
                                     nullptr, nullptr, nullptr, nullptr, 0.f, nullptr, nullptr, tokens, hidden, inter, dtype,
                                     stream);
}

int l32_block_tail_forward_ex(const void* attn_out, const void* residual, const void* norm_weight, float eps, const void* w_gate,
                              const void* w_up, const void* w_down, void* out, void* normed_ws, void* act_ws, void* h_out,
                              float* rms_out, void* gate_cache, void* up_cache, const void* next_norm_weight, float next_eps,
                              void* next_normed, float* next_rms, int64_t tokens, int hidden, int inter, int dtype,
                              void* stream) {
    if (!dtype_ok(dtype)) return L32_ERR_BAD_DTYPE;
    if (!shapes_ok(tokens, hidden, inter)) return L32_ERR_BAD_SHAPE;
    if (tokens == 0) return L32_OK;
    if (attn_out == nullptr || norm_weight == nullptr || w_gate == nullptr || w_up == nullptr || w_down == nullptr || out == nullptr)
        return L32_ERR_NULL;
    if (normed_ws == nullptr || act_ws == nullptr) return L32_ERR_WORKSPACE;
    if ((gate_cache == nullptr) != (up_cache == nullptr)) return L32_ERR_NULL;
    if (next_norm_weight != nullptr && next_normed == nullptr) return L32_ERR_NULL;
    // norm2(attn_out, residual)  [+ h, rms for the backward]
    int rc = l32_add_rmsnorm_forward(attn_out, residual, norm_weight, normed_ws, residual != nullptr ? h_out : nullptr, rms_out,
                                     tokens, hidden, eps, dtype, stream);
    if (rc != L32_OK) return rc;
    // fused gate/up + SiLU*mul  [+ caches]
    rc = l32_swiglu_forward(normed_ws, w_gate, w_up, nullptr, nullptr, act_ws, gate_cache, up_cache, tokens, hidden, inter, dtype,
                            stream);
    if (rc != L32_OK) return rc;
    // down projection whose epilogue adds attn_out: out = attn_out + ff_out  (Model/model.py:273)
    rc = linear_forward_add(act_ws, w_down, nullptr, attn_out, out, tokens, inter, hidden, dtype, stream);
    if (rc != L32_OK || next_norm_weight == nullptr) return rc;
    // chained: the next block's norm1 (or final_norm) of the sum, while `out` is still in L2 (Model/model.py:267, :346)
    return l32_add_rmsnorm_forward(out, nullptr, next_norm_weight, next_normed, nullptr, next_rms, tokens, hidden, next_eps, dtype,
                                   stream);
}

namespace {
int linear_forward_add(const void* a, const void* w, const void* bias, const void* addend, void* y, int64_t tokens,
                       int in_features, int out_features, int dtype, void* stream) {
    if (!dtype_ok(dtype)) return L32_ERR_BAD_DTYPE;
    if (!shapes_ok(tokens, in_features, out_features)) return L32_ERR_BAD_SHAPE;
    if (tokens == 0) return L32_OK;
    if (a == nullptr || w == nullptr || y == nullptr) return L32_ERR_NULL;
    if (tokens <= decode_max_tokens()) {
        const int rc = ffn_decode_linear(a, w, bias, addend, y, static_cast<int>(tokens), in_features, out_features, dtype,
                                         as_stream(stream));
        if (rc != L32_ERR_BAD_SHAPE) return rc;
    }
    GemmProblem g = blank(static_cast<int>(tokens), out_features, dtype);
    g.k[0] = in_features;
    g.a[0] = op(a, in_features, 0);
    g.b[0] = op(w, in_features, 0);
    g.epilogue = EPI_STORE;
    g.d[0] = y;
    g.e[0] = addend;
    g.bias[0] = bias;
    g.ldd = out_features;
    return gemm_sm100(g, as_stream(stream));
}
}  // namespace

int l32_ffn_forward(const void* x, const void* w_gate, const void* w_up, const void* w_down, const void* b_gate,
                    const void* b_up, const void* b_down, void* y, void* act_ws, void* gate_cache, void* up_cache,
                    int64_t tokens, int hidden, int inter, int dtype, void* stream) {
    if (act_ws == nullptr && tokens > 0) return L32_ERR_WORKSPACE;
    int rc = l32_swiglu_forward(x, w_gate, w_up, b_gate, b_up, act_ws, gate_cache, up_cache, tokens, hidden, inter, dtype, stream);
    if (rc != L32_OK) return rc;
    return l32_linear_forward(act_ws, w_down, b_down, y, tokens, inter, hidden, dtype, stream);
}

size_t l32_swiglu_backward_workspace_bytes(int64_t tokens, int inter) {
    if (tokens < 0 || inter <= 0) return 0;
    return 2 * align256(static_cast<size_t>(tokens) * inter * 2);
}

int l32_swiglu_backward(const void* d_act, const void* x, const void* w_gate, const void* w_up, const void* gate_cache,
                        const void* up_cache, void* dx, void* dw_gate, void* dw_up, void* workspace,
                        size_t workspace_bytes, int64_t tokens, int hidden, int inter, int dtype, void* stream) {
    if (!dtype_ok(dtype)) return L32_ERR_BAD_DTYPE;
    if (!shapes_ok(tokens, hidden, inter)) return L32_ERR_BAD_SHAPE;
    if ((dw_gate == nullptr) != (dw_up == nullptr)) return L32_ERR_NULL;
    cudaStream_t s = as_stream(stream);
    if (tokens == 0) {
        if (dw_gate != nullptr) {
            cudaError_t e = cudaMemsetAsync(dw_gate, 0, static_cast<size_t>(inter) * hidden * 2, s);
            if (e == cudaSuccess) e = cudaMemsetAsync(dw_up, 0, static_cast<size_t>(inter) * hidden * 2, s);
            return static_cast<int>(e);
        }
        return L32_OK;
    }
    if (d_act == nullptr || x == nullptr || w_gate == nullptr || w_up == nullptr || gate_cache == nullptr || up_cache == nullptr)
        return L32_ERR_NULL;
    if (workspace == nullptr || workspace_bytes < l32_swiglu_backward_workspace_bytes(tokens, inter) || !is_aligned16(workspace))
        return L32_ERR_WORKSPACE;
    const size_t part = align256(static_cast<size_t>(tokens) * inter * 2);
    void* d_gate = workspace;
    void* d_up = static_cast<uint8_t*>(workspace) + part;
    const int t = static_cast<int>(tokens);
    cudaError_t e = swiglu_bwd_elementwise(d_act, gate_cache, up_cache, d_gate, d_up, tokens * inter, dtype, s);
    if (e != cudaSuccess) return static_cast<int>(e);
    int rc = L32_OK;
    if (dx != nullptr) rc = dgrad_x(d_gate, d_up, w_gate, w_up, dx, t, hidden, inter, dtype, s);
    if (rc != L32_OK) return rc;
    if (dw_gate != nullptr) {
        const WgradItem items[2] = {{d_gate, inter, x, hidden, dw_gate}, {d_up, inter, x, hidden, dw_up}};
        rc = wgrad_group(items, 2, t, dtype, s);
    }
    return rc;
}

size_t l32_ffn_backward_workspace_bytes(int64_t tokens, int inter) {
    if (tokens < 0 || inter <= 0) return 0;
    return 3 * align256(static_cast<size_t>(tokens) * inter * 2);
}

int l32_ffn_backward(const void* dy, const void* x, const void* w_gate, const void* w_up, const void* w_down,
                     const void* gate_cache, const void* up_cache, void* dx, void* dw_gate, void* dw_up, void* dw_down,
                     void* workspace, size_t workspace_bytes, int64_t tokens, int hidden, int inter, int dtype,
                     void* stream) {
    if (!dtype_ok(dtype)) return L32_ERR_BAD_DTYPE;
    if (!shapes_ok(tokens, hidden, inter)) return L32_ERR_BAD_SHAPE;
    if ((dw_gate == nullptr) != (dw_up == nullptr)) return L32_ERR_NULL;
    cudaStream_t s = as_stream(stream);
    const size_t wbytes = static_cast<size_t>(inter) * hidden * 2;
    if (tokens == 0) {
        cudaError_t e = cudaSuccess;
        if (dw_gate != nullptr) {
            e = cudaMemsetAsync(dw_gate, 0, wbytes, s);
            if (e == cudaSuccess) e = cudaMemsetAsync(dw_up, 0, wbytes, s);
        }
        if (e == cudaSuccess && dw_down != nullptr) e = cudaMemsetAsync(dw_down, 0, wbytes, s);
        return static_cast<int>(e);
    }
    if (dy == nullptr || x == nullptr || w_gate == nullptr || w_up == nullptr || w_down == nullptr || gate_cache == nullptr ||
        up_cache == nullptr)
        return L32_ERR_NULL;
    if (workspace == nullptr || workspace_bytes < l32_ffn_backward_workspace_bytes(tokens, inter) || !is_aligned16(workspace))
        return L32_ERR_WORKSPACE;
    const size_t part = align256(static_cast<size_t>(tokens) * inter * 2);
    void* d_gate = workspace;
    void* d_up = static_cast<uint8_t*>(workspace) + part;
    void* act = static_cast<uint8_t*>(workspace) + 2 * part;
    const int t = static_cast<int>(tokens);

    // d_act = dy * w_down (w_down[H,I] consumed as an MN-major B operand); the epilogue turns it into
    // d_gate / d_up (SiLU' recomputed in registers) and re-materialises act for the w_down gradient.
    GemmProblem g = blank(t, inter, dtype);
    g.k[0] = hidden;
    g.a[0] = op(dy, hidden, 0);
    g.b[0] = op(w_down, inter, 1);
    g.epilogue = EPI_SWIGLU_BWD;
    g.d[0] = d_gate;
    g.d[1] = d_up;
    g.d[2] = (dw_down != nullptr) ? act : nullptr;
    g.e[0] = gate_cache;
    g.e[1] = up_cache;
    g.ldd = inter;
    int rc = gemm_sm100(g, s);
    if (rc != L32_OK) return rc;
    if (dx != nullptr) {
        rc = dgrad_x(d_gate, d_up, w_gate, w_up, dx, t, hidden, inter, dtype, s);
        if (rc != L32_OK) return rc;
    }
    WgradItem items[3];
    int count = 0;
    if (dw_gate != nullptr) {
        items[count++] = WgradItem{d_gate, inter, x, hidden, dw_gate};
        items[count++] = WgradItem{d_up, inter, x, hidden, dw_up};
    }
    if (dw_down != nullptr) items[count++] = WgradItem{dy, hidden, act, inter, dw_down};
    if (count > 0) rc = wgrad_group(items, count, t, dtype, s);
    return rc;
}

int l32_ffn_lora_forward(const void* x, const void* w_gate, const void* w_up, const void* w_down, const void* lora_a,
                         const void* lora_bs, void* y, void* act_ws, void* t_out, void* gate_cache, void* up_cache,
                         int64_t tokens, int hidden, int inter, int rank, int dtype, void* stream) {
    if (!dtype_ok(dtype)) return L32_ERR_BAD_DTYPE;
    if (!shapes_ok(tokens, hidden, inter) || rank <= 0 || rank > 64 || (rank % 8) != 0) return L32_ERR_BAD_SHAPE;
    if (tokens == 0) return L32_OK;
    if (w_down == nullptr || lora_a == nullptr || lora_bs == nullptr || y == nullptr || t_out == nullptr) return L32_ERR_NULL;
    if (act_ws == nullptr) return L32_ERR_WORKSPACE;
    cudaStream_t s = as_stream(stream);
    const int t = static_cast<int>(tokens);
    // act through the tiled kernel: the small-M path has no two-phase down projection
    GemmProblem g = blank(t, inter, dtype);
    g.k[0] = hidden;
    g.a[0] = op(x, hidden, 0);
    g.b[0] = op(w_gate, hidden, 0);
    g.b[1] = op(w_up, hidden, 0);
    g.epilogue = EPI_SWIGLU;
    g.d[0] = act_ws;
    g.d[1] = gate_cache;
    g.d[2] = up_cache;
    g.ldd = inter;
    if (x == nullptr || w_gate == nullptr || w_up == nullptr) return L32_ERR_NULL;
    if ((gate_cache == nullptr) != (up_cache == nullptr)) return L32_ERR_NULL;
    int rc = gemm_sm100(g, s);
    if (rc != L32_OK) return rc;
    // t = act lora_a^T  [tokens, rank]
    g = blank(t, rank, dtype);
    g.k[0] = inter;
    g.a[0] = op(act_ws, inter, 0);
    g.b[0] = op(lora_a, inter, 0);
    g.epilogue = EPI_STORE;
    g.d[0] = t_out;
    g.ldd = rank;
    rc = gemm_sm100(g, s);
    if (rc != L32_OK) return rc;
    // y = act w_down^T + t lora_bs^T : one kernel, two accumulation phases (K = inter, then K = rank)
    g = blank(t, hidden, dtype);
    g.num_phases = 2;
    g.k[0] = inter;
    g.k[1] = rank;
    g.a[0] = op(act_ws, inter, 0);
    g.b[0] = op(w_down, inter, 0);
    g.a[1] = op(t_out, rank, 0);
    g.b[1] = op(lora_bs, rank, 0);
    g.epilogue = EPI_STORE;
    g.d[0] = y;
    g.ldd = hidden;
    return gemm_sm100(g, s);
}

size_t l32_ffn_lora_backward_workspace_bytes(int64_t tokens, int inter, int rank) {
    if (tokens < 0 || inter <= 0 || rank <= 0) return 0;
    return 3 * align256(static_cast<size_t>(tokens) * inter * 2) + align256(static_cast<size_t>(tokens) * rank * 2);
}

int l32_ffn_lora_backward(const void* dy, const void* x, const void* w_gate, const void* w_up, const void* w_down,
                          const void* lora_a, const void* lora_bs, const void* t_saved, const void* gate_cache,
                          const void* up_cache, void* dx, void* dw_gate, void* dw_up, void* dlora_a, void* dlora_bs,
                          void* workspace, size_t workspace_bytes, int64_t tokens, int hidden, int inter, int rank, int dtype,
                          void* stream) {
    if (!dtype_ok(dtype)) return L32_ERR_BAD_DTYPE;
    if (!shapes_ok(tokens, hidden, inter) || rank <= 0 || rank > 64 || (rank % 8) != 0) return L32_ERR_BAD_SHAPE;
    if ((dw_gate == nullptr) != (dw_up == nullptr)) return L32_ERR_NULL;
    cudaStream_t s = as_stream(stream);
    if (tokens == 0) {
        cudaError_t e = cudaSuccess;
        const size_t wbytes = static_cast<size_t>(inter) * hidden * 2;
        if (dw_gate != nullptr) {
            e = cudaMemsetAsync(dw_gate, 0, wbytes, s);
            if (e == cudaSuccess) e = cudaMemsetAsync(dw_up, 0, wbytes, s);
        }
        if (e == cudaSuccess && dlora_a != nullptr) e = cudaMemsetAsync(dlora_a, 0, static_cast<size_t>(rank) * inter * 2, s);
        if (e == cudaSuccess && dlora_bs != nullptr) e = cudaMemsetAsync(dlora_bs, 0, static_cast<size_t>(hidden) * rank * 2, s);
        return static_cast<int>(e);
    }
    if (dy == nullptr || x == nullptr || w_gate == nullptr || w_up == nullptr || w_down == nullptr || lora_a == nullptr ||
        lora_bs == nullptr || t_saved == nullptr || gate_cache == nullptr || up_cache == nullptr)
        return L32_ERR_NULL;
    if (workspace == nullptr || workspace_bytes < l32_ffn_lora_backward_workspace_bytes(tokens, inter, rank) ||
        !is_aligned16(workspace))
        return L32_ERR_WORKSPACE;
    const size_t part = align256(static_cast<size_t>(tokens) * inter * 2);
    void* d_gate = workspace;
    void* d_up = static_cast<uint8_t*>(workspace) + part;
    void* act = static_cast<uint8_t*>(workspace) + 2 * part;
    void* u = static_cast<uint8_t*>(workspace) + 3 * part;
    const int t = static_cast<int>(tokens);

    // u = dy lora_bs  [tokens, rank]   (lora_bs [hidden, rank] consumed as an MN-major B operand)
    GemmProblem g = blank(t, rank, dtype);
    g.k[0] = hidden;
    g.a[0] = op(dy, hidden, 0);
    g.b[0] = op(lora_bs, rank, 1);
    g.epilogue = EPI_STORE;
    g.d[0] = u;
    g.ldd = rank;
    int rc = gemm_sm100(g, s);
    if (rc != L32_OK) return rc;
    // d_act = dy w_down + u lora_a (two phases), SiLU' recomputed in the epilogue -> d_gate, d_up (+ act for dlora_a)
    g = blank(t, inter, dtype);
    g.num_phases = 2;
    g.k[0] = hidden;
    g.k[1] = rank;
    g.a[0] = op(dy, hidden, 0);
    g.b[0] = op(w_down, inter, 1);
    g.a[1] = op(u, rank, 0);
    g.b[1] = op(lora_a, inter, 1);
    g.epilogue = EPI_SWIGLU_BWD;
    g.d[0] = d_gate;
    g.d[1] = d_up;
    g.d[2] = (dlora_a != nullptr) ? act : nullptr;
    g.e[0] = gate_cache;
    g.e[1] = up_cache;
    g.ldd = inter;
    rc = gemm_sm100(g, s);
    if (rc != L32_OK) return rc;
    if (dx != nullptr) {
        rc = dgrad_x(d_gate, d_up, w_gate, w_up, dx, t, hidden, inter, dtype, s);
        if (rc != L32_OK) return rc;
    }
    if (dw_gate != nullptr) {
        const WgradItem items[2] = {{d_gate, inter, x, hidden, dw_gate}, {d_up, inter, x, hidden, dw_up}};
        rc = wgrad_group(items, 2, t, dtype, s);
        if (rc != L32_OK) return rc;
    }
    if (dlora_bs != nullptr) {   // [hidden, rank] = dy^T t
        rc = wgrad(dy, hidden, t_saved, rank, dlora_bs, t, dtype, s);
        if (rc != L32_OK) return rc;
    }
    if (dlora_a != nullptr) rc = wgrad(u, rank, act, inter, dlora_a, t, dtype, s);   // [rank, inter] = u^T act
    return rc;
}

int l32_linear_lora_forward(const void* x, const void* x_lora, const void* w, const void* bias, const void* lora_a,
                            const void* lora_bs, void* y, void* t_out, int64_t tokens, int in_features, int out_features, int rank,
                            int dtype, void* stream) {
    if (!dtype_ok(dtype)) return L32_ERR_BAD_DTYPE;
    if (!shapes_ok(tokens, in_features, out_features) || rank <= 0 || rank > 64 || (rank % 8) != 0) return L32_ERR_BAD_SHAPE;
    if (tokens == 0) return L32_OK;
    if (x == nullptr || w == nullptr || lora_a == nullptr || lora_bs == nullptr || y == nullptr || t_out == nullptr) return L32_ERR_NULL;
    cudaStream_t s = as_stream(stream);
    const int t = static_cast<int>(tokens);
    // t = dropout(x) lora_a^T  [tokens, rank]
    GemmProblem g = blank(t, rank, dtype);
    g.k[0] = in_features;
    g.a[0] = op(x_lora != nullptr ? x_lora : x, in_features, 0);
    g.b[0] = op(lora_a, in_features, 0);
    g.epilogue = EPI_STORE;
    g.d[0] = t_out;
    g.ldd = rank;
    int rc = gemm_sm100(g, s);
    if (rc != L32_OK) return rc;
    // y = x w^T + t lora_bs^T (+ bias): one kernel, two accumulation phases (K = in_features, then K = rank)
    g = blank(t, out_features, dtype);
    g.num_phases = 2;
    g.k[0] = in_features;
    g.k[1] = rank;
    g.a[0] = op(x, in_features, 0);
    g.b[0] = op(w, in_features, 0);
    g.a[1] = op(t_out, rank, 0);
    g.b[1] = op(lora_bs, rank, 0);
    g.epilogue = EPI_STORE;
    g.d[0] = y;
    g.bias[0] = bias;
    g.ldd = out_features;
    return gemm_sm100(g, s);
}

int l32_linear_lora_backward(const void* dy, const void* x_lora, const void* w, const void* lora_a, const void* lora_bs,
                             const void* t_saved, const void* dx_addend, void* dx, void* dlora_a, void* dlora_bs, void* u_out,
                             int64_t tokens, int in_features, int out_features, int rank, int dtype, void* stream) {
    if (!dtype_ok(dtype)) return L32_ERR_BAD_DTYPE;
    if (!shapes_ok(tokens, in_features, out_features) || rank <= 0 || rank > 64 || (rank % 8) != 0) return L32_ERR_BAD_SHAPE;
    cudaStream_t s = as_stream(stream);
    if (tokens == 0) {
        cudaError_t e = cudaSuccess;
        if (dlora_a != nullptr) e = cudaMemsetAsync(dlora_a, 0, static_cast<size_t>(rank) * in_features * 2, s);
        if (e == cudaSuccess && dlora_bs != nullptr) e = cudaMemsetAsync(dlora_bs, 0, static_cast<size_t>(out_features) * rank * 2, s);
        return static_cast<int>(e);
    }
    if (dy == nullptr || w == nullptr || lora_a == nullptr || lora_bs == nullptr) return L32_ERR_NULL;
    if ((dlora_a != nullptr && x_lora == nullptr) || (dlora_bs != nullptr && t_saved == nullptr)) return L32_ERR_NULL;
    // u is needed by dlora_a and by the fused (no-dropout) dx; a pure "dx = dy w + addend" call may leave it out
    if (u_out == nullptr && (dlora_a != nullptr || (dx != nullptr && dx_addend == nullptr))) return L32_ERR_NULL;
    const int t = static_cast<int>(tokens);
    GemmProblem g;
    int rc = L32_OK;
    if (u_out != nullptr) {
        // u = dy lora_bs  [tokens, rank]   (lora_bs [out, rank] consumed as an MN-major B operand)
        g = blank(t, rank, dtype);
        g.k[0] = out_features;
        g.a[0] = op(dy, out_features, 0);
        g.b[0] = op(lora_bs, rank, 1);
        g.epilogue = EPI_STORE;
        g.d[0] = u_out;
        g.ldd = rank;
        rc = gemm_sm100(g, s);
        if (rc != L32_OK) return rc;
    }
    if (dx != nullptr) {
        // no dropout: dx = dy w + u lora_a in ONE kernel (two accumulation phases, both weights consumed MN-major);
        // with dropout the caller passes the masked adapter term as `dx_addend` and the epilogue adds it: dx = dy w + addend
        g = blank(t, in_features, dtype);
        g.k[0] = out_features;
        g.a[0] = op(dy, out_features, 0);
        g.b[0] = op(w, in_features, 1);
        if (dx_addend == nullptr) {
            g.num_phases = 2;
            g.k[1] = rank;
            g.a[1] = op(u_out, rank, 0);
            g.b[1] = op(lora_a, in_features, 1);
        } else {
            g.e[0] = dx_addend;
        }
        g.epilogue = EPI_STORE;
        g.d[0] = dx;
        g.ldd = in_features;
        rc = gemm_sm100(g, s);
        if (rc != L32_OK) return rc;
    }
    if (dlora_bs != nullptr) {   // [out, rank] = dy^T t
        rc = wgrad(dy, out_features, t_saved, rank, dlora_bs, t, dtype, s);
        if (rc != L32_OK) return rc;
    }
    if (dlora_a != nullptr) rc = wgrad(u_out, rank, x_lora, in_features, dlora_a, t, dtype, s);   // [rank, in] = u^T dropout(x)
    return rc;
}

size_t l32_lm_head_ce_workspace_bytes(int64_t tokens, int vocab) {
    if (tokens < 0 || vocab <= 0) return 0;
    const size_t tiles_n = static_cast<size_t>((vocab + 255) / 256);
    return align256(static_cast<size_t>(tokens) * tiles_n * 8) + align256(static_cast<size_t>(tokens) * 4);
}

int l32_lm_head_ce_forward(const void* hidden_states, const void* w, const int64_t* labels, long long ignore_index, void* logits,
                           float* lse, float* loss_rows, float* loss_and_count, void* workspace, size_t workspace_bytes,
                           int64_t tokens, int hidden, int vocab, int dtype, void* stream) {
    if (!dtype_ok(dtype)) return L32_ERR_BAD_DTYPE;
    if (!shapes_ok(tokens, hidden, vocab)) return L32_ERR_BAD_SHAPE;
    if (tokens == 0) return L32_OK;
    if (hidden_states == nullptr || w == nullptr || labels == nullptr || logits == nullptr || lse == nullptr ||
        loss_rows == nullptr || loss_and_count == nullptr)
        return L32_ERR_NULL;
    if (workspace == nullptr || workspace_bytes < l32_lm_head_ce_workspace_bytes(tokens, vocab) || !is_aligned16(workspace))
        return L32_ERR_WORKSPACE;
    const int tiles_n = (vocab + 255) / 256;
    void* partials = workspace;
    float* target = reinterpret_cast<float*>(static_cast<uint8_t*>(workspace) + align256(static_cast<size_t>(tokens) * tiles_n * 8));
    // logits = hidden_states w^T with the softmax statistics gathered in the epilogue (no second pass over [tokens, vocab])
    GemmProblem g = blank(static_cast<int>(tokens), vocab, dtype);
    g.k[0] = hidden;
    g.a[0] = op(hidden_states, hidden, 0);
    g.b[0] = op(w, hidden, 0);
    g.epilogue = EPI_CE;
    g.d[0] = logits;
    g.ldd = vocab;
    g.cta_group = 2;      // the statistics are laid out per 256-column tile of the paired kernel
    g.ce.labels = reinterpret_cast<const long long*>(labels);
    g.ce.partials = partials;
    g.ce.target = target;
    int rc = gemm_sm100(g, as_stream(stream));
    if (rc != L32_OK) return rc;
    return static_cast<int>(ce_reduce(partials, target, reinterpret_cast<const long long*>(labels), ignore_index, tokens, tiles_n,
                                      vocab, lse, loss_rows, loss_and_count, as_stream(stream)));
}

int l32_lm_head_ce_backward(const void* logits, const float* lse, const int64_t* labels, long long ignore_index,
                            const float* loss_and_count, const float* grad_loss, const void* hidden_states, const void* w,
                            void* dlogits,
                            void* d_hidden, void* dw, int64_t tokens, int hidden, int vocab, int dtype, void* stream) {
    if (!dtype_ok(dtype)) return L32_ERR_BAD_DTYPE;
    if (!shapes_ok(tokens, hidden, vocab)) return L32_ERR_BAD_SHAPE;
    cudaStream_t s = as_stream(stream);
    if (tokens == 0) {
        if (dw != nullptr) return static_cast<int>(cudaMemsetAsync(dw, 0, static_cast<size_t>(vocab) * hidden * 2, s));
        return L32_OK;
    }
    if (logits == nullptr || lse == nullptr || labels == nullptr || loss_and_count == nullptr || dlogits == nullptr)
        return L32_ERR_NULL;
    if ((d_hidden != nullptr && w == nullptr) || (dw != nullptr && hidden_states == nullptr)) return L32_ERR_NULL;
    if (!is_aligned16(logits) || !is_aligned16(dlogits)) return L32_ERR_BAD_ALIGN;
    cudaError_t e = ce_backward_logits(logits, lse, reinterpret_cast<const long long*>(labels), ignore_index, loss_and_count,
                                       grad_loss, dlogits, tokens, vocab, dtype, s);
    if (e != cudaSuccess) return static_cast<int>(e);
    const int t = static_cast<int>(tokens);
    int rc = L32_OK;
    if (d_hidden != nullptr) {   // d_hidden = dlogits w   (w [vocab, hidden] consumed as an MN-major B operand)
        GemmProblem g = blank(t, hidden, dtype);
        g.k[0] = vocab;
        g.a[0] = op(dlogits, vocab, 0);
        g.b[0] = op(w, hidden, 1);
        g.epilogue = EPI_STORE;
        g.d[0] = d_hidden;
        g.ldd = hidden;
        rc = gemm_sm100(g, s);
        if (rc != L32_OK) return rc;
    }
    if (dw != nullptr) rc = wgrad(dlogits, vocab, hidden_states, hidden, dw, t, dtype, s);   // [vocab, hidden] = dlogits^T h
    return rc;
}

int l32_rope_kv_append(void* q, const void* k_new, const void* v_new, const int64_t* position_ids, void* cache_k, void* cache_v,
                       int batch, int q_len, int heads, int kv_heads, int head_dim, int max_len, int past_len, float rope_base,
                       int dtype, void* stream) {
    if (!dtype_ok(dtype)) return L32_ERR_BAD_DTYPE;
    if (batch < 0 || q_len < 0 || heads <= 0 || kv_heads <= 0 || (heads % kv_heads) != 0 || head_dim <= 0 || (head_dim % 2) != 0 ||
        max_len <= 0 || past_len < 0 || past_len + q_len > max_len || !(rope_base > 1.0f))
        return L32_ERR_BAD_SHAPE;
    if (batch == 0 || q_len == 0) return L32_OK;
    if (q == nullptr || k_new == nullptr || v_new == nullptr || position_ids == nullptr || cache_k == nullptr || cache_v == nullptr)
        return L32_ERR_NULL;
    return rope_kv_append(q, k_new, v_new, reinterpret_cast<const long long*>(position_ids), cache_k, cache_v, batch, q_len, heads,
                          kv_heads, head_dim, max_len, past_len, rope_base, dtype, as_stream(stream));
}

// Heads of every attention entry point: whole KV groups of 64- or 128-wide heads.
static bool attention_heads_ok(int heads, int kv_heads, int head_dim) {
    return heads > 0 && kv_heads > 0 && (heads % kv_heads) == 0 && (head_dim == 64 || head_dim == 128);
}

size_t l32_gqa_attention_workspace_bytes(int batch, int q_len, int heads, int kv_heads, int head_dim, int kv_len) {
    if (batch <= 0 || q_len <= 0 || heads <= 0 || kv_heads <= 0 || (heads % kv_heads) != 0 || kv_len <= 0) return 0;
    return gqa_attention_workspace_bytes(batch, q_len, heads, kv_heads, head_dim, kv_len);
}

int l32_gqa_attention_forward(const void* q, const void* cache_k, const void* cache_v, const uint8_t* key_keep, void* ctx,
                              void* workspace, size_t workspace_bytes, int batch, int q_len, int heads, int kv_heads, int head_dim,
                              int max_len, int kv_len, int past_len, int causal, int dtype, void* stream) {
    if (!dtype_ok(dtype)) return L32_ERR_BAD_DTYPE;
    if (batch < 0 || q_len < 0 || !attention_heads_ok(heads, kv_heads, head_dim) || max_len <= 0 || kv_len < 0 || kv_len > max_len ||
        past_len < 0)
        return L32_ERR_BAD_SHAPE;
    if (batch == 0 || q_len == 0) return L32_OK;
    if (q == nullptr || cache_k == nullptr || cache_v == nullptr || ctx == nullptr) return L32_ERR_NULL;
    if (!is_aligned16(q) || !is_aligned16(cache_k) || !is_aligned16(cache_v) || !is_aligned16(ctx)) return L32_ERR_BAD_ALIGN;
    if (workspace != nullptr && !is_aligned16(workspace)) return L32_ERR_WORKSPACE;
    return gqa_attention(q, cache_k, cache_v, key_keep, ctx, batch, q_len, heads, kv_heads, head_dim, max_len, kv_len, past_len,
                         causal, workspace, workspace_bytes, dtype, as_stream(stream));
}

// Training forward of GroupQueryAttention's attention core (reference Model/model.py:238-253 under autograd): the flash
// forward of l32_gqa_attention_forward over keys [0, q_len), which also stores the per-row log-sum-exp for the backward.
int l32_gqa_attention_forward_train(const void* q_rot, const void* cache_k, const void* cache_v, const uint8_t* key_keep, void* ctx,
                                    float* lse, int batch, int q_len, int heads, int kv_heads, int head_dim, int max_len, int causal,
                                    int dtype, void* stream) {
    if (!dtype_ok(dtype)) return L32_ERR_BAD_DTYPE;
    if (batch < 0 || q_len < 0 || !attention_heads_ok(heads, kv_heads, head_dim) || max_len < q_len || max_len <= 0)
        return L32_ERR_BAD_SHAPE;
    if (batch == 0 || q_len == 0) return L32_OK;
    if (q_rot == nullptr || cache_k == nullptr || cache_v == nullptr || ctx == nullptr || lse == nullptr) return L32_ERR_NULL;
    if (!is_aligned16(q_rot) || !is_aligned16(cache_k) || !is_aligned16(cache_v) || !is_aligned16(ctx)) return L32_ERR_BAD_ALIGN;
    return gqa_attention_train(q_rot, cache_k, cache_v, key_keep, ctx, lse, batch, q_len, heads, kv_heads, head_dim, max_len, causal,
                               dtype, as_stream(stream));
}

size_t l32_gqa_attention_backward_workspace_bytes(int batch, int q_len, int heads) {
    return gqa_attention_backward_workspace_bytes(batch, q_len, heads);
}

// Backward of the same (reference Model/model.py:238-253 under autograd: the saved softmax, repeat_kv and RoPE backward).
int l32_gqa_attention_backward(const void* d_ctx, const void* q_rot, const void* cache_k, const void* cache_v, const void* ctx,
                               const float* lse, const uint8_t* key_keep, const int64_t* position_ids, void* dq, void* dk, void* dv,
                               void* workspace, size_t workspace_bytes, int batch, int q_len, int heads, int kv_heads, int head_dim,
                               int max_len, int causal, float rope_base, int dtype, void* stream) {
    if (!dtype_ok(dtype)) return L32_ERR_BAD_DTYPE;
    if (batch < 0 || q_len < 0 || !attention_heads_ok(heads, kv_heads, head_dim) || max_len < q_len || max_len <= 0 ||
        !(rope_base > 1.0f))
        return L32_ERR_BAD_SHAPE;
    if (batch == 0 || q_len == 0) return L32_OK;
    if (d_ctx == nullptr || q_rot == nullptr || cache_k == nullptr || cache_v == nullptr || ctx == nullptr || lse == nullptr ||
        position_ids == nullptr || dq == nullptr || dk == nullptr || dv == nullptr || workspace == nullptr)
        return L32_ERR_NULL;
    if (workspace_bytes < gqa_attention_backward_workspace_bytes(batch, q_len, heads) || !is_aligned16(workspace))
        return L32_ERR_WORKSPACE;
    if (!is_aligned16(d_ctx) || !is_aligned16(q_rot) || !is_aligned16(cache_k) || !is_aligned16(cache_v) || !is_aligned16(ctx) ||
        !is_aligned16(dq) || !is_aligned16(dk) || !is_aligned16(dv))
        return L32_ERR_BAD_ALIGN;
    return gqa_attention_backward(d_ctx, q_rot, cache_k, cache_v, ctx, lse, key_keep, reinterpret_cast<const long long*>(position_ids),
                                  dq, dk, dv, workspace, batch, q_len, heads, kv_heads, head_dim, max_len, causal, rope_base, dtype,
                                  as_stream(stream));
}

// Paged KV cache (no reference counterpart: the reference's cache is one torch.cat'ed tensor per layer).  Only the host-side
// arguments can be checked here; the table and length values in device memory are trusted (include/l32_ffn.h).
static bool paged_shape_ok(int batch, int q_len, int heads, int kv_heads, int head_dim, int num_pages, int max_pages_per_seq) {
    return batch >= 0 && q_len >= 0 && attention_heads_ok(heads, kv_heads, head_dim) && num_pages > 0 && max_pages_per_seq > 0 &&
           static_cast<long long>(max_pages_per_seq) * L32_KV_PAGE <= 0x7fffffffll &&
           static_cast<long long>(num_pages) * kv_heads <= 0x7fffffffll;
}

// The checks the three paged attention forwards share, in this order: dtype; shape, with the form's own shape rule (form_ok),
// and the max_kv_len bound; the empty batch; null pointers, with the form's own pointers (ptrs_ok); alignment; then the
// alignment of a workspace that is given.  Returns the code of the first that fails; *run is set when all pass and the batch
// is not empty.
static int paged_forward_check(int dtype, bool form_ok, bool ptrs_ok, const void* q, const void* pool_k, const void* pool_v,
                               const int32_t* block_table, const int32_t* past_lens, const void* ctx, const void* workspace,
                               int batch, int q_len, int heads, int kv_heads, int head_dim, int num_pages, int max_pages_per_seq,
                               int max_kv_len, bool* run) {
    *run = false;
    if (!dtype_ok(dtype)) return L32_ERR_BAD_DTYPE;
    if (!paged_shape_ok(batch, q_len, heads, kv_heads, head_dim, num_pages, max_pages_per_seq) || !form_ok || max_kv_len < 0 ||
        static_cast<long long>(max_kv_len) > static_cast<long long>(max_pages_per_seq) * L32_KV_PAGE)
        return L32_ERR_BAD_SHAPE;
    if (batch == 0 || q_len == 0) return L32_OK;
    if (q == nullptr || pool_k == nullptr || pool_v == nullptr || block_table == nullptr || past_lens == nullptr || ctx == nullptr ||
        !ptrs_ok)
        return L32_ERR_NULL;
    if (!is_aligned16(q) || !is_aligned16(pool_k) || !is_aligned16(pool_v) || !is_aligned16(ctx)) return L32_ERR_BAD_ALIGN;
    if (workspace != nullptr && !is_aligned16(workspace)) return L32_ERR_WORKSPACE;
    *run = true;
    return L32_OK;
}

int l32_rope_kv_append_paged(void* q, const void* k_new, const void* v_new, const int64_t* position_ids, void* pool_k, void* pool_v,
                             const int32_t* block_table, const int32_t* past_lens, const int32_t* new_lens, int batch, int q_len,
                             int heads, int kv_heads, int head_dim, int num_pages, int max_pages_per_seq, float rope_base, int dtype,
                             void* stream) {
    if (!dtype_ok(dtype)) return L32_ERR_BAD_DTYPE;
    if (!paged_shape_ok(batch, q_len, heads, kv_heads, head_dim, num_pages, max_pages_per_seq) || !(rope_base > 1.0f))
        return L32_ERR_BAD_SHAPE;
    if (batch == 0 || q_len == 0) return L32_OK;
    if (q == nullptr || k_new == nullptr || v_new == nullptr || position_ids == nullptr || pool_k == nullptr || pool_v == nullptr ||
        block_table == nullptr || past_lens == nullptr)
        return L32_ERR_NULL;
    return rope_kv_append_paged(q, k_new, v_new, reinterpret_cast<const long long*>(position_ids), pool_k, pool_v, block_table,
                                past_lens, new_lens, batch, q_len, heads, kv_heads, head_dim, max_pages_per_seq, rope_base, dtype,
                                as_stream(stream));
}

int l32_gqa_attention_forward_paged(const void* q, const void* pool_k, const void* pool_v, const int32_t* block_table,
                                    const int32_t* past_lens, const int32_t* new_lens, void* ctx, void* workspace, size_t workspace_bytes,
                                    int batch, int q_len, int heads, int kv_heads, int head_dim, int num_pages, int max_pages_per_seq,
                                    int max_kv_len, int dtype, void* stream) {
    bool run;
    const int rc = paged_forward_check(dtype, true, true, q, pool_k, pool_v, block_table, past_lens, ctx, workspace, batch, q_len,
                                       heads, kv_heads, head_dim, num_pages, max_pages_per_seq, max_kv_len, &run);
    if (!run) return rc;
    return gqa_attention_paged(q, pool_k, pool_v, block_table, past_lens, new_lens, ctx, workspace, workspace_bytes, batch, q_len, heads,
                               kv_heads, head_dim, num_pages, max_pages_per_seq, max_kv_len, dtype, as_stream(stream));
}

static bool cascade_shape_ok(int batch, int heads, int kv_heads, int head_dim, int max_kv_len, int max_items) {
    return batch >= 0 && attention_heads_ok(heads, kv_heads, head_dim) && heads / kv_heads >= 2 &&
           heads / kv_heads <= L32_CASCADE_TILE_ROWS && max_kv_len >= 0 && max_items > 0 && max_items <= L32_CASCADE_MAX_ITEMS;
}

size_t l32_gqa_attention_cascade_workspace_bytes(int batch, int heads, int kv_heads, int head_dim, int max_kv_len, int max_items) {
    if (!cascade_shape_ok(batch, heads, kv_heads, head_dim, max_kv_len, max_items) || batch == 0) return 0;
    return gqa_attention_cascade_workspace_bytes(batch, heads, kv_heads, head_dim, max_kv_len, max_items);
}

int l32_gqa_attention_forward_paged_cascade(const void* q, const void* pool_k, const void* pool_v, const int32_t* block_table,
                                            const int32_t* past_lens, const int32_t* new_lens, const int32_t* plan_items,
                                            const int32_t* plan_members, const int32_t* plan_seq, void* ctx, void* workspace,
                                            size_t workspace_bytes, int batch, int heads, int kv_heads, int head_dim, int num_pages,
                                            int max_pages_per_seq, int max_kv_len, int max_items, int dtype, void* stream) {
    const bool plan_ok = plan_items != nullptr && plan_members != nullptr && plan_seq != nullptr && workspace != nullptr;
    bool run;
    const int rc = paged_forward_check(dtype, cascade_shape_ok(batch, heads, kv_heads, head_dim, max_kv_len, max_items), plan_ok, q,
                                       pool_k, pool_v, block_table, past_lens, ctx, workspace, batch, 1, heads, kv_heads, head_dim,
                                       num_pages, max_pages_per_seq, max_kv_len, &run);
    if (!run) return rc;
    if (workspace_bytes < gqa_attention_cascade_workspace_bytes(batch, heads, kv_heads, head_dim, max_kv_len, max_items))
        return L32_ERR_WORKSPACE;
    return gqa_attention_paged_cascade(q, pool_k, pool_v, block_table, past_lens, new_lens, plan_items, plan_members, plan_seq,
                                       max_items, ctx, workspace, batch, heads, kv_heads, head_dim, num_pages, max_pages_per_seq,
                                       max_kv_len, dtype, as_stream(stream));
}

// Speculative decoding: the verify step's attention, n-gram drafts and acceptance (include/l32_ffn.h).  The tables, lengths and
// token values in device memory are trusted, as for the paged cache.
static bool verify_shape_ok(int batch, int q_len, int heads, int kv_heads, int head_dim) {
    return batch >= 0 && q_len >= 0 && attention_heads_ok(heads, kv_heads, head_dim) && heads / kv_heads >= 2 &&
           static_cast<long long>(heads / kv_heads) * q_len <= L32_VERIFY_TILE_ROWS;
}

size_t l32_gqa_attention_verify_workspace_bytes(int batch, int q_len, int heads, int kv_heads, int head_dim, int max_kv_len) {
    if (!verify_shape_ok(batch, q_len, heads, kv_heads, head_dim) || max_kv_len < 0 || batch == 0 || q_len == 0) return 0;
    return gqa_attention_verify_workspace_bytes(batch, q_len, heads, kv_heads, head_dim, max_kv_len);
}

int l32_gqa_attention_forward_paged_verify(const void* q, const void* pool_k, const void* pool_v, const int32_t* block_table,
                                           const int32_t* past_lens, const int32_t* new_lens, void* ctx, void* workspace,
                                           size_t workspace_bytes, int batch, int q_len, int heads, int kv_heads, int head_dim,
                                           int num_pages, int max_pages_per_seq, int max_kv_len, int dtype, void* stream) {
    bool run;
    const int rc = paged_forward_check(dtype, verify_shape_ok(batch, q_len, heads, kv_heads, head_dim), true, q, pool_k, pool_v,
                                       block_table, past_lens, ctx, workspace, batch, q_len, heads, kv_heads, head_dim, num_pages,
                                       max_pages_per_seq, max_kv_len, &run);
    if (!run) return rc;
    return gqa_attention_paged_verify(q, pool_k, pool_v, block_table, past_lens, new_lens, ctx, workspace, workspace_bytes, batch,
                                      q_len, heads, kv_heads, head_dim, num_pages, max_pages_per_seq, max_kv_len, dtype,
                                      as_stream(stream));
}

int l32_ngram_draft_paged(const int32_t* token_pool, const int32_t* block_table, const int32_t* past_lens, const int64_t* pending,
                          int64_t* ids, int32_t* draft_len, int batch, int k, int n_min, int n_max, int num_pages,
                          int max_pages_per_seq, void* stream) {
    if (batch < 0 || k < 1 || n_min < 1 || n_max < n_min || n_max > L32_NGRAM_MAX || num_pages <= 0 || max_pages_per_seq <= 0 ||
        static_cast<long long>(max_pages_per_seq) * L32_KV_PAGE > 0x7fffffffll)
        return L32_ERR_BAD_SHAPE;
    if (batch == 0) return L32_OK;
    if (token_pool == nullptr || block_table == nullptr || past_lens == nullptr || pending == nullptr || ids == nullptr)
        return L32_ERR_NULL;
    return ngram_draft_paged(token_pool, block_table, past_lens, reinterpret_cast<const long long*>(pending),
                             reinterpret_cast<long long*>(ids), draft_len, batch, k, n_min, n_max, max_pages_per_seq, as_stream(stream));
}

int l32_speculative_accept(const int64_t* ids, const int64_t* sampled, int32_t* token_pool, const int32_t* block_table,
                           const int32_t* past_lens, const int32_t* new_lens, int64_t* out, int batch, int width, int num_pages,
                           int max_pages_per_seq, void* stream) {
    if (batch < 0 || width < 1 || num_pages <= 0 || max_pages_per_seq <= 0 ||
        static_cast<long long>(max_pages_per_seq) * L32_KV_PAGE > 0x7fffffffll)
        return L32_ERR_BAD_SHAPE;
    if (batch == 0) return L32_OK;
    if (ids == nullptr || token_pool == nullptr || block_table == nullptr || past_lens == nullptr || new_lens == nullptr)
        return L32_ERR_NULL;
    return speculative_accept(reinterpret_cast<const long long*>(ids), reinterpret_cast<const long long*>(sampled), token_pool,
                              block_table, past_lens, new_lens, reinterpret_cast<long long*>(out), batch, width, max_pages_per_seq,
                              as_stream(stream));
}

// Next-token sampling (no reference kernel: the reference's decode loop samples with torch, Inference/Inference.py
// select_next_token).  The per-row parameters live in device memory and are trusted, like the paged cache's tables.
int l32_sample_tokens(const void* logits, const float* temperature, const int32_t* top_k, const float* top_p, const uint64_t* seed,
                      const int64_t* position, int64_t* tokens_out, float* kept_min_logit, int batch, int vocab, int dtype,
                      void* stream) {
    if (!dtype_ok(dtype)) return L32_ERR_BAD_DTYPE;
    if (batch < 0 || vocab < 8 || vocab > L32_SAMPLE_MAX_VOCAB || (vocab % 8) != 0) return L32_ERR_BAD_SHAPE;
    if (batch == 0) return L32_OK;
    if (logits == nullptr || temperature == nullptr || top_k == nullptr || top_p == nullptr || seed == nullptr ||
        position == nullptr || tokens_out == nullptr)
        return L32_ERR_NULL;
    if (!is_aligned16(logits)) return L32_ERR_BAD_ALIGN;
    return sample_tokens(logits, temperature, top_k, top_p, reinterpret_cast<const unsigned long long*>(seed),
                         reinterpret_cast<const long long*>(position), reinterpret_cast<long long*>(tokens_out), kept_min_logit,
                         batch, vocab, dtype, as_stream(stream));
}

int l32_gemm(const void* a, int64_t lda, int a_mn_major, const void* b, int64_t ldb, int b_mn_major, const void* a1,
             int64_t lda1, const void* b1, int64_t ldb1, void* d, int64_t ldd, int m, int n, int k, int k1, int dtype,
             int cta_group, int max_ctas, void* stream) {
    if (!dtype_ok(dtype)) return L32_ERR_BAD_DTYPE;
    if (a == nullptr || b == nullptr || d == nullptr) return L32_ERR_NULL;
    GemmProblem g = blank(m, n, dtype);
    g.k[0] = k;
    g.a[0] = op(a, lda, a_mn_major);
    g.b[0] = op(b, ldb, b_mn_major);
    if (a1 != nullptr) {
        if (b1 == nullptr) return L32_ERR_NULL;
        g.num_phases = 2;
        g.k[1] = k1;
        g.a[1] = op(a1, lda1, a_mn_major);
        g.b[1] = op(b1, ldb1, b_mn_major);
    }
    g.epilogue = EPI_STORE;
    g.d[0] = d;
    g.ldd = ldd;
    g.cta_group = cta_group;
    g.max_ctas = max_ctas;
    return gemm_sm100(g, as_stream(stream));
}

int l32_tp_signal(void* const* peer_flags, int world, int index, uint32_t value, uint32_t* zero8, void* stream) {
    if (peer_flags == nullptr) return L32_ERR_NULL;
    if (world < 1 || world > kMaxTpWorld || index < 0) return L32_ERR_BAD_SHAPE;
    for (int i = 0; i < world; ++i)
        if (peer_flags[i] == nullptr) return L32_ERR_NULL;
    return static_cast<int>(tp_signal(peer_flags, world, index, value, zero8, as_stream(stream)));
}

int l32_tp_peer_copy(void* dst, const void* src, size_t bytes, int ctas, int warps, int unroll, int seg_bytes, void* stream) {
    if (dst == nullptr || src == nullptr) return L32_ERR_NULL;
    if (!is_aligned16(dst) || !is_aligned16(src) || (bytes % 16) != 0) return L32_ERR_BAD_ALIGN;
    if (ctas < 1 || warps < 1 || warps > 32) return L32_ERR_BAD_SHAPE;
    if (seg_bytes != 0 && (seg_bytes < 16 || seg_bytes > 8192 || (8192 % seg_bytes) != 0 || (bytes % 8192) != 0)) return L32_ERR_BAD_SHAPE;
    return static_cast<int>(tp_peer_copy(dst, src, bytes, ctas, warps, unroll, seg_bytes, as_stream(stream)));
}

namespace {
bool tp_args_ok(int rank, int world, int64_t rows_per_rank, int64_t tokens) {
    return world >= 1 && world <= kMaxTpWorld && rank >= 0 && rank < world && rows_per_rank > 0 &&
           rows_per_rank * world >= tokens && rows_per_rank <= 0x7fffffff;
}

// All-gather of the A operand fused into the GEMM `g` (g.a[0] = a_full must already be set).  Clears the arrival
// counters on the stream.  When a_full is not the buffer the peers pull from (peer_a[rank]) the own rows are copied in
// by the pullers as well, so a_full may be a fresh tensor the caller keeps (e.g. saved for the backward).
int setup_allgather(GemmProblem& g, void* a_full, const void* const* peer_a, const uint32_t* ready, uint32_t* done,
                    uint32_t epoch, int rank, int world, int64_t rows_per_rank, cudaStream_t s) {
    if (world <= 1) {
        if (peer_a != nullptr && peer_a[0] != nullptr && peer_a[0] != a_full) return L32_ERR_BAD_SHAPE;   // nothing would copy the rows
        return L32_OK;
    }
    if (peer_a == nullptr || ready == nullptr || done == nullptr) return L32_ERR_NULL;
    // arrival counters of the pull: cleared here so that a call never sees the counts of an earlier one
    cudaError_t e = cudaMemsetAsync(done, 0, sizeof(uint32_t) * kMaxTpWorld, s);
    if (e != cudaSuccess) return static_cast<int>(e);
    g.ag.world = world;
    g.ag.rank = rank;
    g.ag.rows_per_rank = static_cast<int>(rows_per_rank);
    for (int r = 0; r < world; ++r) {
        if (peer_a[r] == nullptr || !is_aligned16(peer_a[r])) return L32_ERR_NULL;
        g.ag.peer_src[r] = peer_a[r];
    }
    g.ag.local_dst = a_full;
    g.ag.ready = ready;
    g.ag.done = done;
    g.ag.epoch = epoch;
    g.ag.done_base = 0;
    g.ag.copy_own = (peer_a[rank] != a_full) ? 1 : 0;
    g.m_rotate_rows = static_cast<int>(rank * rows_per_rank);
    // one raster group = the m-tiles of one rank's chunk, so tiles only ever wait for the chunk being consumed
    const int tile_m = 256;
    int grp = static_cast<int>(rows_per_rank / tile_m);
    if (grp < 1) grp = 1;
    if (grp > 8) grp = 8;
    g.raster_group = grp;
    return L32_OK;
}

int setup_reduce_scatter(GemmProblem& g, void* const* peer_slots, int rank, int world, int64_t rows_per_rank, int64_t tokens) {
    if (peer_slots == nullptr) return L32_ERR_NULL;
    g.rs.world = world;
    g.rs.rank = rank;
    g.rs.rows_per_rank = static_cast<int>(rows_per_rank);
    for (int o = 0; o < world; ++o) {
        if (peer_slots[o] == nullptr || !is_aligned16(peer_slots[o])) return L32_ERR_NULL;
        g.rs.peer_dst[o] = peer_slots[o];
    }
    // start with the rows owned by the next rank so that at any moment the ranks push to different owners
    g.m_rotate_rows = static_cast<int>(((rank + 1) % world) * rows_per_rank);
    if (g.m_rotate_rows >= tokens) g.m_rotate_rows = 0;
    return L32_OK;
}
}  // namespace

int l32_tp_swiglu_forward_allgather(void* x_full, const void* const* peer_x, const uint32_t* ready, uint32_t* done,
                                    uint32_t epoch, int rank, int world, int64_t rows_per_rank, const void* w_gate,
                                    const void* w_up, const void* b_gate, const void* b_up, void* act, void* gate_cache,
                                    void* up_cache, int64_t tokens, int hidden, int inter_local, int dtype, void* stream) {
    if (!dtype_ok(dtype)) return L32_ERR_BAD_DTYPE;
    if (!shapes_ok(tokens, hidden, inter_local)) return L32_ERR_BAD_SHAPE;
    if (world < 1 || world > kMaxTpWorld || rank < 0 || rank >= world || rows_per_rank <= 0 ||
        rows_per_rank * world < tokens || rows_per_rank > 0x7fffffff)
        return L32_ERR_BAD_SHAPE;
    if (tokens == 0) return L32_OK;
    if (x_full == nullptr || w_gate == nullptr || w_up == nullptr || act == nullptr) return L32_ERR_NULL;
    if ((gate_cache == nullptr) != (up_cache == nullptr)) return L32_ERR_NULL;
    GemmProblem g = blank(static_cast<int>(tokens), inter_local, dtype);
    g.k[0] = hidden;
    g.a[0] = op(x_full, hidden, 0);
    g.b[0] = op(w_gate, hidden, 0);
    g.b[1] = op(w_up, hidden, 0);
    g.epilogue = EPI_SWIGLU;
    g.d[0] = act;
    g.d[1] = gate_cache;
    g.d[2] = up_cache;
    g.bias[0] = b_gate;
    g.bias[1] = b_up;
    g.ldd = inter_local;
    g.cta_group = 2;
    const int rc = setup_allgather(g, x_full, peer_x, ready, done, epoch, rank, world, rows_per_rank, as_stream(stream));
    if (rc != L32_OK) return rc;
    return gemm_sm100(g, as_stream(stream));
}

int l32_tp_linear_forward_reduce_scatter(const void* a, const void* w, void* const* peer_slots, int rank, int world,
                                         int64_t rows_per_rank, int64_t tokens, int in_local, int out_features, int dtype,
                                         void* stream) {
    if (!dtype_ok(dtype)) return L32_ERR_BAD_DTYPE;
    if (!shapes_ok(tokens, in_local, out_features)) return L32_ERR_BAD_SHAPE;
    if (world < 1 || world > kMaxTpWorld || rank < 0 || rank >= world || rows_per_rank <= 0 ||
        rows_per_rank * world < tokens || rows_per_rank > 0x7fffffff)
        return L32_ERR_BAD_SHAPE;
    if (tokens == 0) return L32_OK;
    if (a == nullptr || w == nullptr || peer_slots == nullptr) return L32_ERR_NULL;
    GemmProblem g = blank(static_cast<int>(tokens), out_features, dtype);
    g.k[0] = in_local;
    g.a[0] = op(a, in_local, 0);
    g.b[0] = op(w, in_local, 0);
    g.epilogue = EPI_STORE;
    g.ldd = out_features;
    g.cta_group = 2;
    const int rc = setup_reduce_scatter(g, peer_slots, rank, world, rows_per_rank, tokens);
    if (rc != L32_OK) return rc;
    return gemm_sm100(g, as_stream(stream));
}

/* ---- tensor-parallel backward: d_act GEMM with the all-gather of dY pulled in, dX GEMM with the reduce-scatter pushed out */
int l32_tp_ffn_backward_dact_allgather(void* dy_full, const void* const* peer_dy, const uint32_t* ready, uint32_t* done,
                                       uint32_t epoch, int rank, int world, int64_t rows_per_rank, const void* w_down,
                                       const void* gate_cache, const void* up_cache, void* d_gate, void* d_up, void* act_out,
                                       int64_t tokens, int hidden, int inter_local, int dtype, void* stream) {
    if (!dtype_ok(dtype)) return L32_ERR_BAD_DTYPE;
    if (!shapes_ok(tokens, hidden, inter_local) || !tp_args_ok(rank, world, rows_per_rank, tokens)) return L32_ERR_BAD_SHAPE;
    if (tokens == 0) return L32_OK;
    if (dy_full == nullptr || w_down == nullptr || gate_cache == nullptr || up_cache == nullptr || d_gate == nullptr ||
        d_up == nullptr)
        return L32_ERR_NULL;
    // d_act = dy w_down_shard (w_down_shard [hidden, inter_local] consumed MN-major); SiLU' recomputed in the epilogue
    GemmProblem g = blank(static_cast<int>(tokens), inter_local, dtype);
    g.k[0] = hidden;
    g.a[0] = op(dy_full, hidden, 0);
    g.b[0] = op(w_down, inter_local, 1);
    g.epilogue = EPI_SWIGLU_BWD;
    g.d[0] = d_gate;
    g.d[1] = d_up;
    g.d[2] = act_out;
    g.e[0] = gate_cache;
    g.e[1] = up_cache;
    g.ldd = inter_local;
    g.cta_group = 2;
    const int rc = setup_allgather(g, dy_full, peer_dy, ready, done, epoch, rank, world, rows_per_rank, as_stream(stream));
    if (rc != L32_OK) return rc;
    return gemm_sm100(g, as_stream(stream));
}

int l32_tp_ffn_backward_dx_reduce_scatter(const void* d_gate, const void* d_up, const void* w_gate, const void* w_up,
                                          void* const* peer_slots, int rank, int world, int64_t rows_per_rank, int64_t tokens,
                                          int hidden, int inter_local, int dtype, void* stream) {
    if (!dtype_ok(dtype)) return L32_ERR_BAD_DTYPE;
    if (!shapes_ok(tokens, hidden, inter_local) || !tp_args_ok(rank, world, rows_per_rank, tokens)) return L32_ERR_BAD_SHAPE;
    if (tokens == 0) return L32_OK;
    if (d_gate == nullptr || d_up == nullptr || w_gate == nullptr || w_up == nullptr) return L32_ERR_NULL;
    // partial dx = d_gate w_gate_shard + d_up w_up_shard: one two-phase GEMM, rows pushed to their owners' slots
    GemmProblem g = blank(static_cast<int>(tokens), hidden, dtype);
    g.num_phases = 2;
    g.k[0] = g.k[1] = inter_local;
    g.a[0] = op(d_gate, inter_local, 0);
    g.a[1] = op(d_up, inter_local, 0);
    g.b[0] = op(w_gate, hidden, 1);
    g.b[1] = op(w_up, hidden, 1);
    g.epilogue = EPI_STORE;
    g.ldd = hidden;
    g.cta_group = 2;
    const int rc = setup_reduce_scatter(g, peer_slots, rank, world, rows_per_rank, tokens);
    if (rc != L32_OK) return rc;
    return gemm_sm100(g, as_stream(stream));
}

/* ---- tensor-parallel attention: q/k/v of the shard with the all-gather pulled in, the backward's three-phase dX pushed out */
int l32_tp_linear_group_forward_allgather(void* x_full, const void* const* peer_x, const uint32_t* ready, uint32_t* done,
                                          uint32_t epoch, int rank, int world, int64_t rows_per_rank, const void* const* w,
                                          void* const* y, const int* out_features, int count, int64_t tokens, int in_features,
                                          int dtype, void* stream) {
    if (!dtype_ok(dtype)) return L32_ERR_BAD_DTYPE;
    if (count < 1 || count > 3 || !tp_args_ok(rank, world, rows_per_rank, tokens)) return L32_ERR_BAD_SHAPE;
    if (w == nullptr || y == nullptr || out_features == nullptr) return L32_ERR_NULL;
    for (int i = 0; i < count; ++i) {
        if (!shapes_ok(tokens, in_features, out_features[i])) return L32_ERR_BAD_SHAPE;
        if (w[i] == nullptr || y[i] == nullptr) return L32_ERR_NULL;
    }
    if (tokens == 0) return L32_OK;
    if (x_full == nullptr) return L32_ERR_NULL;
    cudaStream_t s = as_stream(stream);
    GemmProblem g = blank(static_cast<int>(tokens), out_features[0], dtype);
    g.k[0] = in_features;
    g.a[0] = op(x_full, in_features, 0);
    g.b[0] = op(w[0], in_features, 0);
    g.epilogue = EPI_STORE;
    g.d[0] = y[0];
    g.ldd = out_features[0];
    g.cta_group = 2;
    if (count > 1) {
        g.group_count = count;
        for (int i = 0; i < count; ++i) {
            GroupMember& q = g.group[i];
            q.a = x_full; q.lda = in_features; q.m = static_cast<int>(tokens);
            q.b = w[i]; q.ldb = in_features; q.n = out_features[i];
            q.d = y[i]; q.ldd = out_features[i];
        }
    }
    const int rc = setup_allgather(g, x_full, peer_x, ready, done, epoch, rank, world, rows_per_rank, s);
    if (rc != L32_OK) return rc;
    return gemm_sm100(g, s);
}

int l32_tp_linear_forward_allgather(void* a_full, const void* const* peer_a, const uint32_t* ready, uint32_t* done,
                                    uint32_t epoch, int rank, int world, int64_t rows_per_rank, const void* w, int w_mn_major,
                                    void* y, int64_t tokens, int in_features, int out_features, int dtype, void* stream) {
    if (!dtype_ok(dtype)) return L32_ERR_BAD_DTYPE;
    if (!shapes_ok(tokens, in_features, out_features) || !tp_args_ok(rank, world, rows_per_rank, tokens) ||
        (w_mn_major != 0 && w_mn_major != 1))
        return L32_ERR_BAD_SHAPE;
    if (tokens == 0) return L32_OK;
    if (a_full == nullptr || w == nullptr || y == nullptr) return L32_ERR_NULL;
    cudaStream_t s = as_stream(stream);
    GemmProblem g = blank(static_cast<int>(tokens), out_features, dtype);
    g.k[0] = in_features;
    g.a[0] = op(a_full, in_features, 0);
    g.b[0] = op(w, w_mn_major ? out_features : in_features, w_mn_major);
    g.epilogue = EPI_STORE;
    g.d[0] = y;
    g.ldd = out_features;
    g.cta_group = 2;
    const int rc = setup_allgather(g, a_full, peer_a, ready, done, epoch, rank, world, rows_per_rank, s);
    if (rc != L32_OK) return rc;
    return gemm_sm100(g, s);
}

int l32_tp_linear_group_backward_dx_reduce_scatter(const void* const* dy, const void* const* w, const int* k, int num_phases,
                                                   void* const* peer_slots, int rank, int world, int64_t rows_per_rank,
                                                   int64_t tokens, int hidden, int dtype, void* stream) {
    if (!dtype_ok(dtype)) return L32_ERR_BAD_DTYPE;
    if (num_phases < 1 || num_phases > 3 || !tp_args_ok(rank, world, rows_per_rank, tokens)) return L32_ERR_BAD_SHAPE;
    if (k == nullptr) return L32_ERR_NULL;
    for (int i = 0; i < num_phases; ++i)
        if (!shapes_ok(tokens, hidden, k[i])) return L32_ERR_BAD_SHAPE;
    if (tokens == 0) return L32_OK;
    if (dy == nullptr || w == nullptr) return L32_ERR_NULL;
    for (int i = 0; i < num_phases; ++i)
        if (dy[i] == nullptr || w[i] == nullptr) return L32_ERR_NULL;
    // partial dx = sum_i dy_i w_i (w_i [k_i, hidden] consumed MN-major): one GEMM, rows pushed to their owners' slots
    GemmProblem g = blank(static_cast<int>(tokens), hidden, dtype);
    g.num_phases = num_phases;
    for (int i = 0; i < num_phases; ++i) {
        g.k[i] = k[i];
        g.a[i] = op(dy[i], k[i], 0);
        g.b[i] = op(w[i], hidden, 1);
    }
    g.epilogue = EPI_STORE;
    g.ldd = hidden;
    g.cta_group = 2;
    const int rc = setup_reduce_scatter(g, peer_slots, rank, world, rows_per_rank, tokens);
    if (rc != L32_OK) return rc;
    return gemm_sm100(g, as_stream(stream));
}

int l32_tp_ffn_forward_fused(void* x_full, const void* const* peer_x, const uint32_t* ready, uint32_t* done, uint32_t epoch,
                             int rank, int world, int64_t rows_per_rank, const void* w_gate, const void* w_up,
                             const void* w_down, void* act_ws, uint32_t* act_done, void* const* peer_slots, int64_t tokens,
                             int hidden, int inter_local, int dtype, void* stream) {
    if (!dtype_ok(dtype)) return L32_ERR_BAD_DTYPE;
    if (!shapes_ok(tokens, hidden, inter_local)) return L32_ERR_BAD_SHAPE;
    if (world < 1 || world > kMaxTpWorld || rank < 0 || rank >= world || rows_per_rank <= 0 ||
        rows_per_rank * world < tokens || rows_per_rank > 0x7fffffff)
        return L32_ERR_BAD_SHAPE;
    if (tokens == 0) return L32_OK;
    if (x_full == nullptr || w_gate == nullptr || w_up == nullptr || w_down == nullptr || act_ws == nullptr ||
        act_done == nullptr || peer_slots == nullptr)
        return L32_ERR_NULL;
    cudaStream_t s = as_stream(stream);
    const int tile_m = 256;
    const int tiles_m = static_cast<int>((tokens + tile_m - 1) / tile_m);
    cudaError_t e = cudaMemsetAsync(act_done, 0, sizeof(uint32_t) * static_cast<size_t>(tiles_m), s);
    if (e != cudaSuccess) return static_cast<int>(e);
    GemmProblem g = blank(static_cast<int>(tokens), inter_local, dtype);
    g.k[0] = hidden;
    g.a[0] = op(x_full, hidden, 0);
    g.b[0] = op(w_gate, hidden, 0);
    g.b[1] = op(w_up, hidden, 0);
    g.epilogue = EPI_FFN_TP;
    g.d[0] = act_ws;
    g.ldd = inter_local;
    g.cta_group = 2;
    g.dn.w = w_down;
    g.dn.ld = inter_local;
    g.dn.n = hidden;
    g.dn.act_done = act_done;
    int rc = setup_reduce_scatter(g, peer_slots, rank, world, rows_per_rank, tokens);
    if (rc != L32_OK) return rc;
    int grp = static_cast<int>(rows_per_rank / tile_m);
    if (grp < 1) grp = 1;
    if (grp > 8) grp = 8;
    if (world > 1) {
        if (peer_x == nullptr || peer_x[rank] != x_full) return L32_ERR_BAD_SHAPE;   // this variant gathers in place
        rc = setup_allgather(g, x_full, peer_x, ready, done, epoch, rank, world, rows_per_rank, s);
        if (rc != L32_OK) return rc;
    }
    g.raster_group = grp;   // one group of m-tiles = (a divisor of) one rank's chunk: pulls, math and pushes move in step
    g.m_rotate_rows = static_cast<int>(rank * rows_per_rank);
    return gemm_sm100(g, s);
}

int l32_tp_reduce_partials(const void* slots, const uint32_t* flags, uint32_t epoch, int world, int rank, const void* addend,
                           void* y, int64_t rows, int64_t slot_rows, int hidden, int dtype, void* stream) {
    if (!dtype_ok(dtype)) return L32_ERR_BAD_DTYPE;
    if (world < 1 || world > kMaxTpWorld || rank < 0 || rank >= world || rows < 0 || slot_rows < rows || hidden <= 0 ||
        (hidden % 8) != 0)
        return L32_ERR_BAD_SHAPE;
    if (rows == 0) return L32_OK;
    if (slots == nullptr || y == nullptr || (world > 1 && flags == nullptr)) return L32_ERR_NULL;
    if (!is_aligned16(slots) || !is_aligned16(y) || !is_aligned16(addend)) return L32_ERR_BAD_ALIGN;
    return static_cast<int>(tp_reduce_partials(slots, flags, epoch, world, rank, addend, y, rows, slot_rows, hidden, dtype,
                                               as_stream(stream)));
}

int l32_debug_tile_order(int kind, int t, const int* cfg, int* out3) {
    if (cfg == nullptr || out3 == nullptr) return L32_ERR_NULL;
    if (kind == 0) debug_tile_order(t, cfg[0], cfg[1], cfg[2], cfg[3], cfg[4], cfg[5], cfg[6], out3);
    else if (kind == 1) debug_ffn_tile_order(t, cfg[0], cfg[1], cfg[2], cfg[3], cfg[4], cfg[5], out3);
    else return L32_ERR_BAD_SHAPE;
    return L32_OK;
}

int l32_debug_gemm_plan(int epilogue, int m, int n, int cta_group, int max_ctas, int num_sms, int* out) {
    if (out == nullptr) return L32_ERR_NULL;
    if (epilogue != EPI_STORE && epilogue != EPI_SWIGLU && epilogue != EPI_SWIGLU_BWD && epilogue != EPI_CE) return L32_ERR_BAD_SHAPE;
    return debug_gemm_plan(epilogue, m, n, cta_group, max_ctas, num_sms, out);
}

int l32_swiglu_act(const void* gate, const void* up, void* act, int64_t n, int dtype, void* stream) {
    if (!dtype_ok(dtype)) return L32_ERR_BAD_DTYPE;
    if (n < 0 || (n % 8) != 0) return L32_ERR_BAD_SHAPE;
    if (n > 0 && (gate == nullptr || up == nullptr || act == nullptr)) return L32_ERR_NULL;
    return static_cast<int>(swiglu_act_elementwise(gate, up, act, n, dtype, as_stream(stream)));
}

}  // extern "C"
