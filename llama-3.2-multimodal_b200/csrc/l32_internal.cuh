// Internal declarations shared by the kernel translation units and the C-ABI layer (api.cu).
#pragma once
#include "ptx_sm100.cuh"
#include "../../include/l32_ffn.h"   // L32_OK / L32_ERR_* return codes
#include <cstddef>

namespace l32 {

enum : int { L32_BF16 = 0, L32_FP16 = 1 };

// Process-wide count of kernels this library has launched (reported by bench.py as `gpu_launches`).
void count_launch(int n = 1);
unsigned long long launch_count();

inline bool is_aligned16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15u) == 0; }
int num_sms();   // of the current device
// Bound of every spin on a flag raised by another SM / GPU, after which the kernel traps (L32_TP_TIMEOUT_S, default 120 s).
uint64_t spin_timeout_ns();
// Kernel attributes (opt-in shared memory size) are per device: one "already configured" flag per device ordinal.
constexpr int kMaxDevices = 64;
inline int current_device_slot() {
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= kMaxDevices) return 0;
    return dev;
}

// ---- rmsnorm.cu
cudaError_t add_rmsnorm_fwd(const void* x, const void* residual, const void* weight, void* y, void* h_out, float* rms,
                            int64_t rows, int C, float eps, int dtype, cudaStream_t s);
cudaError_t rmsnorm_bwd(const void* dy, const void* h, const void* weight, const float* rms, const void* addend, void* dx,
                        void* dx_plain, void* dw, float* workspace, int64_t rows, int C, int dtype,
                        cudaStream_t s);   // dx = norm backward (+ addend); dx_plain: optional, the norm backward without it
size_t rmsnorm_bwd_workspace_bytes(int64_t rows, int C);

// ---- gemm_sm100.cu : D[M,N] = sum_p A_p[M,K_p] * B_p[N,K_p]^T on tcgen05, fused epilogues
enum : int {
    EPI_STORE = 0,       // D -> d[0]                                     (tile 128*cta_group x 256)
    EPI_SWIGLU = 1,      // b[0]=gate weights, b[1]=up weights; act = silu(g)*u -> d[0]; optional g -> d[1], u -> d[2]
    EPI_SWIGLU_BWD = 2,  // D = d_act; e[0]=gate cache, e[1]=up cache; d_gate -> d[0], d_up -> d[1], optional act -> d[2]
    EPI_CE = 4,          // EPI_STORE (logits -> d[0]) + per-row, per-column-tile softmax statistics and the target logit
                         // (GemmProblem::ce): lm_head + cross entropy without a second pass over the logits
    EPI_FFN_TP = 3,      // tensor-parallel feed-forward in ONE kernel: the EPI_SWIGLU problem (act -> d[0]) and the down
                         // projection of that act (GemmProblem::dn, reduce-scatter epilogue) share the persistent tile loop,
                         // the down tiles of one group of rows interleaved with the gate/up tiles of the next group
};

struct GemmOperand {
    const void* ptr;   // base pointer (16-byte aligned)
    int64_t ld;        // row pitch in elements (multiple of 8)
    int mn_major;      // 0: memory is [rows = M or N][cols = K]  (K contiguous)
                       // 1: memory is [rows = K][cols = M or N]  (M/N contiguous)
};

constexpr int kMaxTpWorld = 8;

// Tensor-parallel extensions of the tiled GEMM (both optional, world == 0 disables):
//  * all-gather fused into the A operand: the rows of A owned by other ranks are PULLED from peer memory by the
//    otherwise idle warps of every CTA, chunk by chunk in the order the tiles consume them, while the tensor cores
//    work on the chunks that have already arrived;
//  * reduce-scatter fused into the epilogue: each output row is stored straight into the buffer of the rank that
//    owns it (peer stores over NVLink), slot [this rank]; the owner sums the slots.
struct TpAllGather {
    int world, rank;
    int rows_per_rank;              // A rows owned by each rank (last rank may own fewer: rows beyond m are ignored)
    const void* peer_src[kMaxTpWorld];   // peer_src[s]: base of rank s's full-size A buffer (only its own rows are valid)
    void* local_dst;                // this rank's full-size A buffer (the GEMM's A operand)
    const uint32_t* ready;          // local flags, ready[s] >= epoch once rank s's own rows are final
    uint32_t* done;                 // local counters, done[s] += 1 per puller warp that finished chunk s
    uint32_t epoch;                 // step number (monotonic, >= 1)
    uint32_t done_base;             // value of every done[s] before this launch
    int copy_own;                   // 1: local_dst is not the buffer the peers pull from -- the own rows are copied in too
};
struct TpReduceScatter {
    int world, rank;
    int rows_per_rank;              // output rows owned by each rank
    void* peer_dst[kMaxTpWorld];    // peer_dst[o]: rank o's slot for THIS rank's partial, [rows_per_rank, ldd]
};

// Second problem of EPI_FFN_TP: y_partial[m, n] = act[m, k = GemmProblem::n] * w[n, k]^T, rows scattered by GemmProblem::rs.
struct TpFfnDown {
    const void* w;          // this rank's w_down shard [n, k], K-major (null: not an EPI_FFN_TP problem)
    int64_t ld;             // its row pitch, elements
    int n;                  // output columns (hidden size)
    uint32_t* act_done;     // [ceil(m / 256)] arrival counters, ZERO on entry: epilogue warps that finished act tiles
};

// EPI_CE: lm_head + cross entropy.  partials: [m][ceil(n / 256)] float2 (max, sum exp(v - max)); target: [m] floats.
struct CeOutputs {
    const long long* labels;   // [m] int64 target column per row (out-of-range = no target, e.g. ignore_index)
    void* partials;
    float* target;
};

// One problem of a grouped launch: D[m, n] = A B^T with the group's common K, majors and dtype (GemmProblem::group).
struct GroupMember {
    const void* a;   // K-major: [m, k] (pitch lda);  MN-major: [k, m]
    const void* b;   // K-major: [n, k] (pitch ldb);  MN-major: [k, n]
    void* d;         // [m, n], pitch ldd
    int64_t lda, ldb, ldd;
    int m, n;
};

struct GemmProblem {
    int m, n;               // D is [m, n]; for EPI_SWIGLU n = intermediate size (act columns)
    int num_phases;         // 1 to 3: D = sum_p A_p*B_p^T (EPI_SWIGLU: must be 1)
    int k[3];               // reduction length of each phase
    GemmOperand a[3];       // a[p] used when p < num_phases
    GemmOperand b[3];       // EPI_SWIGLU: b[0] = gate weights, b[1] = up weights (both K-major)
    int epilogue;           // EPI_*
    void* d[3];             // outputs, see EPI_*; optional ones may be null
    const void* e[2];       // EPI_SWIGLU_BWD: gate / up caches [m, n];  EPI_STORE: e[0] = optional addend [m, n] (D += addend)
    int64_t ldd;            // row pitch of every output / epilogue input, elements
    const void* bias[2];    // optional per-column bias (bias[0] for D / gate, bias[1] for up)
    int dtype;              // L32_BF16 / L32_FP16
    int cta_group;          // 0 = auto, 1 or 2
    int raster_group;       // 0 = auto: m-tiles per raster group
    int max_ctas;           // 0 = all SMs (testing / tuning knob)
    int m_rotate_rows;      // visit the m-tiles starting at this row (rounded down to a tile), wrapping around
    TpAllGather ag;         // ag.world == 0: off
    TpReduceScatter rs;     // rs.world == 0: off (EPI_STORE and the down half of EPI_FFN_TP)
    TpFfnDown dn;           // EPI_FFN_TP only
    CeOutputs ce;           // EPI_CE only
    int group_count;        // > 1: grouped launch (EPI_STORE, cta_group 2): `group` replaces m / n / a[].ptr / b[].ptr / d
    GroupMember group[3];   //      (k[0], a[0].mn_major, b[0].mn_major and dtype are shared; with `ag` every member
                            //      reads the same K-major A = a[0], [m, k[0]] with a dense pitch)
};
int gemm_sm100(const GemmProblem& p, cudaStream_t s);   // returns L32_* / cudaError_t
void debug_tile_order(int t, int tiles_m, int tiles_n, int group, int m_rotate, int il_world, int il_tpc, int il_rank, int* out3);
void debug_ffn_tile_order(int t, int tiles_m, int n_gu, int n_dn, int group, int m_rotate, int prefix, int* out3);
int debug_gemm_plan(int epilogue, int m, int n, int cta_group, int max_ctas, int sms, int* out7);

// ---- elementwise.cu (n = element count, multiple of 8)
cudaError_t swiglu_bwd_elementwise(const void* d_act, const void* gate, const void* up, void* d_gate, void* d_up,
                                   int64_t n, int dtype, cudaStream_t s);
cudaError_t swiglu_act_elementwise(const void* gate, const void* up, void* act, int64_t n, int dtype, cudaStream_t s);

// ---- ffn_decode.cu : weight-streaming small-M FFN (tokens <= 128)
//      return L32_ERR_BAD_SHAPE when the problem is outside the kernel's envelope (the caller then uses the tiled GEMM)
int ffn_decode_swiglu(const void* x, const void* w_gate, const void* w_up, const void* b_gate, const void* b_up, void* act,
                      void* gate_cache, void* up_cache, int tokens, int hidden, int inter, int dtype, cudaStream_t s);
int ffn_decode_linear(const void* a, const void* w, const void* bias, const void* addend, void* y, int tokens,
                      int in_features, int out_features, int dtype, cudaStream_t s);
//      up to three y_i = a w_i^T with the same a (e.g. the q / k / v projections of a decode step) as ONE launch
int ffn_decode_linear_group(const void* a, const void* const* w, void* const* y, const int* out_features, int count, int tokens,
                            int in_features, int dtype, cudaStream_t s);

// ---- lmhead.cu : cross-entropy reductions around the EPI_CE GEMM
cudaError_t ce_reduce(const void* partials, const float* target, const long long* labels, long long ignore_index, int64_t rows,
                      int tiles_n, int vocab, float* lse, float* loss_rows, float* loss_and_count, cudaStream_t s);
cudaError_t ce_backward_logits(const void* logits, const float* lse, const long long* labels, long long ignore_index,
                               const float* loss_and_count, const float* grad_loss, void* dlogits, int64_t rows, int vocab,
                               int dtype, cudaStream_t s);

// ---- attention.cu : RoPE + KV-cache append, flash-style GQA forward (head_dim 64 / 128)
int rope_kv_append(void* q, const void* k_new, const void* v_new, const long long* position_ids, void* cache_k, void* cache_v,
                   int batch, int q_len, int heads, int kv_heads, int head_dim, int max_len, int past_len, float rope_base,
                   int dtype, cudaStream_t s);
size_t gqa_attention_workspace_bytes(int batch, int q_len, int heads, int kv_heads, int head_dim, int kv_len);
int gqa_attention(const void* q, const void* cache_k, const void* cache_v, const uint8_t* keep, void* out, int batch, int q_len,
                  int heads, int kv_heads, int head_dim, int max_len, int kv_len, int past_len, int causal, void* workspace,
                  size_t workspace_bytes, int dtype, cudaStream_t s);
int gqa_attention_train(const void* q, const void* cache_k, const void* cache_v, const uint8_t* keep, void* out, float* lse, int batch,
                        int q_len, int heads, int kv_heads, int head_dim, int max_len, int causal, int dtype, cudaStream_t s);
// paged KV cache (pools [num_pages, kv_heads, L32_KV_PAGE, head_dim], block table, per-sequence lengths in device memory)
int rope_kv_append_paged(void* q, const void* k_new, const void* v_new, const long long* position_ids, void* pool_k, void* pool_v,
                         const int* block_table, const int* past_lens, const int* new_lens, int batch, int q_len, int heads,
                         int kv_heads, int head_dim, int max_pages_per_seq, float rope_base, int dtype, cudaStream_t s);
int gqa_attention_paged(const void* q, const void* pool_k, const void* pool_v, const int* block_table, const int* past_lens,
                        const int* new_lens, void* out, void* workspace, size_t workspace_bytes, int batch, int q_len, int heads,
                        int kv_heads, int head_dim, int num_pages, int max_pages_per_seq, int max_kv_len, int dtype, cudaStream_t s);
size_t gqa_attention_cascade_workspace_bytes(int batch, int heads, int kv_heads, int head_dim, int max_kv_len, int max_items);
int gqa_attention_paged_cascade(const void* q, const void* pool_k, const void* pool_v, const int* block_table, const int* past_lens,
                                const int* new_lens, const int* items, const int* members, const int* seq_plan, int max_items,
                                void* out, void* workspace, int batch, int heads, int kv_heads, int head_dim, int num_pages,
                                int max_pages_per_seq, int max_kv_len, int dtype, cudaStream_t s);
// speculative verify step: each sequence has up to q_len new tokens, group * q_len <= 128 rows in one query tile per kv head
size_t gqa_attention_verify_workspace_bytes(int batch, int q_len, int heads, int kv_heads, int head_dim, int max_kv_len);
int gqa_attention_paged_verify(const void* q, const void* pool_k, const void* pool_v, const int* block_table, const int* past_lens,
                               const int* new_lens, void* out, void* workspace, size_t workspace_bytes, int batch, int q_len, int heads,
                               int kv_heads, int head_dim, int num_pages, int max_pages_per_seq, int max_kv_len, int dtype,
                               cudaStream_t s);
// RoPE angle of rotation pair i (of d / 2) at position `pos`: pos * base^(-2 i / d), cos / sin in fp32.  The forward rotation
// (rope_kv_append_kernel) and the inverse rotation of the backward epilogues share it, so both use bit-identical angles.
L32_DEVICE void rope_cos_sin(float pos, int i, int d, float log2_base, float& cs, float& sn) {
    const float inv_freq = exp2f(-log2_base * (2.0f * static_cast<float>(i) / static_cast<float>(d)));
    sincosf(pos * inv_freq, &sn, &cs);
}

// ---- attention_bwd.cu : attention backward for training calls (no cache, past_len = 0, keys = queries)
size_t gqa_attention_backward_workspace_bytes(int batch, int q_len, int heads);
int gqa_attention_backward(const void* d_ctx, const void* q, const void* cache_k, const void* cache_v, const void* ctx, const float* lse,
                           const uint8_t* keep, const long long* position_ids, void* dq, void* dk, void* dv, void* workspace, int batch,
                           int q_len, int heads, int kv_heads, int head_dim, int max_len, int causal, float rope_base, int dtype,
                           cudaStream_t s);

// ---- sampling.cu : next-token sampling (contract: l32_sample_tokens); one thread-block cluster per row
int sample_tokens(const void* logits, const float* temperature, const int* top_k, const float* top_p,
                  const unsigned long long* seed, const long long* position, long long* tokens_out, float* kept_min_logit,
                  int batch, int vocab, int dtype, cudaStream_t s);

// ---- speculative.cu : token history of a paged cache, n-gram drafts and exact acceptance (contract: include/l32_ffn.h)
int ngram_draft_paged(const int* token_pool, const int* block_table, const int* past_lens, const long long* pending, long long* ids,
                      int* draft_len, int batch, int k, int n_min, int n_max, int max_pages_per_seq, cudaStream_t s);
int speculative_accept(const long long* ids, const long long* sampled, int* token_pool, const int* block_table, const int* past_lens,
                       const int* new_lens, long long* out, int batch, int width, int max_pages_per_seq, cudaStream_t s);

// ---- tp.cu : tensor-parallel glue (cross-GPU flags, reduction of the partial slots)
cudaError_t tp_signal(void* const* peer_flags, int world, int index, uint32_t value, uint32_t* zero8, cudaStream_t s);
cudaError_t tp_peer_copy(void* dst, const void* src, size_t bytes, int ctas, int warps, int unroll, int seg_bytes,
                         cudaStream_t s);
cudaError_t tp_reduce_partials(const void* slots, const uint32_t* flags, uint32_t epoch, int world, int rank,
                               const void* addend, void* y, int64_t rows, int64_t slot_rows, int hidden, int dtype,
                               cudaStream_t s);

// ---- tensor-map helper (gemm_sm100.cu): 2-D row-major [rows, cols] 16-bit tensor, 128-byte swizzled box
int make_tensor_map_2d(CUtensorMap* map, const void* ptr, uint64_t rows, uint64_t cols, uint64_t ld_elems,
                       uint32_t box_rows, uint32_t box_cols, int dtype);
int make_tensor_map_2d_sw(CUtensorMap* map, const void* ptr, uint64_t rows, uint64_t cols, uint64_t ld_elems,
                          uint32_t box_rows, uint32_t box_cols, int dtype, int swizzle_bytes);
// 3-D [planes, rows, cols] 16-bit tensor with rows `ld_elems` and planes `plane_elems` apart, box {64 cols, box_rows, 1 plane},
// 128-byte swizzled.  A box row at or beyond `rows` of its plane is zero-filled, never read from the next plane.
int make_tensor_map_3d(CUtensorMap* map, const void* ptr, uint64_t planes, uint64_t rows, uint64_t cols, uint64_t ld_elems,
                       uint64_t plane_elems, uint32_t box_rows, int dtype);
// The same with a box of box_planes planes: {64 cols, box_rows, box_planes}, landing as box_planes * box_rows consecutive
// 128-byte rows in shared memory.
int make_tensor_map_3d_box(CUtensorMap* map, const void* ptr, uint64_t planes, uint64_t rows, uint64_t cols, uint64_t ld_elems,
                           uint64_t plane_elems, uint32_t box_rows, uint32_t box_planes, int dtype);

}  // namespace l32
