/* libaf2b200.so — C ABI of the B200-native Evoformer trunk hot path.
 *
 * The reference (lucidrains/alphafold2 @ 931466e) is 100 % Python and has no FFI: its boundary for this
 * path is the nn.Module API (alphafold2_pytorch/alphafold2.py).  Each entry point below therefore replaces
 * the forward() of one reference module and is bound from Python with ctypes (alphafold2_b200/_lib.py);
 * INTEGRATION.md shows the stub a reference maintainer would add.
 *
 * Conventions
 *   - every pointer is a DEVICE pointer on the current CUDA device (sm_100a only); nothing is allocated
 *     or retained by the library: outputs and workspace are caller-owned;
 *   - activations x / m are fp32, channel-last, contiguous; weights are packed bf16 (see packing.py) with
 *     fp32 biases / LayerNorm affine parameters; masks are 1-byte bools (torch.bool);
 *   - residual adds are performed in place on the fp32 stream (x <- x + f(x));
 *   - launches are asynchronous on `stream` (a cudaStream_t); CUDA-graph capturable (no sync, no malloc);
 *   - return 0 on success, negative on error (af2_last_error() holds the message). There is NO CPU fallback.
 */
#ifndef AF2B200_H
#define AF2B200_H
#ifdef __cplusplus
extern "C" {
#endif

typedef void* af2_stream_t; /* cudaStream_t */

#define AF2_OK 0
#define AF2_ERR_BAD_ARG (-1)
#define AF2_ERR_CUDA (-2)
#define AF2_ERR_UNSUPPORTED_DEVICE (-3)
#define AF2_ERR_WORKSPACE (-4)

const char* af2_last_error(void);
int af2_abi_version(void);
/* 0 if the current device is compute capability 10.x, AF2_ERR_UNSUPPORTED_DEVICE otherwise */
int af2_check_device(void);
/* 2 (default): LN->projection clusters run on the fused CTA-pair kernel; 1: its single-CTA variant; 0: unfused
 * LayerNorm + GEMM launches (also selectable with the environment variable AF2_PROJ_CTAS, read by af2_check_device) */
void af2_set_proj_mode(int ctas);
/* 1 (default): af2_feed_forward runs the whole block (LayerNorm -> Linear -> GEGLU -> Linear -> residual) as one fused kernel
 * when the shape allows it (d = 128 or 256, hidden a multiple of 64, the fused projection path in mode 2); 0: two launches
 * (fused LayerNorm -> Linear -> GEGLU, then the residual GEMM).  Also selectable with the environment variable AF2_FF_FUSED. */
void af2_set_ff_fused(int on);
/* debug aid: with AF2_PROJ_TRACE=1 in the environment the fused projection kernel records clock64 stamps of one CTA
 * (MMA issue, epilogue and producer progress per tile); this copies the 2048 stamps of the last launch to `out` */
int af2_debug_proj_trace(long long* out);
/* same for the attention kernel (AF2_ATTN_TRACE=1): 8 stamps per key block of CTA 0 (tools/attn_trace.py), 1024 entries */
int af2_debug_attn_trace(long long* out);

/* Kernel launches issued by this library since load (bench.py's gpu_launches). */
unsigned long long af2_launch_count(void);
/* Optional CUDA-event profiling per kernel class (0 linear GEMM, 1 per-channel GEMM, 2 attention, 3 LayerNorm,
 * 4 channel->token, 5 misc): enable(1) clears the records; read() synchronises and sums elapsed ms, algorithmic
 * FLOPs and bytes of the recorded launches of one class and returns their count. */
void af2_profile_enable(int on);
long long af2_profile_read(int cls, double* ms, double* flops, double* bytes);

/* ---------------- FeedForward: alphafold2.py:74-94 (+ residual of :439 / :444) -----------------------
 * x <- x + W2 (a * gelu_erf(g)) + b2,  [a|g] = W1 LN(x) + b1.
 * w1 is packed per column tile of `bn` accumulator columns as [bn/2 value rows | bn/2 gate rows]
 * (zero rows pad the last tile); b1 is permuted the same way. */
typedef struct {
  const float* ln_gamma; const float* ln_beta;        /* FeedForward.norm          [d]            */
  const void* w1; const float* b1;                    /* FeedForward.net.0         packed [n1p, d]  */
  const void* w2; const float* b2;                    /* FeedForward.net.3         [d, hid] , [d]   */
  int bn;                                             /* column tile used for the w1 packing        */
  /* fused LayerNorm->projection kernel (proj_tc.cuh): every projection of the module that reads LN(x), concatenated,
   * each segment zero-padded to a multiple of 256 accumulator columns; b_cat is the matching fp32 bias (zeros where none).
   * NULL -> the unfused LayerNorm + GEMM launches are used.  FeedForward: w_cat == w1, b_cat == b1 (bn must be 256). */
  const void* w_cat; const float* b_cat;
  const void* w_ext;   /* bias block of the fused kernel: bf16 [rows(w_cat)][16], columns 0 / 1 = hi / lo bf16 split of b_cat */
} af2_ff_weights;
int af2_feed_forward(const af2_ff_weights* w, float* x, long long tokens, int d, int hidden,
                     void* workspace, long long workspace_bytes, af2_stream_t stream);
long long af2_feed_forward_workspace(long long tokens, int d, int hidden);

/* ---------------- AxialAttention: alphafold2.py:192-255 driving Attention :98-190 (+ residual) --------
 * x [B, h, w, d] <- x + to_out( softmax(q k^T + bias, mask) v * sigmoid(gating) ).
 * row_attn = 1: attend along w for every (b, h) row; 0: along h for every (b, w) column.
 * edges: RAW fp32 pair tensor [B, n, n, d] (n = attended length) or NULL; bias = edges . w_edge^T,
 * identical for every folded row/column, orientation [head, query, key] (quirks Q4/Q5). */
typedef struct {
  const float* ln_gamma; const float* ln_beta;        /* AxialAttention.norm                        */
  const void* w_qkv;                                  /* [3I, d]: to_q * dim_head^-0.5 | to_kv      */
  const void* w_gate; const float* b_gate;            /* Attention.gating          [I, d], [I]      */
  const void* w_out; const float* b_out;              /* Attention.to_out          [d, I], [d]      */
  const float* w_edge;                                /* edges_to_attn_bias.0      [H, d] fp32/NULL */
  const void* w_cat; const float* b_cat;              /* [pad256(3I) rows w_qkv | pad256(I) rows w_gate], bias likewise */
  const void* w_ext;
} af2_attn_weights;
int af2_axial_attention(const af2_attn_weights* w, float* x, const float* edges, const unsigned char* mask,
                        int B, int h, int wdim, int d, int heads, int dim_head, int row_attn,
                        void* workspace, long long workspace_bytes, af2_stream_t stream);
/* af2_axial_attention with flags: bit 0 = tied ("global") queries -- the queries are averaged over the folded batch before
 * the dot products (alphafold2.py:142-151; AxialAttention(global_query_attn=True), :250; used by the extra-MSA stack :518-527) */
int af2_axial_attention_ex(const af2_attn_weights* w, float* x, const float* edges, const unsigned char* mask, int B,
                           int h, int wdim, int d, int heads, int dim_head, int row_attn, int flags, void* workspace,
                           long long workspace_bytes, af2_stream_t stream);
long long af2_axial_attention_workspace(int B, int h, int wdim, int d, int heads, int dim_head, int row_attn);

/* ---------------- TriangleMultiplicativeModule: alphafold2.py:257-317 (+ residual :381-382) ----------
 * x [B, N, N, d] <- x + to_out( LN_c( mix(L, R) ) * sigmoid(out_gate) ),  hidden_dim == d.
 * outgoing (mix=0): O[i,j,c] = sum_k L[i,k,c] R[j,k,c];  ingoing (mix=1): O[i,j,c] = sum_k L[k,j,c] R[k,i,c].
 * w_left / w_right are packed per tile as [value rows | gate rows] like w1 above. */
typedef struct {
  const float* ln_gamma; const float* ln_beta;        /* .norm                                      */
  const void* w_left; const float* b_left;            /* left_proj + left_gate, packed              */
  const void* w_right; const float* b_right;          /* right_proj + right_gate, packed            */
  const void* w_ogate; const float* b_ogate;          /* out_gate                  [d, d], [d]      */
  const float* on_gamma; const float* on_beta;        /* to_out_norm                                */
  const void* w_out; const float* b_out;              /* to_out                    [d, d], [d]      */
  int bn;
  const void* w_cat; const float* b_cat;              /* [w_left packed | w_right packed | pad256(d) rows w_ogate]  */
  const void* w_ext; const void* w_ext_out;           /* bias blocks of w_cat and (fused tail) of w_out              */
} af2_trimul_weights;
int af2_triangle_multiply(const af2_trimul_weights* w, float* x, const unsigned char* mask, int B, int N, int d,
                          int ingoing, void* workspace, long long workspace_bytes, af2_stream_t stream);
long long af2_triangle_multiply_workspace(int B, int N, int d);

/* ---------------- OuterMean: alphafold2.py:321-351 (+ residual :379) ---------------------------------
 * x [B, N, N, d] <- x + proj_out( sum_s L[s,i,:] * R[s,j,:] / S  [/ (count_ij + eps) when masked] ).
 * Never materialises the (S, N, N, d) tensor of alphafold2.py:341. */
typedef struct {
  const float* ln_gamma; const float* ln_beta;        /* .norm                                      */
  const void* w_lr; const float* b_lr;                /* [2d, d]: left_proj | right_proj, [2d]      */
  const void* w_out; const float* b_out;              /* proj_out                  [d, d], [d]      */
  const void* w_cat; const float* b_cat;              /* pad256(2d) rows of w_lr, bias likewise                      */
  const void* w_ext; const void* w_ext_out;
} af2_outer_weights;
int af2_outer_mean(const af2_outer_weights* w, float* x, const float* m, const unsigned char* msa_mask,
                   int B, int S, int N, int d, float eps, void* workspace, long long workspace_bytes,
                   af2_stream_t stream);
long long af2_outer_mean_workspace(int B, int S, int N, int d);

/* ---------------- stage-level entry points used by the axis-sharded (multi-GPU) schedule ---------------------
 * The reference has no multi-device path; these split the modules above at the points where the sharded
 * schedule (alphafold2_b200/parallel.py) must exchange operands over NCCL.  Batch size 1 per call.
 *   channel-major operand layout: bf16 [channels][chan_stride], token t of a [rows, inner] token grid at
 *   (t / inner) * align8(inner) + t % inner (pad columns zero). */
/* pair bias of a band of pair rows: out bf16 [H][rows][align8(n)] = <x[r, j, :], w_edge[h, :]> (w_edge as packed) */
int af2_pair_bias(const float* x_rows, const float* w_edge, void* bias_out, int rows, int n, int d, int heads,
                  af2_stream_t stream);
/* af2_axial_attention with a precomputed bias [B][H][n][align8(n)] (or NULL) instead of raw edges */
int af2_axial_attention_prebias(const af2_attn_weights* w, float* x, const void* bias_bf16, const unsigned char* mask,
                                int B, int h, int wdim, int d, int heads, int dim_head, int row_attn, void* workspace,
                                long long workspace_bytes, af2_stream_t stream);
/* LN + left/right (masked, gated) -> channel-major Lc, Rc [d][chan_stride]; sigmoid(out_gate) -> gate [tokens, d] */
int af2_triangle_project(const af2_trimul_weights* w, const float* x, const unsigned char* mask, long long tokens,
                         int inner, int d, void* Lc, void* Rc, long long chan_stride, void* gate, void* workspace,
                         long long workspace_bytes, af2_stream_t stream);
long long af2_triangle_project_workspace(long long tokens, int d);
/* x [rows, cols, d] += to_out(LN_c(O) * gate);  Rg holds `pieces` gathered shards, piece_stride elements apart.
 *   outgoing: O[i][j] = sum_k L[i][k] R[j][k], L [c][rows][align8(K)], piece p = R rows j of shard p [c][cols/pieces][align8(K)]
 *   ingoing : O[i][j] = sum_k R[k][i] L[k][j], L [c][K][align8(cols)], piece p = R columns i of shard p [c][K][align8(rows/pieces)] */
int af2_triangle_contract(const af2_trimul_weights* w, float* x, const void* Lc, long long cs_l, const void* Rg,
                          long long cs_r, long long piece_stride, int pieces, const void* gate, int rows, int cols,
                          int K, int d, int ingoing, void* workspace, long long workspace_bytes, af2_stream_t stream);
long long af2_triangle_contract_workspace(int rows, int cols, int d);
/* LN + left|right projections of m [S, inner, d] (masked) -> channel-major LRc [2d][chan_stride] */
int af2_outer_project(const af2_outer_weights* w, const float* m, const unsigned char* msa_mask, long long tokens,
                      int inner, int d, void* LRc, long long chan_stride, void* workspace, long long workspace_bytes,
                      af2_stream_t stream);
long long af2_outer_project_workspace(long long tokens, int d);
/* pair rows [row0, row0+rows): x [rows, N, d] += proj_out(sum_s L[s][i] R[s][j] * scale_ij); msa_mask_full [S][N] or NULL */
int af2_outer_contract(const af2_outer_weights* w, float* x, const void* Lc, long long cs_l, const void* Rg,
                       long long cs_r, long long piece_stride, int pieces, const unsigned char* msa_mask_full,
                       int row0, int rows, int N, int S, int d, float eps, void* workspace, long long workspace_bytes,
                       af2_stream_t stream);
long long af2_outer_contract_workspace(int rows, int N, int d);

/* ---------------- rotary.py:9-20 apply_rotary_pos_emb (dead code at HEAD; standalone op) -------------
 * x, y [b, h, n, dh] fp32; sin, cos [sincos_batch, n, rot] with sincos_batch in {1, b}. */
int af2_rotary(const float* x, const float* sin_, const float* cos_, float* y, int b, int h, int n, int dh,
               int rot, int sincos_batch, af2_stream_t stream);

/* ---------------- building blocks, exported for the parity tests -------------------------------------- */
/* y_bf16[T, d] = LayerNorm(x) (nn.LayerNorm semantics) */
int af2_layernorm_bf16(const float* x, const float* gamma, const float* beta, void* y_bf16, long long T, int d,
                       float eps, af2_stream_t stream);
/* C[b] = A[b] B[b]^T (mn_major = 0: A [M,K], B [N,K]) or A[b]^T B[b] (mn_major = 1: A [K,M], B [K,N]);
 * bf16 operands, fp32 accumulation, fp32 output C [batch, M, ldc]. */
int af2_gemm_bf16_f32(const void* A, long long lda, long long a_batch, const void* Bm, long long ldb,
                      long long b_batch, float* C, long long ldc, long long c_batch, int M, int N, int K,
                      int batch, int mn_major, af2_stream_t stream);

/* ======================================================================================================================
 * STRICT precision mode (alphafold2_b200.set_precision(model, "strict")): the same modules with fp32 activations between
 * kernels and split-bf16 operands on the tensor cores (v = p0 + p1 + p2, three bf16 planes = 24 mantissa bits; the six
 * products down to 2^-24 accumulated in fp32), so that results match the reference's fp32 path inside the north star's
 * rtol 1e-3 / atol 1e-4 also after 12 blocks.  Split weights: bf16 [rows][3][align8(cols)] (plane-major per row), built by
 * ops.split_weight().
 * ====================================================================================================================== */
typedef struct {
  const float* ln_gamma; const float* ln_beta;        /* FeedForward.norm                                   */
  const void* w1; const float* b1;                    /* net.0  split [2*hid][3][align8(d)], fp32 [2*hid]    */
  const void* w2; const float* b2;                    /* net.3  split [d][3][align8(hid)],   fp32 [d]        */
} af2_ff_weights_strict;
long long af2_feed_forward_strict_workspace(long long tokens, int d, int hidden);
int af2_feed_forward_strict(const af2_ff_weights_strict* w, float* x, long long tokens, int d, int hidden, void* workspace,
                            long long workspace_bytes, af2_stream_t stream);                 /* alphafold2.py:74-94 */

typedef struct {
  const float* ln_gamma; const float* ln_beta;        /* AxialAttention.norm                                              */
  const void* w_qkvg; const float* b_qkvg;            /* [to_q * dim_head^-0.5 ; to_kv ; gating] split [4I][3][align8(d)], bias [4I] (zeros | gating.bias) */
  const void* w_out; const float* b_out;              /* attn.to_out split [d][3][align8(I)], fp32 [d]                    */
  const float* w_edge;                                /* edges_to_attn_bias.0.weight fp32 [H][d] or NULL                  */
} af2_attn_weights_strict;
long long af2_axial_attention_strict_workspace(int B, int h, int w, int d, int heads, int dim_head, int row_attn);
int af2_axial_attention_strict(const af2_attn_weights_strict* w, float* x, const float* edges, const unsigned char* mask, int B,
                               int h, int wdim, int d, int heads, int dim_head, int row_attn, int flags, void* workspace,
                               long long workspace_bytes, af2_stream_t stream);              /* alphafold2.py:98-255; flags as af2_axial_attention_ex */

typedef struct {
  const float* ln_gamma; const float* ln_beta;        /* norm                                                                          */
  const void* w5; const float* b5;                    /* [left_proj; right_proj; left_gate; right_gate; out_gate] split [5d][3][align8(d)], fp32 [5d] */
  const float* on_gamma; const float* on_beta;        /* to_out_norm                                                                   */
  const void* w_out; const float* b_out;              /* to_out split [d][3][align8(d)], fp32 [d]                                      */
} af2_trimul_weights_strict;
long long af2_triangle_multiply_strict_workspace(int B, int N, int d);
int af2_triangle_multiply_strict(const af2_trimul_weights_strict* w, float* x, const unsigned char* mask, int B, int N, int d,
                                 int ingoing, void* workspace, long long workspace_bytes, af2_stream_t stream);   /* alphafold2.py:257-317 */

typedef struct {
  const float* ln_gamma; const float* ln_beta;        /* norm                                                       */
  const void* w_lr; const float* b_lr;                /* [left_proj; right_proj] split [2d][3][align8(d)], fp32 [2d] */
  const void* w_out; const float* b_out;              /* proj_out split [d][3][align8(d)], fp32 [d]                 */
} af2_outer_weights_strict;
long long af2_outer_mean_strict_workspace(int B, int S, int N, int d);
int af2_outer_mean_strict(const af2_outer_weights_strict* w, float* x, const float* m, const unsigned char* msa_mask, int B, int S,
                          int N, int d, float eps, void* workspace, long long workspace_bytes, af2_stream_t stream);   /* alphafold2.py:321-351 */

/* building blocks exported for the parity tests of the split-operand GEMM */
int af2_split_bf16(const float* x, void* y_split, long long rows, int K, af2_stream_t stream);
int af2_gemm_split_f32(const void* A_split, const void* B_split, float* C, long long ldc, int M, int N, int K, int batch,
                       af2_stream_t stream);

/* ---------------- pre- / post-trunk glue as fused kernels (SURVEY.md 8f n1) -------------------------------------------
 * af2_embed_pair_init: alphafold2.py:676-726 -- token embedding gather, m = (emb[msa] + msa_embed) + emb[seq],
 *   x[i][j] = (left[i] + right[j]) + pos_emb[clamp(idx_i - idx_j, -R, R) + R] with [left|right] = to_pairwise_repr(emb[seq] + seq_embed).
 *   seq [B][n], msa [B][S][n] int64 token ids (msa / m may be NULL); seq_embed, msa_embed, seq_index optional (NULL).
 * af2_distogram_head: alphafold2.py:821-823 -- out = Linear_{d -> buckets}(LayerNorm((x + x^T) / 2)), all fp32. */
long long af2_embed_pair_init_workspace(int B, int n, int d);
int af2_embed_pair_init(const long long* seq, const long long* msa, const float* token_emb, int vocab, const float* seq_embed,
                        const float* msa_embed, const float* w_pair, const float* b_pair, const float* pos_emb, int max_rel_dist,
                        const long long* seq_index, float* x, float* m, int B, int S, int n, int d, void* workspace,
                        long long workspace_bytes, af2_stream_t stream);
int af2_distogram_head(const float* x, const float* gamma, const float* beta, const float* w, const float* bias, float* out, int B,
                       int n, int d, int buckets, af2_stream_t stream);

/* L2 residency hint for the fp32 pair stream: every kernel launched on `stream` afterwards treats [ptr, ptr + bytes) as
 * persisting in L2 (cudaAccessPolicyWindow; clipped to the device's set-aside / window limits).  ptr == NULL clears it. */
int af2_l2_persist(const void* ptr, long long bytes, float hit_ratio, af2_stream_t stream);

/* ---- peer-memory exchange for the sharded trunk (alphafold2_b200/parallel.py; no reference counterpart: the reference
 * has no multi-GPU path, SURVEY.md 8(e)) ----
 * Every rank owns one arena (af2_peer_alloc: cudaMalloc, zeroed; the first af2_peer_ctrl_bytes() bytes are the barrier
 * control block) which the other ranks of the node map with CUDA IPC (export -> 64-byte handle -> open).  One
 * af2_peer_exchange launch re-lays a row shard out as column shards (or back): chunk p = `rows` rows of `row_bytes`
 * contiguous bytes, read at src + p*src_peer_stride + row*src_row_stride, stored into rank p's arena at
 * dst_off + row*dst_row_stride, followed inside the same kernel by a flag barrier over all P ranks (channel 0 or 1: two
 * exchanges may be in flight on two streams).  peer_base is a DEVICE array of the P arena bases as mapped in this
 * process (own arena at index `rank`).  Every rank must issue the same sequence of exchanges per channel.
 * af2_peer_error returns 1 if a barrier ever gave up waiting (20 s) for a rank. */
int af2_peer_ctrl_bytes(void);
int af2_peer_can_access(int device, int peer_device);
int af2_peer_alloc(long long bytes, void** ptr);
int af2_peer_free(void* ptr);
int af2_peer_export(const void* ptr, unsigned char* handle64);
int af2_peer_open(const unsigned char* handle64, void** ptr);
int af2_peer_close(void* ptr);
int af2_peer_error(const void* my_base);
int af2_peer_exchange(const void* src, long long src_peer_stride, long long src_row_stride, void* const* peer_base,
                      long long dst_off, long long dst_row_stride, int rows, long long row_bytes, int channel, int rank, int P,
                      af2_stream_t stream);

#ifdef __cplusplus
}
#endif
#endif /* AF2B200_H */
