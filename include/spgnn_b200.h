/*
 * spgnn_b200 — C ABI of the B200-native SPGNN GNN-stage kernels (libspgnn_b200.so).
 *
 * The reference (DIAGNijmegen/spgnn) is pure Python and reaches its arithmetic through
 * DGL's Python API (models.py:8).  There is no FFI in the reference to mirror, so each
 * entry point below names the reference call site / DGL operator it replaces.  The
 * reference-side binding a maintainer would add is the ctypes stub in INTEGRATION.md
 * (spgnn_b200/_lib.py is that stub, as shipped).
 *
 * Conventions
 *   - every pointer is a DEVICE pointer unless the name ends in _host; the caller
 *     (PyTorch) owns all memory; nothing is allocated, retained or freed here;
 *   - `stream` is a cudaStream_t passed as void*; all work is stream-ordered on it,
 *     no call synchronises the device; calls are re-entrant and keep no global state;
 *   - return 0 on success, <0 on error (SPGNN_E_*); text via spgnn_last_error()
 *     (thread-local);
 *   - float tensors are fp32 row-major with an explicit leading dimension (ld*, in
 *     elements); "idx" tensors are int32 unless stated int64 (the DGL-visible ones).
 *   - N = nodes in the batch, E = directed edges incl. self loops, B = graphs,
 *     H = heads, F = out feats per head.
 */
#ifndef SPGNN_B200_H
#define SPGNN_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define SPGNN_OK            0
#define SPGNN_E_INVALID    -1   /* bad argument (shape, alignment, null) */
#define SPGNN_E_CUDA       -2   /* a CUDA runtime call failed */
#define SPGNN_E_UNSUPPORTED -3  /* shape outside what the kernels were built for */
#define SPGNN_E_WORKSPACE  -4   /* workspace too small */

#define SPGNN_ACT_NONE 0
#define SPGNN_ACT_ELU  1
#define SPGNN_ACT_TANH 2
#define SPGNN_ACT_RELU 3
#define SPGNN_ACT_LEAKY 4      /* slope passed separately; the GAT layer entry points use F.leaky_relu's 0.01 */

const char* spgnn_last_error(void);
int  spgnn_abi_version(void);
/* Number of kernels this library has launched in this process (diagnostic counter; bench.py's gpu_launches). */
int64_t spgnn_launch_count(void);
/* SM count etc. of the current device (used by the host side to size workspaces). */
int  spgnn_device_info(int* sm_count, int* cc_major, int* cc_minor);

/* ------------------------------------------------------------------------------------
 * Graph construction and batching.
 * Replaces: nx.DiGraph(adj) -> DGLGraph -> dgl.remove_self_loop -> g.add_edges(nodes,nodes)
 *           (job_runner.py:1779-1801, :1319-1344, :822-838) and dgl.batch (job_runner.py:1390,
 *           :1882, :2046).  Integer work: results are bit-identical to DGL's.
 * ---------------------------------------------------------------------------------- */

/* Exclusive prefix scan of int64 counts: out[0]=0, out[i+1]=out[i]+in[i], n inputs, n+1 outputs.
 * ws: at least spgnn_scan_ws_bytes(n) bytes. */
int64_t spgnn_scan_ws_bytes(int64_t n);
int spgnn_scan_i64(const int64_t* in, int64_t* out, int64_t n, void* ws, void* stream);

/* Dense adjacency -> DGL edge list, per graph.
 *   adj      uint8, graphs concatenated; graph g is an n_g x n_g row-major block at adj_off[g]
 *   n_nodes  int64 [B]; adj_off int64 [B+1] (= scan of n_g^2); node_off int64 [B+1]
 * pass 1 (count): row_cnt[int64, N] = off-diagonal non-zeros per row; n_edges[int64,B] = sum + n_g
 * pass 2 (fill):  given edge_off = scan(n_edges) and row_off = scan over rows of row_cnt (int64 [N+1]),
 *                 writes LOCAL src/dst int64 [E]: off-diagonal non-zeros in row-major order, then (k,k), k<n_g. */
int spgnn_adj_count(const uint8_t* adj, const int64_t* adj_off, const int64_t* n_nodes, const int64_t* node_off,
                    int64_t B, int64_t N, int64_t* row_cnt, int64_t* n_edges, void* stream);
int spgnn_adj_fill(const uint8_t* adj, const int64_t* adj_off, const int64_t* n_nodes, const int64_t* node_off,
                   const int64_t* edge_off, const int64_t* row_off, int64_t B, int64_t N,
                   int64_t* src_local, int64_t* dst_local, void* stream);

/* dgl.batch + CSC/CSR build.
 *   in : node_off/edge_off int64 [B+1]; src_local/dst_local int64 [E] (per-graph local ids, DGL edge order)
 *   out: src/dst int64 [E] global ids (== dgl.batch(...).edges());
 *        node_gid int32 [N];
 *        in_ptr int32 [N+1], in_src int32 [E], in_eid int32 [E]   — in-edges of each node, ascending edge id
 *        out_ptr int32 [N+1], out_dst int32 [E], out_slot int32 [E] — out-edges; out_slot = position in in_* arrays
 *        flags int32 [4]: [0] = number of zero-in-degree nodes, [1] = number of out-of-range endpoints,
 *        [2] = largest in-degree, [3] = largest out-degree
 *   ws : spgnn_batch_ws_bytes(N, E) bytes of scratch. */
int64_t spgnn_batch_ws_bytes(int64_t N, int64_t E);
int spgnn_batch_build(const int64_t* node_off, const int64_t* edge_off, int64_t B, int64_t N, int64_t E,
                      const int64_t* src_local, const int64_t* dst_local,
                      int64_t* src, int64_t* dst, int32_t* node_gid,
                      int32_t* in_ptr, int32_t* in_src, int32_t* in_eid,
                      int32_t* out_ptr, int32_t* out_dst, int32_t* out_slot,
                      int32_t* flags, void* ws, void* stream);

/* ------------------------------------------------------------------------------------
 * Dense projection (DGL GATConv.fc / res_fc, GraphConv weight, SAGEConv fc_*, GIN MLP, gnn_out):
 * SURVEY §2.1 K1/K8.  fp32 in, fp32 out.
 *   C[M,N] (ldc) = [A1 | A2][M,K1+K2] * W[N, K1+K2 (ldw)]^T  (+ bias[N]) (act)
 * A2 may be null (K2 = 0): the two-source form removes torch.cat([h_s,h_p]) (models.py:477,481).
 * mode: 0 = fp32 SIMT, 1 = tcgen05 tensor cores with split-bf16 operands (a = hi + lo; hi*hi + hi*lo + lo*hi,
 *       fp32 accumulate in TMEM; relative error ~1e-5) — falls back to mode 0 when 16-byte alignment of the
 *       operands / leading dimensions is not given.  ws: scratch for the pre-split weight, spgnn_linear_fwd_ws /
 *       spgnn_linear_bwd_input_ws bytes (mode 1 only).
 * ---------------------------------------------------------------------------------- */
int64_t spgnn_linear_fwd_ws(int64_t N, int64_t K1, int64_t K2);
int spgnn_linear_fwd(const float* A1, int64_t lda1, int64_t K1, const float* A2, int64_t lda2, int64_t K2,
                     const float* W, int64_t ldw, const float* bias, int act, float slope,
                     float* C, int64_t ldc, int64_t M, int64_t N, int mode, void* ws, int64_t ws_bytes, void* stream);
/* dA[M,K] (ldda) = dC[M,N] (lddc) * W[N, k_off : k_off+K] (ldw) */
int64_t spgnn_linear_bwd_input_ws(int64_t N, int64_t K);
int spgnn_linear_bwd_input(const float* dC, int64_t lddc, const float* W, int64_t ldw, int64_t k_off,
                           float* dA, int64_t ldda, int64_t M, int64_t N, int64_t K, int mode,
                           void* ws, int64_t ws_bytes, void* stream);
/* dW[N, k_off : k_off+K] (lddw) = dC[M,N]^T * A[M,K] (lda); split over M into `splits` partial sums in ws
 * (splits*N*K floats, see spgnn_linear_bwd_weight_ws) that a second kernel reduces deterministically. */
int64_t spgnn_linear_bwd_weight_ws(int64_t M, int64_t N, int64_t K);
int spgnn_linear_bwd_weight(const float* dC, int64_t lddc, const float* A, int64_t lda,
                            float* dW, int64_t lddw, int64_t k_off, int64_t M, int64_t N, int64_t K,
                            void* ws, int mode, void* stream);
/* Two-source form: dW[N, K1+K2] (lddw) = dC[M,N]^T * [A1 | A2] in ONE pass over dC (mode 1: 256 x BN tensor-core tiles
 * with two TMEM accumulators sharing the dC tile). */
int64_t spgnn_linear_bwd_weight2_ws(int64_t M, int64_t N, int64_t K1, int64_t K2);
int spgnn_linear_bwd_weight2(const float* dC, int64_t lddc, const float* A1, int64_t lda1, int64_t K1,
                             const float* A2, int64_t lda2, int64_t K2, float* dW, int64_t lddw,
                             int64_t M, int64_t N, void* ws, int mode, void* stream);
/* ------------------------------------------------------------------------------------
 * Dense projection over "planes" operands — the production path of the same DGL projections (GATConv.fc / res_fc,
 * gnn_out; models.py:301-314, 425-456, 1167-1170).
 * Planes: an fp32-valued matrix X[rows, cols] stored as TWO bf16 matrices, X = hi + lo (|residual| <= 2^-17 |X|),
 * both [rows, ld] row-major; the pointer passed is `hi`, lo = hi + plane_stride (elements).  ld and plane_stride must
 * be multiples of 8 (16-byte rows), the base 16-byte aligned.  Same bytes as fp32, but the tensor cores consume them
 * directly: operands go global -> shared by TMA and every product is hi*hi + hi*lo + lo*hi with fp32 accumulation
 * (relative error ~1e-5).  The aggregation kernels (spgnn_gat_layer_*) and spgnn_split_planes PRODUCE planes, so no
 * GEMM converts anything.  Weights stay fp32 in the ABI; they are split into `ws` once per call.
 *   split_planes      : out planes [M, ldo] = dropout([x1 | x2], p) * 1/(1-p); mask = 16 hash bits per element of
 *                       hash(seed, row * ceil(K/4) + col/4) (GATConv feat_drop on torch.cat([h_s,h_p]),
 *                       models.py:431-435,477); p = 0 is a plain conversion.  When the result is one part of a
 *                       larger concatenation, concat_chunks = ceil(K_concat/4) and chunk_off = first column / 4
 *                       place it in the consumer's mask numbering (0, 0 = the tensor stands alone).
 *   planes_linear_fwd : C[M,N] fp32 (ldc) = [A1 | A2] * W[N, K1+K2 (ldw)]^T (+bias)(act)
 *   planes_linear_bwd_input  : dA[M,K] fp32 (ldda) = dC[M,N] * W[N, k_off : k_off+K]
 *   planes_linear_bwd_weight : dW[N, K1+K2] fp32 (lddw) = dC[M,N]^T * [X1 | X2]; reduction over the M nodes split
 *                       into partial sums in ws, reduced in fixed order (deterministic).
 * ---------------------------------------------------------------------------------- */
int spgnn_split_planes(const float* x1, int64_t ld1, int64_t K1, const float* x2, int64_t ld2, int64_t K2,
                       float p, uint64_t seed, int64_t concat_chunks, int64_t chunk_off,
                       uint16_t* out_hi, int64_t ldo, int64_t plane_stride, int64_t M, void* stream);
int64_t spgnn_planes_linear_fwd_ws(int64_t N, int64_t K1, int64_t K2);
int spgnn_planes_linear_fwd(const uint16_t* A1, int64_t lda1, int64_t ps1, int64_t K1,
                            const uint16_t* A2, int64_t lda2, int64_t ps2, int64_t K2,
                            const float* W, int64_t ldw, const float* bias, int act, float slope,
                            float* C, int64_t ldc, int64_t M, int64_t N, void* ws, int64_t ws_bytes, void* stream);
int64_t spgnn_planes_linear_bwd_input_ws(int64_t N, int64_t K);
int spgnn_planes_linear_bwd_input(const uint16_t* dC, int64_t lddc, int64_t ps, const float* W, int64_t ldw,
                                  int64_t k_off, float* dA, int64_t ldda, int64_t M, int64_t N, int64_t K,
                                  void* ws, int64_t ws_bytes, void* stream);
/* Same, with the feat_drop mask of the consuming layer folded into the epilogue: dA is the gradient of the DROPPED
 * input, dA[r, c] *= keep(r, c) / (1 - drop_p), keep from the plane producers' hash convention (16 bits per element,
 * chunk index r * concat_chunks + (k_off + c) / 4, k_off % 4 == 0; concat_chunks <= 0: ceil((k_off + K) / 4)).  drop_p == 0: identical to the call above.
 * The producer layer's backward then reads an already-masked gradient source (its GSrc.drop_p = 0). */
int spgnn_planes_linear_bwd_input_masked(const uint16_t* dC, int64_t lddc, int64_t ps, const float* W, int64_t ldw,
                                         int64_t k_off, float* dA, int64_t ldda, int64_t M, int64_t N, int64_t K,
                                         float drop_p, uint64_t seed, int64_t concat_chunks,
                                         void* ws, int64_t ws_bytes, void* stream);
int64_t spgnn_planes_linear_bwd_weight_ws(int64_t M, int64_t N, int64_t K1, int64_t K2);
int spgnn_planes_linear_bwd_weight(const uint16_t* dC, int64_t lddc, int64_t psc,
                                   const uint16_t* X1, int64_t ldx1, int64_t psx1, int64_t K1,
                                   const uint16_t* X2, int64_t ldx2, int64_t psx2, int64_t K2,
                                   float* dW, int64_t lddw, int64_t M, int64_t N,
                                   void* ws, int64_t ws_bytes, void* stream);
/* Elementwise half of a projection's backward in one pass: d = g * act'(y) (y = the forward OUTPUT; act NONE or
 * y NULL: d = g) written as planes [M, ldo] for planes_linear_bwd_input / _bwd_weight, plus (colsum_out != NULL) the
 * column sums of d = the bias gradient (row bands in ws, spgnn_act_bwd_planes_ws(N) bytes, reduced in fixed order).
 * g / y: fp32, 16-byte aligned rows padded to a multiple of 4 columns.  Replaces act_bwd + split_planes + colsum.
 * drop_p > 0: g is the gradient of a tensor that was dropped on its way into its consumer by
 * spgnn_split_planes(p, seed) standing alone (chunk index row * ceil(N/4) + col/4): the same mask is applied to g
 * first (Linear -> Dropout -> Linear chains, e.g. the GIN MLPs of models.py:358-383, without a dropout pass). */
int64_t spgnn_act_bwd_planes_ws(int64_t N);
int spgnn_act_bwd_planes(const float* g, int64_t ldg, const float* y, int64_t ldy, int act, float slope,
                         float drop_p, uint64_t drop_seed, uint16_t* out_hi, int64_t ldo, int64_t plane_stride,
                         int64_t M, int64_t N, float* colsum_out, void* ws, void* stream);
/* The launch plan planes_linear_bwd_weight would use (host only, no device work; for tests and profiling):
 * out[0..7] = {swap (1: the gradient dC is the M-side operand), np_tiles, nq_tiles, row splits, CTAs, rows per
 * split, 64-column blocks on the M side, on the N side} and, when cap >= 9, out[8] = 1 if the two sources X1 / X2 get
 * one launch each (their blocks tile badly together; out[0..7] then describe the first launch, X1 alone).  Returns the
 * number of ints written (8 or 9). */
int64_t spgnn_planes_linear_bwd_weight_plan(int64_t M, int64_t N, int64_t K1, int64_t K2, int32_t* out, int64_t cap);

/* out[n] = sum_m X[m, n]  (bias gradients).  ws: spgnn_colsum_ws(N) bytes. */
int64_t spgnn_colsum_ws(int64_t N);
int spgnn_colsum(const float* X, int64_t ldx, int64_t M, int64_t N, float* out, void* ws, void* stream);

/* ------------------------------------------------------------------------------------
 * GATConv weight packing.  One projection yields z, the residual projection (res_fc, models.py:301-314) and both
 * attention logits when its weight is P = [W_fc ; W_res ; W_l ; W_r] with W_l[h, :] = sum_f attn_l[h, f] W_fc[hF+f, :]
 * (el = (x W_fc^T).attn_l = x.(W_fc^T attn_l); DGL GATConv el/er, SURVEY §8a A1).
 *   pack_weight     : out [(HF * (1 + has W_res) + 2H), ldo] fp32, rows in the order above, columns [K, ldo) zeroed
 *   pack_weight_bwd : gradient of P -> dW_fc [HF, lddw] (= dP rows + attn_l dP_l + attn_r dP_r), dW_res [HF, lddr],
 *                     d attn_l / d attn_r [HF] (= <W_fc row, dP_l / dP_r of its head>); any output may be NULL.
 * ---------------------------------------------------------------------------------- */
int spgnn_gat_pack_weight(const float* W_fc, int64_t ldw, const float* W_res, int64_t ldr,
                          const float* attn_l, const float* attn_r, int64_t H, int64_t F, int64_t K,
                          float* out, int64_t ldo, void* stream);
int spgnn_gat_pack_weight_bwd(const float* dP, int64_t ldp, const float* W_fc, int64_t ldw,
                              const float* attn_l, const float* attn_r, int64_t H, int64_t F, int64_t K,
                              int has_res, float* dW_fc, int64_t lddw, float* dW_res, int64_t lddr,
                              float* d_attn_l, float* d_attn_r, void* stream);

/* ------------------------------------------------------------------------------------
 * GAT edge-softmax + aggregation + residual + bias + activation (+ head mean), fused.
 * Replaces DGL GATConv.forward K3-K9 (SURVEY §2.1) as called at models.py:324,326,478,479,482,535,538.
 *   Y   [N, ldy]: cols [0,HF) z;  [res_off, res_off+HF) residual projection (res_mode 1);
 *                 el at col el_off+h, er at col er_off+h  (logits come out of the projection as
 *                 extra columns: el = x . (W_fc^T attn_l))
 *   res_mode 0 none, 1 linear (in Y), 2 identity: xres [N, ldxres] viewed [N, -1, F] (D == F -> broadcast)
 *   out [N, ldo]: HF wide, or F wide when mean_heads
 *   att [E, H] : softmax weights per in-edge slot (before dropout), saved for backward
 *   attn dropout: keep-prob 1-p, mask = hash(seed, slot*H+h); p = 0 disables.
 * ---------------------------------------------------------------------------------- */
int spgnn_gat_agg_fwd(const float* Y, int64_t ldy, int64_t res_off, int64_t el_off, int64_t er_off,
                      int res_mode, const float* xres, int64_t ldxres, int64_t xres_cols,
                      const float* bias, int act, float negative_slope, int mean_heads,
                      float attn_drop_p, uint64_t seed,
                      const int32_t* in_ptr, const int32_t* in_src,
                      int64_t N, int64_t H, int64_t F,
                      float* out, int64_t ldo, float* att, void* stream);
/* Backward.  g_out [N, ldg] (HF or F wide when mean_heads); out = saved forward output (ignored when
 * mean_heads: pre-activations are recomputed); writes dY [N, ldy] (same column layout as Y: dz, dres, del,
 * der) and, for res_mode 2, dxres [N, ldxres] (overwritten).  The bias gradient is the column sum of g:
 * for res_mode 1 that is spgnn_colsum over the dres columns of dY, otherwise over g_ws.
 * g_ws: float [N, H*F] (only read/written when res_mode != 1); ds_ws: float [E*H] scratch. */
int spgnn_gat_agg_bwd(const float* g_out, int64_t ldg, const float* out, int64_t ldo,
                      const float* Y, int64_t ldy, int64_t res_off, int64_t el_off, int64_t er_off,
                      int res_mode, const float* xres, int64_t ldxres, int64_t xres_cols,
                      const float* bias, int act, float negative_slope, int mean_heads,
                      float attn_drop_p, uint64_t seed, const float* att,
                      const int32_t* in_ptr, const int32_t* in_src,
                      const int32_t* out_ptr, const int32_t* out_dst, const int32_t* out_slot,
                      int64_t N, int64_t H, int64_t F,
                      float* dY, float* dxres, float* g_ws, float* ds_ws, void* stream);

/* ------------------------------------------------------------------------------------
 * GAT layer of the planes pipeline: the same fused edge-softmax + aggregation + residual + bias + activation
 * (+ head mean) as spgnn_gat_agg_*, but the layer OUTPUT is written as planes — one copy per consumer, with that
 * consumer's feat_drop mask already applied (GATConv.feat_drop on torch.cat([h_s,h_p]), models.py:431-456,476-482) —
 * and the backward reads the masked gradient contributions of every consumer (the dX of the next projections)
 * directly and writes dY as planes for the dX / dW projections.  torch.cat, dropout and the fp32 -> bf16 split never
 * make a pass of their own over HBM.  The bias gradient (column sum of g) comes out of the same backward kernel.
 *   Y  [N, ldy] fp32: cols [0,HF) z; [res_off, res_off+HF) residual projection (res_mode 1); el at el_off+h,
 *      er at er_off+h.  res_mode 0 = no residual, 1 = linear (identity residuals use spgnn_gat_agg_*).
 *   forward : att [E,H] out; `out` fp32 [N, ldo] optional; sinks[n_sinks] planes copies of the output
 *             (width HF, or F when mean_heads).  Dropout mask of a sink = 16 hash bits per element of
 *             hash(seed, row * concat_chunks + chunk_off + col/4) — the convention of spgnn_split_planes, with
 *             concat_chunks = ceil(K_concat/4) of the consumer's concatenated input and chunk_off = this tensor's
 *             first column in it / 4.
 *   backward: gsrc[n_gsrc] fp32 gradient contributions (pointer already at this tensor's first column inside the
 *             consumer's dX), each masked with the consumer's dropout as above; outputs dY planes [N, dY_ld] (same
 *             column layout as Y), ds_ws [E*H] scratch, g_ws fp32 [N,HF] (only when res_mode 0),
 *             dbias [HF] (optional; needs dbias_ws of spgnn_gat_layer_dbias_ws bytes).  Pre-activations are
 *             recomputed from Y, so the forward output need not be kept.
 * ---------------------------------------------------------------------------------- */
typedef struct spgnn_sink {
    uint16_t* hi; int64_t ld; int64_t plane_stride;
    int64_t concat_chunks; int64_t chunk_off;
    float drop_p; uint32_t reserved; uint64_t seed;
} spgnn_sink;
typedef struct spgnn_gsrc {
    const float* g; int64_t ld;
    int64_t concat_chunks; int64_t chunk_off;
    float drop_p; uint32_t reserved; uint64_t seed;
} spgnn_gsrc;
typedef struct spgnn_gat_layer {
    const int32_t* in_ptr; const int32_t* in_src;
    const int32_t* out_ptr; const int32_t* out_dst; const int32_t* out_slot;
    int64_t N; int32_t H; int32_t F;
    const float* Y; int64_t ldy; int64_t res_off; int64_t el_off; int64_t er_off;
    int32_t res_mode; int32_t act; float negative_slope; int32_t mean_heads;
    const float* bias; float attn_drop_p; uint32_t reserved0; uint64_t attn_seed;
    float* att;
    float* out; int64_t ldo; int32_t n_sinks; int32_t reserved1; spgnn_sink sinks[2];
    int32_t n_gsrc; int32_t reserved2; spgnn_gsrc gsrc[3];
    uint16_t* dY_hi; int64_t dY_ld; int64_t dY_ps;
    float* g_ws; float* ds_ws; float* dbias; float* dbias_ws;
    /* optional: per-graph node offsets [B+1] (int64) and the largest graph of the batch.  When given (and F % 64
     * == 0, no head mean, the largest graph fits in shared memory) the layer runs one CTA per graph with the
     * graph's z rows staged in shared memory by TMA, 64 columns at a time: every neighbour gather is a shared-memory
     * read and DRAM traffic equals the algorithmic bytes; the backward then fuses the destination and source sides.
     * max_degree = largest in- or out-degree of the batch (spgnn_batch_build flags[2], flags[3]); 0 = unknown. */
    const int64_t* node_off; int64_t B; int64_t max_nodes; int64_t max_degree;
} spgnn_gat_layer;
int64_t spgnn_gat_layer_sizeof(void);
int64_t spgnn_gat_layer_dbias_ws(int64_t N, int64_t H, int64_t F);
int spgnn_gat_layer_fwd(const spgnn_gat_layer* L, void* stream);
int spgnn_gat_layer_bwd(const spgnn_gat_layer* L, void* stream);

/* ------------------------------------------------------------------------------------
 * Aggregate-first evaluation of the head-averaged GAT OUTPUT layer (models.py:311-314 / :436-440 followed by
 * `.mean(1)`, models.py:326,482): `GATConv(k_in -> H x F, residual)` with H*F >> k_in (192 -> 2 x 1024 in SPGNN-3).
 * Aggregation is linear, so  sum_u a[u->v,h] (x[u] W_h^T) = (sum_u a[u->v,h] x[u]) W_h^T : the edge softmax and
 * the neighbour aggregation run on the NARROW input (k_in columns) and one tcgen05 GEMM per (row tile, head)
 *     pre_h = [Ax_h | x] * [W_fc,h | W_res,h]^T + b_h ,   out = 1/H sum_h act(pre_h)
 * applies activation and head mean in its epilogue: the [N, 2*H*F] projection (20 GB at 4096 trees) is never
 * written to HBM.  The backward RECOMPUTES pre_h with the same kernel (mode 1) and emits
 * dpre_h = g/H * act'(pre_h) as planes, plus the bias gradient; dW / d[Ax|x] are ordinary planes GEMMs on dpre.
 *   eler  fp32 [N, 2H]: el[h] at column h, er[h] at column H+h (a [2H, k_in] projection of the same input).
 *   XA    planes [N, (H+1)*kp], kp = k_in rounded up to 64: block h < H = Ax_h, block H = x (a copy of the
 *         concatenated, already feat-dropped input); padding columns are written as zeros.  K1 % 64 == 0.
 *   aggx_fwd : att [E,H] and XA from (X1 | X2, eler).
 *   aggx_bwd : from dXA fp32 [H][N, ld_dxa] (cols [0,k4) = d(Ax_h), [k4, 2*k4) = d(x) through the residual;
 *              k4 = k_in rounded up to 4; the second half is read only when has_res) computes the edge-softmax
 *              backward on the narrow rows, d_eler (fp32 + planes, for the dW of the logit projection) and
 *              dX fp32 [N, k_in] = d(concatenated input), including the logit path d_eler * w_eler.
 * ---------------------------------------------------------------------------------- */
typedef struct spgnn_gat_wide {
    const int32_t* in_ptr; const int32_t* in_src;
    const int32_t* out_ptr; const int32_t* out_dst; const int32_t* out_slot;
    int64_t N; int32_t H; int32_t has_res;
    const uint16_t* X1; int64_t ldx1; int64_t psx1;
    const uint16_t* X2; int64_t ldx2; int64_t psx2;
    int32_t K1; int32_t K2;
    const float* eler; int64_t ld_eler;
    float negative_slope; float attn_drop_p; uint64_t attn_seed;
    float* att;
    uint16_t* XA; int64_t ldxa; int64_t psxa; int64_t kp;
    const float* dXA; int64_t ld_dxa; int64_t head_stride;
    const float* w_eler; int64_t ld_w;
    float* ds_ws;
    float* d_eler; int64_t ld_de;
    uint16_t* d_eler_planes; int64_t ld_dep; int64_t ps_dep;
    float* dX; int64_t ld_dx;
} spgnn_gat_wide;
int64_t spgnn_gat_wide_sizeof(void);
int spgnn_gat_aggx_fwd(const spgnn_gat_wide* L, void* stream);
int spgnn_gat_aggx_bwd(const spgnn_gat_wide* L, void* stream);

/* The wide GEMM.  W: fp32 packed weight [>= (1+has_res)*H*F rows, ldw]: rows [0,HF) = W_fc, [HF,2HF) = W_res,
 * k_in valid columns each.  bias [H*F] or NULL.
 *   mode 0: out fp32 [N, ldo] (optional) and/or out planes (optional) <- 1/H sum_h act(pre_h)      (width F)
 *   mode 1: g = sum of n_g fp32 [N, F] gradient sources; dpre planes [N, H*F] <- g/H * act'(pre_h);
 *           dbias [H*F] (optional) <- column sums of dpre (per-CTA partial rows reduced in fixed order).
 * ws: spgnn_wide_linear_ws bytes. */
int64_t spgnn_wide_linear_ws(int64_t H, int64_t F, int64_t kp, int has_res);
int spgnn_wide_linear(const uint16_t* XA, int64_t ldxa, int64_t psxa, int64_t kp, int64_t k_in, int64_t M,
                      int H, int F, int has_res, const float* W, int64_t ldw, const float* bias, int act, int mode,
                      float* out, int64_t ldo, uint16_t* out_planes, int64_t ldp, int64_t psp,
                      const float* g0, int64_t ldg0, const float* g1, int64_t ldg1, const float* g2, int64_t ldg2,
                      uint16_t* dpre, int64_t ldd, int64_t psd, float* dbias,
                      void* ws, int64_t ws_bytes, void* stream);
/* Mode 0 that also writes dact fp32 [N, ldda >= H*F] <- act'(pre_h) for every head h (column h*F + f), the values
 * mode 1 recomputes, bit for bit.  Same ws as spgnn_wide_linear. */
int spgnn_wide_linear_fwd_dact(const uint16_t* XA, int64_t ldxa, int64_t psxa, int64_t kp, int64_t k_in, int64_t M,
                               int H, int F, int has_res, const float* W, int64_t ldw, const float* bias, int act,
                               float* out, int64_t ldo, uint16_t* out_planes, int64_t ldp, int64_t psp,
                               float* dact, int64_t ldda, void* ws, int64_t ws_bytes, void* stream);
/* The dpre of mode 1 when the layer output feeds a linear head (W_head [C, ldwh >= F], C <= 64) and dact was saved:
 * gl = the head's output-gradient planes [M, C] (ld ldgl, plane stride psgl);  with g = gl * W_head (the head's dX,
 * never stored) and up to two further fp32 [M, F] sources g0, g1,
 *   dpre planes [M, H*F] <- (g0 + g1 + g) / H * dact_h;  dbias [H*F] (optional) <- column sums of dpre.
 * ws: spgnn_wide_dpre_ws bytes. */
int64_t spgnn_wide_dpre_ws(int64_t H, int64_t F);
int spgnn_wide_dpre(const uint16_t* gl, int64_t ldgl, int64_t psgl, int64_t C, int64_t M, int H, int F,
                    const float* W_head, int64_t ldwh, const float* dact, int64_t ldda,
                    const float* g0, int64_t ldg0, const float* g1, int64_t ldg1,
                    uint16_t* dpre, int64_t ldd, int64_t psd, float* dbias, void* ws, int64_t ws_bytes, void* stream);

/* ------------------------------------------------------------------------------------
 * Weighted-sum aggregation (DGL SpMM copy_u.sum with degree norms): GraphConv, GINConv-mean, SAGEConv mean / gcn.
 *   out[v, :] = act( post[v] * (sum_{s in seg(v)} pre[nbr[s]] * x[nbr[s], :] + [self_in] pre[v] * x[v, :])
 *                    + self_coef * x[v, :] + add[v, :] + bias )            for v < N
 * The two self terms are read only for v < n_self (n_self <= N; on a sampled block the destination rows): self_in
 * puts x[v] inside the norm (SAGEConv 'gcn': (sum + x[v]) / (deg + 1)), self_coef outside it (read from device
 * memory, GIN's 1+eps, when self_coef_ptr != null, value = 1 + *self_coef_ptr; else 0).  pre/post/add/bias may be
 * null.  Forward uses the in-CSC with N = destination rows, backward the out-CSR with pre/post swapped and N = source
 * rows.  Replaces GraphConv (models.py:172-182), GINConv "mean" (models.py:358-383) and SAGEConv "mean" / "gcn"
 * message passing.
 * ---------------------------------------------------------------------------------- */
int spgnn_spmm(const float* x, int64_t ldx, const int32_t* ptr, const int32_t* nbr,
               const float* pre, const float* post, const float* self_eps_ptr, int self_in, int64_t n_self,
               const float* add, int64_t ld_add, const float* bias, int act, float slope,
               float* out, int64_t ldo, int64_t N, int64_t F, void* stream);
/* deg^-1/2 and 1/deg (clamped at 1) from a ptr array: norm_sqrt[N], norm_inv[N] (either may be null) */
int spgnn_degree_norms(const int32_t* ptr, int64_t N, float* norm_sqrt, float* norm_inv, void* stream);
/* out[i] = 1 / max(deg(i) + add, 1) from a ptr array (SAGEConv mean: add 0, gcn: add 1) */
int spgnn_inv_degree(const int32_t* ptr, int64_t N, float add, float* out, void* stream);

/* SAGEConv "pool": neigh[v,f] = max_{u->v} m[u,f]; arg[v,f] = in-slot of the max (first max).
 * Backward: dm[u,f] = sum over out-edges (u->v, slot s) of g[v,f] * [arg[v,f] == s].
 * Replaces DGL SpMM copy_u.max (models.py:668-679). */
int spgnn_sage_maxpool_fwd(const float* m, int64_t ldm, const int32_t* in_ptr, const int32_t* in_src,
                           float* out, int64_t ldo, int32_t* arg, int64_t N, int64_t F, void* stream);
int spgnn_sage_maxpool_bwd(const float* g, int64_t ldg, const int32_t* arg,
                           const int32_t* out_ptr, const int32_t* out_dst, const int32_t* out_slot,
                           float* dm, int64_t lddm, int64_t N, int64_t F, void* stream);

/* ------------------------------------------------------------------------------------
 * SAGEConv "lstm" reducer (DGL 0.7 _lstm_reducer: nn.LSTM(D, D, batch_first=True) over each destination's in-edge
 * messages in in-CSC order, zero initial state, h_T = the aggregate; gate order i, f, g, o).
 * Rows are the destinations sorted by in-degree, descending and stable, so step t runs over the first n_t rows
 * (n_t = #destinations with in-degree > t) and its rows are a contiguous block at row off_t = sum_{s<t} n_s of the
 * per-step buffers (sum_t n_t = E).
 *   lstm_order_count / _scatter : the stable counting sort.  key = max_deg - deg (so descending degree), chunk = 256
 *       destinations; count writes counts[key * n_chunks + chunk] (int64), the caller scans them (spgnn_scan_i64)
 *       into offs, scatter writes perm[row] = destination and rank[destination] = row.  max_deg < 12288.
 *   lstm_cell_fwd (step t): pre = P[src(v, t)] + R[r] (R = H_{t-1}[:n_t] W_hh^T, null at t = 0), with P = X W_ih^T +
 *       b_ih + b_hh [n_src, 4D]; c = f c_prev + i g, h = o tanh(c).  Saves the gate activations (fp32 stored as
 *       their high / low 16-bit halves in the two planes of `gates`, the layout the backward overwrites with the
 *       gate-gradient planes in place) and c.  Rows r < n_next continue: h goes as planes to `h_next` (row r), the
 *       operand of step t+1's GEMM; the other rows end here: h goes to out[perm[r]] (fp32).
 *   lstm_cell_bwd (step t): dh = r < n_next ? dh_rec[r] (= dgates_{t+1} W_hh) : g_out[perm[r]]; dc carried in
 *       dc[r]; writes the pre-activation gradients as planes over the saved gates.
 *   lstm_dp : dP[u] = sum over u's out-edges (u -> v, in-slot s) of dgates row off[s - in_ptr[v]] + rank[v]; a
 *       deterministic gather over the out-CSR, no atomics.
 * D % 4 == 0; planes row strides (ld) multiples of 8.
 * ---------------------------------------------------------------------------------- */
int spgnn_lstm_order_count(const int32_t* in_ptr, int64_t N, int64_t max_deg, int64_t* counts, void* stream);
int spgnn_lstm_order_scatter(const int32_t* in_ptr, int64_t N, int64_t max_deg, const int64_t* offs,
                             int32_t* perm, int32_t* rank, void* stream);
int spgnn_lstm_cell_fwd(int64_t t, int64_t n_t, int64_t n_next, const int32_t* perm, const int32_t* in_ptr,
                        const int32_t* in_src, const float* P, int64_t ldp, const float* R, int64_t ldr,
                        uint16_t* gates, int64_t ldg, int64_t psg, const float* c_prev, float* c_cur,
                        uint16_t* h_next, int64_t ldh, int64_t psh, float* out, int64_t ldo, int64_t D, void* stream);
int spgnn_lstm_cell_bwd(int64_t t, int64_t n_t, int64_t n_next, const int32_t* perm, const float* g_out,
                        int64_t ldgo, const float* dh_rec, int64_t ldr, float* dc, uint16_t* gates, int64_t ldg,
                        int64_t psg, const float* c_prev, const float* c_cur, int64_t D, void* stream);
int spgnn_lstm_dp(const uint16_t* dgates, int64_t ldg, int64_t psg, const int64_t* off, const int32_t* rank,
                  const int32_t* in_ptr, const int32_t* out_ptr, const int32_t* out_dst, const int32_t* out_slot,
                  float* dP, int64_t lddp, int64_t n_src, int64_t D, void* stream);

/* Elementwise helpers the layer stacks need between projections.
 *   bias_act      : y = act(x + bias)           (GraphConv aggregate-first epilogue, GIN MLP, SAGE output)
 *   act_bwd       : dx = g * act'(y)  from the saved OUTPUT y (elu/tanh/relu/leaky all invertible this way)
 *   concat_dropout: out[:, :K1] = drop(x1), out[:, K1:K1+K2] = drop(x2), scaled by 1/(1-p); mask = hash(seed, idx)
 *                   (GATConv feat_drop on torch.cat([h_s,h_p]), models.py:431-435,477); bwd applies the same mask. */
int spgnn_bias_act(const float* x, int64_t ldx, const float* bias, int act, float slope,
                   float* y, int64_t ldy, int64_t M, int64_t N, void* stream);
int spgnn_act_bwd(const float* g, int64_t ldg, const float* y, int64_t ldy, int act, float slope,
                  float* dx, int64_t lddx, int64_t M, int64_t N, void* stream);
int spgnn_concat_dropout(const float* x1, int64_t ld1, int64_t K1, const float* x2, int64_t ld2, int64_t K2,
                         float p, uint64_t seed, float* out, int64_t ldo, int64_t M, void* stream);
int spgnn_concat_dropout_bwd(const float* g, int64_t ldg, int64_t K1, int64_t K2, float p, uint64_t seed,
                             float* d1, int64_t ldd1, float* d2, int64_t ldd2, int64_t M, void* stream);

/* ------------------------------------------------------------------------------------
 * Positional-encoding inits on device.
 *   anchor_select : job_runner.py:1727-1757 + :1712-1725 — softmax(fvs_out), 21 x masked column arg-max (first
 *                   max), then for the first 18 anchors the farthest descendant leaf in the DAG
 *                   {u->v : u<v adjacent} (ties -> largest index; the anchor itself when it has no descendant).
 *                   anchors int32 [B, pos_dim] LOCAL node ids; pos_dim in {21, 39}.
 *   pe_dist_init  : job_runner.py:1759-1777 — pos_enc[n,k] = hops(n, anchor_k)/diameter on the self-loop-free
 *                   graph; diam int32 [B]; flags[0] counts disconnected graphs.  Trees (symmetric, 2(n-1) non-self
 *                   edges, connected: every airway graph) take a kernel that runs the pos_dim anchor waves plus
 *                   two BFS for the diameter; any other graph takes the all-pairs bit-parallel BFS.  ws:
 *                   spgnn_pe_dist_ws_bytes(B, max_nodes) bytes, always required.
 *   pe_rw_init    : job_runner.py:1684-1702 — diag((A D^-1)^k), k=1..pos_dim, fp64 accumulate, fp32 out.
 * All take a batched adjacency (ptr, nbr; self loops are skipped) and node_off int64 [B+1].  pe_dist_init follows
 * nx shortest paths v -> anchor, so pass the OUT-CSR (out_ptr, out_dst); the others take the in-CSC.  For the
 * symmetric adjacencies the reference builds (dataset.py:418-419) the two are the same graph.
 * ---------------------------------------------------------------------------------- */
int spgnn_anchor_select(const float* fvs_out, int64_t ld, int64_t n_class,
                        const int64_t* node_off, const int32_t* in_ptr, const int32_t* in_src,
                        int64_t B, int64_t pos_dim, int64_t max_nodes, int32_t* anchors, void* stream);
int64_t spgnn_pe_dist_ws_bytes(int64_t B, int64_t max_nodes);
int spgnn_pe_dist_init(const int64_t* node_off, const int32_t* in_ptr, const int32_t* in_src,
                       const int32_t* anchors, int64_t B, int64_t pos_dim, int64_t max_nodes,
                       float* pos_enc, int64_t ldp, int32_t* diam, int32_t* flags, void* ws, void* stream);
int spgnn_pe_rw_init(const int64_t* node_off, const int32_t* in_ptr, const int32_t* in_src,
                     int64_t B, int64_t pos_dim, int64_t max_nodes, float* pos_enc, int64_t ldp, void* stream);

/* ------------------------------------------------------------------------------------
 * Decision rule and loss (callers of the path).
 *   segmented_argmax : job_runner.py:158-165 — per graph, per class c in [1, n_class): the node with the highest
 *                      softmax probability of class c (first max); out int64 [B, n_class-1] GLOBAL node ids.
 *   masked_ce_fwd/bwd: job_runner.py:1885-1900 — F.cross_entropy(out[mask], y[mask], weight): sums[0] = sum w*nll,
 *                      sums[1] = sum w over kept nodes (double[2], zeroed by the call); keep = (y != 0) || u01(hash(seed,node)) < rate, or an explicit
 *                      uint8 mask when mask != null.  bwd: dlogits = keep * w_y * (softmax - onehot) * (scale / sums[1]).
 * ---------------------------------------------------------------------------------- */
int spgnn_segmented_argmax(const float* logits, int64_t ld, int64_t n_class, const int64_t* node_off, int64_t B,
                           int64_t* out, void* stream);
int spgnn_masked_ce_fwd(const float* logits, int64_t ld, int64_t n_class, const int64_t* y, const uint8_t* mask,
                        float rate, uint64_t seed, const float* class_w, int64_t N, double* sums, void* stream);
int spgnn_masked_ce_bwd(const float* logits, int64_t ld, int64_t n_class, const int64_t* y, const uint8_t* mask,
                        float rate, uint64_t seed, const float* class_w, const double* sums, float scale,
                        int64_t N, float* dlogits, int64_t ldd, void* stream);
/* SGD with momentum over a flat bucket (torch.optim.SGD semantics: buf = mu*buf + g; p -= lr*buf). */
int spgnn_sgd_momentum(float* p, const float* g, float* buf, int64_t n, float lr, float mu, float grad_scale,
                       int first_step, void* stream);
/* Per-step salt of every dropout / sampling seed (seeds are kernel arguments: a step replayed from a CUDA graph would
 * repeat its masks).  Copies *dev_value (device memory, e.g. a step counter bumped by the first node of the captured
 * step) into the library's constant-memory salt, stream-ordered and capturable; every mask of the kernels that
 * follow uses seed + salt * 0x9E3779B97F4A7C15.  The salt is 0 until this is called.  spgnn_seed_salt_units: number
 * of translation units holding a copy (one memcpy node each). */
int spgnn_seed_salt_set(const uint64_t* dev_value, void* stream);
int spgnn_seed_salt_units(void);
/* The full update of torch.optim.SGD (the reference's optimiser, job_runner.py:239-249 with
 * exp_settings OPTIMIZER = {momentum, lr[, weight_decay, dampening, nesterov]}) over a contiguous range of the bucket:
 *   g = grad_scale*g + weight_decay*p;  buf = first_step ? g : mu*buf + (1-dampening)*g  (mu != 0);
 *   g = nesterov ? g + mu*buf : buf;  p -= lr*g.   buf may be null when mu == 0. */
int spgnn_sgd_step(float* p, const float* g, float* buf, int64_t n, float lr, float mu, float dampening,
                   float weight_decay, int nesterov, float grad_scale, int first_step, void* stream);
/* torch.optim.Adam (decoupled = 0) / AdamW (decoupled = 1) over the live chunks of a flat bucket, as torch's
 * _single_tensor_adam.  chunks: int64 [n_chunks, 3] = {offset, length, parameter index}, each chunk inside one
 * parameter and inside the buckets (not checked); live: int64 [n_live], the distinct indices of the parameters that
 * have a gradient this step.  steps: int64 per parameter, in device memory: the call first adds 1 to steps[live[i]]
 * (its own launch), then for every element of every chunk, with t = steps[parameter]:
 *   g = maximize ? -g : g;  Adam: g += weight_decay*p   AdamW: p *= 1 - lr*weight_decay   (weight_decay != 0);
 *   m = lerp(m, g, 1-beta1);  v = beta2*v + (1-beta2)*g^2;  amsgrad: vmax = max(vmax, v), used in place of v;
 *   p -= (lr / (1 - beta1^t)) * m / (sqrt(v) / sqrt(1 - beta2^t) + eps)   (bias corrections in fp64).
 * t never comes from the host, so a CUDA graph that captured this call advances it on every replay.  Elements
 * outside the chunks are not touched.  betas in [0, 1), lr, eps, weight_decay >= 0; max_exp_avg_sq non-null iff
 * amsgrad; p, g, exp_avg, exp_avg_sq, max_exp_avg_sq 16-byte aligned.  Two launches. */
int spgnn_adam_step(float* p, const float* g, float* exp_avg, float* exp_avg_sq, float* max_exp_avg_sq,
                    int64_t* steps, const int64_t* chunks, int64_t n_chunks, const int64_t* live, int64_t n_live,
                    double lr, double beta1, double beta2, double eps, double weight_decay, int amsgrad, int maximize,
                    int decoupled, void* stream);

/* ------------------------------------------------------------------------------------
 * Wire format of a scan batch (host loader -> device batch builder; replaces the dense per-scan H2D copies of
 * job_runner.py:1872-1875).  Lossless: the device decodes into the tensors the dense path builds, bit for bit.
 *   zero-suppressed rows: mask [rows, ceil(cols/32)] uint32 (bit b of word w: the fp32 BIT PATTERN of column 32w+b
 *                         is non-zero), vals = the non-zero values in row-major order, row_off int64 [rows + 1].
 *     spgnn_host_pack_rows_count : HOST code (no CUDA call): fills row_off, returns the number of values (-1: error).
 *     spgnn_host_pack_rows_fill  : HOST code: fills mask and vals.  threads <= 0: all hardware threads.
 *     spgnn_unpack_rows          : device: out fp32 [rows, ldo] (every column < cols written).
 *   edge lists: off-diagonal non-zeros of each scan's adjacency in row-major order (DGL edge order) as int32 LOCAL
 *               (src, dst); ne_off int64 [B + 1] = prefix of the per-scan counts.
 *     spgnn_edges_expand         : device: the int64 LOCAL edge lists spgnn_batch_build takes, with the N self
 *                                  loops appended last per graph (job_runner.py:1800), and n_edges int64 [B].
 * ---------------------------------------------------------------------------------- */
int64_t spgnn_host_pack_rows_count(const float* x, int64_t ldx, int64_t rows, int64_t cols, int64_t* row_off, int threads);
int spgnn_host_pack_rows_fill(const float* x, int64_t ldx, int64_t rows, int64_t cols, const int64_t* row_off,
                              uint32_t* mask, float* vals, int threads);
/* HOST code: dense adjacency blocks (uint8 [n_g, n_g], concatenated; job_runner.py:797 'adj') -> the int32 edge lists
 * above.  _count fills ne_off [B + 1] and returns the number of edges (-1: error); _fill writes them and the batch's
 * largest in-/out-degree INCLUDING the self loop the device appends. */
int64_t spgnn_host_adj_edges_count(const uint8_t* adj_cat, const int64_t* n_nodes, int64_t B, int64_t* ne_off, int threads);
int spgnn_host_adj_edges_fill(const uint8_t* adj_cat, const int64_t* n_nodes, int64_t B, const int64_t* ne_off,
                              int32_t* src, int32_t* dst, int32_t* max_degree, int threads);
int spgnn_unpack_rows(const uint32_t* mask, const float* vals, const int64_t* row_off, int64_t rows, int64_t cols,
                      float* out, int64_t ldo, void* stream);
int spgnn_edges_expand(const int32_t* src32, const int32_t* dst32, const int64_t* ne_off, const int64_t* node_off,
                       int64_t B, int64_t NE, int64_t N, int64_t* src_local, int64_t* dst_local, int64_t* n_edges,
                       void* stream);

/* ------------------------------------------------------------------------------------
 * Neighbour-sampled blocks for SAGE mini-batches (DGL MultiLayerNeighborSampler + to_block + the block CSC/CSR;
 * job_runner.py:1460-1514 via sampling.DeviceBlockSampler).  All L layers in one launch of one CTA, stream-ordered.
 *   graph    : in_ptr int32 [N+1], in_src int32 (in-CSC, ascending edge id per destination)
 *   seeds    : int64 [S] distinct node ids in [0, N) (checked on the device as well)
 *   per layer l (0 = input layer; the output layer L-1 is drawn first, its destinations are the seeds and every
 *   layer's destinations are the next layer's sources):
 *     fanouts_host[l]      : edges kept per destination, min(fanout, in-degree), uniformly without replacement;
 *                            -1 keeps all.  Key of CSC slot s: mix64(mix64(seed ^ mix64(salt ^ (l+1) << 56)) ^ s);
 *                            the `fanout` smallest (key, slot) pairs are kept, emitted in ascending slot order.
 *     caps_host[3l..3l+2]  : capacities {destinations, sources, edges} of the buffers below
 *     bufs_host[6l..6l+5]  : device addresses of in_ptr int32 [cap_dst+1], in_src int32 [cap_e] (local source ids),
 *                            out_ptr int32 [cap_src+1], out_dst int32 [cap_e], out_slot int32 [cap_e] (stable by
 *                            source; out_slot = position in the in-CSC), src_ids int64 [cap_src] (the destinations,
 *                            then every other source once in ascending id)
 *   pos      : int32 [N], all -1 on entry and on return (the call resets what it sets)
 *   edst_ws  : int32 [edst_cap >= largest cap_e]; keys_ws: uint64 [keys_cap], a power of two >= every cap_e and
 *              cap_src - cap_dst that exceeds 4096 (0 / null when none does)
 *   sizes    : int64 [2L+1]: (num_src, num_edges) of layer l at 2l, 2l+1; sizes[2L] = 0, or the error code when a
 *              capacity was too small (1), a seed was out of range (2) or repeated (3), in_src held a bad id (4).
 *              The caller reads it before trusting anything else.
 * gather_rows: out[r, :] = x[idx[r], :] in 32-bit words for r < min(cap, *count) (count null: r < cap); rows whose
 *              idx is outside [0, n_rows) are skipped. */
int spgnn_sample_blocks(const int32_t* in_ptr, const int32_t* in_src, int64_t N, const int64_t* seeds, int64_t S,
                        int64_t L, const int64_t* fanouts_host, const int64_t* caps_host, const int64_t* bufs_host,
                        uint64_t seed, uint64_t salt, int32_t* pos, int32_t* edst_ws, int64_t edst_cap,
                        uint64_t* keys_ws, int64_t keys_cap, int64_t* sizes, void* stream);
int spgnn_gather_rows(const void* x, int64_t ldx_words, int64_t n_rows, const int64_t* idx, const int64_t* count,
                      int64_t cap, int64_t words, void* out, int64_t ldo_words, void* stream);

/* ------------------------------------------------------------------------------------
 * Synthetic airway trees on device (bench input; integer part bit-identical to spgnn_b200/synth.py).
 * ---------------------------------------------------------------------------------- */
int spgnn_synth_trees(int64_t first_tree, int64_t B, uint32_t seed, int ragged, int64_t k_fixed,
                      const int64_t* node_off, int64_t* parent_local, int64_t* labels, void* stream);
int spgnn_synth_sizes(int64_t first_tree, int64_t B, uint32_t seed, int ragged, int64_t k_fixed,
                      int64_t* n_nodes, int64_t* n_edges, void* stream);
int spgnn_synth_edges(const int64_t* node_off, const int64_t* edge_off, const int64_t* parent_local, int64_t B,
                      int64_t* src_local, int64_t* dst_local, void* stream);
int spgnn_synth_features(int64_t first_tree, int64_t B, uint32_t seed, const int64_t* node_off, int64_t N,
                         float* fvs, int64_t ldf, int64_t fv_dim, float* fvs_out, int64_t ldo, int64_t n_class,
                         void* stream);

#ifdef __cplusplus
}
#endif
#endif /* SPGNN_B200_H */
