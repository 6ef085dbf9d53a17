/*
 * lac_b200.h -- C ABI of liblac_b200.so: the B200-native arithmetic-coding hot path of
 * pramasoul/lac (logits -> quantised integer CDF -> range-narrowing encode / decode).
 *
 * Every entry point takes plain pointers and sizes.  Pointers named d_* are DEVICE
 * pointers (cudaMalloc / torch tensor .data_ptr()); h_* are HOST pointers.  `stream` is a
 * cudaStream_t passed as void* (NULL = legacy default stream).  Calls are asynchronous on
 * that stream unless the name ends in _host (those synchronise before returning).
 * Return value: 0 (LAC_OK) or a negative lac_status; lac_last_error() has the text.
 *
 * There is no CPU implementation behind this ABI: without a CUDA device every compute
 * entry point returns LAC_E_CUDA.
 *
 * Reference interfaces replaced (pramasoul/lac):
 *   arith_code.py:117-128     ProbPredictor.calc_dist / dist        -> lac_cdf_build_f32
 *   llama_compress.py:24-30   Llama_AC.calc_dist (logits -> table)  -> lac_cdf_build_f32 / lac_cdf_lookup_f32
 *   arith_code.py:98-110      CDFPredictor.symbol_to_range          -> lac_cdf_lookup_f32, lac_ac_encode_logits_f32
 *   arith_code.py:169-219     A_to_bin.receive_symbol/step/flush/run/encode
 *                                                                   -> lac_ac_encode_logits_f32 / lac_ac_encode_pairs / lac_ac_encode_tables
 *   arith_code.py:94-97,248-334 CDFPredictor.val_to_symbol, A_from_bin -> lac_ac_decode_logits_f32 / lac_ac_decode_tables
 *   arith_code.py:336-351     group_bits / ungroup_bits             -> byte layout of every bitstream here (MSB first)
 *   arithmetic_coding.py:73-93,50-56,128-208,212-225 ACSampler compress path, flush_compress, Region, CarryBuffer,
 *                                                  packbits          -> lac_acs_encode_tables
 *   arithmetic_coding.py:94-124 ACSampler expand path               -> lac_acs_decode_tables
 *   arith_code.py:111-135     ProbPredictor with prob(s) = count of s -> lac_ac_encode_adaptive / lac_ac_decode_adaptive
 *                             (same counts under ACSampler)           -> lac_acs_encode_adaptive / lac_acs_decode_adaptive
 *
 * Workspace: the logits-driven calls need 256 * ceil(vocab / 32768) bytes of device scratch per logits row they
 * look at in one launch (lac_workspace_bytes).  Pass d_ws / ws_bytes to keep the call free of allocations (what a
 * per-token loop or a CUDA graph wants); with d_ws = NULL, or a workspace too small for the smallest launch (one
 * row for the row calls, n_streams rows for the stream calls), the call uses a stream-ordered allocation
 * (cudaMallocAsync) of at most 64 MB.  A workspace smaller than the full need is fine: the call then works through
 * the rows / tokens in several launches.
 */
#ifndef LAC_B200_H
#define LAC_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define LAC_ABI_VERSION 4

typedef enum {
    LAC_OK = 0,
    LAC_E_ARG = -1,     /* bad argument (NULL pointer, vocab / precision out of range, misaligned) */
    LAC_E_CUDA = -2,    /* CUDA runtime error or no device; see lac_last_error() */
    LAC_E_CAP = -3,     /* an output bitstream buffer was too small (reported via status words) */
    LAC_E_SYMBOL = -4,  /* a symbol id outside [0, vocab) */
    LAC_E_STREAM = -5   /* decoder: truncated or foreign bitstream (the reference raises at arith_code.py:277-278) */
} lac_status;

/* Per-stream status bits the kernels OR into the state words (lac_enc_state.status / lac_dec_state.status). */
#define LAC_ST_CAP 1u       /* output capacity exceeded: stream truncated */
#define LAC_ST_SYMBOL 2u    /* symbol out of range */
#define LAC_ST_TABLE 4u     /* unusable table (zero-width symbol / total 0) */
#define LAC_ST_TRUNC 8u     /* decoder: more bits consumed than the stream holds (truncated / foreign stream) */

int lac_abi_version(void);
const char *lac_last_error(void);
/* sm_count / cc = NULL allowed.  Returns LAC_E_CUDA when no device is usable. */
int lac_device_info(int *sm_count, int *cc_major, int *cc_minor, int64_t *hbm_bytes);

/* ------------------------------------------------------------------------------------
 * (a) logits -> LQ32 integer CDF (DESIGN.md section 3).  Fixed total 2^32, every symbol
 * frequency >= 1, bit-exact with oracle/lac_oracle.c:orc_lq32_cdf.
 *
 * d_logits  [rows] rows of `vocab` fp32, row r at d_logits + r * row_stride (elements)
 * vocab     1 .. 262144.  16-byte aligned rows (base aligned, vocab and strides multiples of 4) take the TMA
 *           path; anything else a scalar-load path with identical results.
 * ---------------------------------------------------------------------------------- */

/* Device scratch (bytes) that lets a logits-driven call over `rows` rows run in one launch without allocating. */
int64_t lac_workspace_bytes(int64_t rows, int32_t vocab);

/* Full table: d_cum[r * vocab + i] = exclusive cumulative frequency of symbol i (cum[0] = 0;
 * the total 2^32 is implicit).  Replaces calc_dist (llama_compress.py:24-30). */
int lac_cdf_build_f32(const float *d_logits, int64_t rows, int32_t vocab, int64_t row_stride,
                      uint32_t *d_cum, void *d_ws, int64_t ws_bytes, void *stream);

/* Encode-side lookup: for row r and symbol d_syms[r] write d_pairs[2r] = cum[sym],
 * d_pairs[2r+1] = cum[sym+1] (0 encodes 2^32 for the last symbol).  One HBM pass over the logits
 * (row summaries) plus one warp per row; the table itself is never written to memory.  Replaces calc_dist +
 * symbol_to_range's table reads.  A symbol outside [0, vocab) yields the pair (0xFFFFFFFF, 0xFFFFFFFF), which
 * lac_ac_encode_pairs turns into LAC_ST_SYMBOL on the stream, and sets LAC_ST_SYMBOL in d_status[r] (optional). */
int lac_cdf_lookup_f32(const float *d_logits, int64_t rows, int32_t vocab, int64_t row_stride,
                       const int32_t *d_syms, uint32_t *d_pairs, uint32_t *d_status, void *d_ws,
                       int64_t ws_bytes, void *stream);

/* ------------------------------------------------------------------------------------
 * (b) batched multi-stream range coder, arith_code.A_to_bin / A_from_bin semantics.
 * One independent coder per stream; `prec` is AC(..., prec) (reference default 16,
 * llama_compress.py uses 48).  Bitstreams are MSB-first bytes == bytes(group_bits(bits)).
 * ---------------------------------------------------------------------------------- */

/* Encoder state, one per stream, device resident, initialise with lac_enc_init. */
typedef struct {
    int64_t low;      /* A_to_bin.l */
    int64_t high;     /* A_to_bin.h */
    uint64_t nbits;   /* bits emitted so far (A_to_bin.emitted_bits) */
    uint32_t status;  /* LAC_ST_* */
    uint32_t _pad;
} lac_enc_state;

/* Decoder state, one per stream. */
typedef struct {
    int64_t low;      /* A_from_bin.l */
    int64_t high;     /* A_from_bin.h */
    int64_t value;    /* code value in the same coordinates (replaces the lb/hb window, arith_code.py:264-267) */
    uint64_t pos;     /* next bit of the stream to read */
    uint32_t status;
    uint32_t _pad;
} lac_dec_state;

int lac_enc_init(lac_enc_state *d_state, int64_t n_streams, int prec, void *stream);
/* d_offsets: n_streams + 1 byte offsets into d_bytes (stream s = [off[s], off[s+1])). */
int lac_dec_init(lac_dec_state *d_state, int64_t n_streams, int prec, const uint8_t *d_bytes,
                 const int64_t *d_offsets, void *stream);

/* Encode `T` tokens per stream from (lo, hi) pairs on the fixed total 2^32 (the output of
 * lac_cdf_lookup_f32; prec must be >= 34 so symbol_to_range's unfudged branch applies).
 * Pair of (stream s, token t) at d_pairs + 2 * (s * stream_stride + t * tok_stride).
 * d_ntok (optional): per-stream token counts <= T for ragged batches.
 * Stream s writes bytes to d_out + s * out_stride; at most out_stride bytes.
 * finish != 0: run A_to_bin.flush() and zero-pad the last byte; d_state[s].nbits is the
 * stream length in bits. */
int lac_ac_encode_pairs(const uint32_t *d_pairs, int64_t n_streams, int64_t T, int64_t stream_stride,
                        int64_t tok_stride, const int32_t *d_ntok, lac_enc_state *d_state,
                        uint8_t *d_out, int64_t out_stride, int finish, int prec, void *stream);

/* Encode straight from logits: one HBM pass over the logits (row summaries) and ONE fused kernel that looks up
 * (cum[sym], cum[sym + 1]) of every coded symbol and runs the range coder; the pairs never reach global memory.
 * Token t of stream s reads the logits row at d_logits + s * stream_stride + t * tok_stride (elements) and the
 * symbol d_syms[s * sym_stride + t].  T = 1 is the model-in-the-loop step.  T = 0 with finish != 0 only flushes.
 * Everything else as for lac_ac_encode_pairs.  Rows past a stream's d_ntok count are not coded but may be read. */
int lac_ac_encode_logits_f32(const float *d_logits, int64_t n_streams, int64_t T, int64_t stream_stride,
                             int64_t tok_stride, int32_t vocab, const int32_t *d_syms, int64_t sym_stride,
                             const int32_t *d_ntok, lac_enc_state *d_state, uint8_t *d_out, int64_t out_stride,
                             int finish, int prec, void *d_ws, int64_t ws_bytes, void *stream);

/* Decode (one HBM pass over the logits for the row summaries, then one warp per stream): for every
 * stream, T sequential tokens; token t of stream s reads the logits row at
 * d_logits + s * stream_stride + t * tok_stride (elements), rebuilds the LQ32 CDF on chip, finds the symbol containing the code value (val_to_symbol), narrows (l, h) and
 * renormalises from the stream's bits.  Symbols go to d_syms[s * sym_stride + t].
 * T = 1 is the model-in-the-loop step.  A stream from which more bits were consumed than it holds gets
 * LAC_ST_TRUNC in d_state[s].status (lac_dec_status collects it).  Rows past a stream's d_ntok count are not
 * decoded but may be read. */
int lac_ac_decode_logits_f32(const float *d_logits, int64_t n_streams, int64_t T, int64_t stream_stride,
                             int64_t tok_stride, int32_t vocab, const int32_t *d_ntok,
                             lac_dec_state *d_state, const uint8_t *d_bytes, const int64_t *d_offsets,
                             int32_t *d_syms, int64_t sym_stride, int prec, void *d_ws, int64_t ws_bytes,
                             void *stream);

/* OR of the status words of n_streams encoder / decoder states, written to *d_or (device, 4 bytes): one small
 * kernel, so a caller can check a whole batch with a single 4-byte read. */
int lac_enc_status(const lac_enc_state *d_state, int64_t n_streams, uint32_t *d_or, void *stream);
int lac_dec_status(const lac_dec_state *d_state, int64_t n_streams, uint32_t *d_or, void *stream);

/* ------------------------------------------------------------------------------------
 * The reference's uniform base class Predictor(n) (arith_code.py:64-74): symbol s of n maps to
 * [floor(s w / n), floor((s + 1) w / n)).  AC() without arguments is AC(Predictor(3), 16).
 * Symbols int32 at d_syms[s * sym_stride + t]; everything else as for the pair / table coders.
 * Streams whose interval is narrower than n symbols set LAC_ST_TABLE (the reference never
 * terminates there); decode returns the symbol whose range holds the code value.
 * ---------------------------------------------------------------------------------- */
int lac_ac_encode_uniform(const int32_t *d_syms, int64_t n_streams, int64_t T, int64_t sym_stride,
                          const int32_t *d_ntok, int32_t n_symbols, lac_enc_state *d_state,
                          uint8_t *d_out, int64_t out_stride, int finish, int prec, void *stream);
int lac_ac_decode_uniform(int64_t n_streams, int64_t T, const int32_t *d_ntok, int32_t n_symbols,
                          lac_dec_state *d_state, const uint8_t *d_bytes, const int64_t *d_offsets,
                          int32_t *d_syms, int64_t sym_stride, int prec, void *stream);

/* ------------------------------------------------------------------------------------
 * General integer tables ("given identical integer frequency tables the bitstream is
 * bit-exact with the reference coder"): int64 inclusive cumulative tables exactly as
 * CDFPredictor.dist holds them, any total < 2^63, including the fudged_dist rescale
 * (arith_code.py:83-93).  Table of (stream s, token t) at
 * d_dist + s * stream_stride + t * tok_stride (elements); strides of 0 share tables.
 * d_minp: predictor.minp per table, same indexing with strides divided by vocab
 * (minp index = s * minp_stream_stride + t * minp_tok_stride).
 * Symbols int32 at d_syms[s * sym_stride + t].
 * flags: LAC_F_WRAP64 reproduces Llama_AC's numpy-int64 overflow in fudged_dist.
 * ---------------------------------------------------------------------------------- */
#define LAC_F_WRAP64 1

int lac_ac_encode_tables(const int64_t *d_dist, int32_t vocab, int64_t stream_stride, int64_t tok_stride,
                         const int64_t *d_minp, int64_t minp_stream_stride, int64_t minp_tok_stride,
                         const int32_t *d_syms, int64_t sym_stride, int64_t n_streams, int64_t T,
                         const int32_t *d_ntok, lac_enc_state *d_state, uint8_t *d_out, int64_t out_stride,
                         int finish, int prec, int flags, void *stream);

int lac_ac_decode_tables(const int64_t *d_dist, int32_t vocab, int64_t stream_stride, int64_t tok_stride,
                         const int64_t *d_minp, int64_t minp_stream_stride, int64_t minp_tok_stride,
                         int64_t n_streams, int64_t T, const int32_t *d_ntok, lac_dec_state *d_state,
                         const uint8_t *d_bytes, const int64_t *d_offsets, int32_t *d_syms,
                         int64_t sym_stride, int prec, int flags, void *stream);

/* ACSampler semantics (arithmetic_coding.py): uint64 inclusive cumulative tables as
 * sample_scaled_cdf receives them, denominator = table[-1].
 * finish = 1: flush_compress() + packbits.flush(), bit-exact with the reference.  That flush
 *   does not pin the final interval, so the last tokens of such a stream can be undecodable
 *   by any decoder (the reference's own expand path round-trips 16 of the 30 golden cases).
 * finish = 2: safe termination (A_to_bin.flush on the Region state): always decodable.
 * The decoder returns the symbol whose encoder interval contains the zero-padded code value
 * (DESIGN.md section 6). */
int lac_acs_encode_tables(const uint64_t *d_cdf, int32_t vocab, int64_t stream_stride, int64_t tok_stride,
                          const int32_t *d_syms, int64_t sym_stride, int64_t n_streams, int64_t T,
                          const int32_t *d_ntok, lac_enc_state *d_state, uint8_t *d_out, int64_t out_stride,
                          int finish, int prec, void *stream);

int lac_acs_decode_tables(const uint64_t *d_cdf, int32_t vocab, int64_t stream_stride, int64_t tok_stride,
                          int64_t n_streams, int64_t T, const int32_t *d_ntok, lac_dec_state *d_state,
                          const uint8_t *d_bytes, const int64_t *d_offsets, int32_t *d_syms,
                          int64_t sym_stride, int prec, void *stream);

/* ------------------------------------------------------------------------------------
 * Adaptive frequency models: prob(s) = counts[s], and after every coded or decoded token
 * counts[sym] += inc (the reference predictor reads its table, then accepts the symbol).
 * The counts live on the device: int64 [n_streams][vocab], stream s at d_counts + s * vocab,
 * read at entry and written back at exit, so a stream can be fed in several calls.  Encoder and
 * decoder each need their own copy, starting from the same counts.
 *   lac_ac_*:  CDFPredictor semantics on dist = inclusive cumsum(counts), minp = the smallest
 *              positive count, fudged_dist when dist[-1] > w * minp (arith_code.py:83-135).
 *   lac_acs_*: ACSampler semantics on cdf = cumsum(counts); finish as lac_acs_encode_tables.
 * Bounds: 1 <= vocab <= LAC_ADAPTIVE_MAX_VOCAB, inc >= 0 (0: a static table).  A stream stops
 * with LAC_ST_TABLE, the others going on, on a negative count, a table total that would reach
 * 2^62, a symbol of zero width or a zero total; LAC_ST_SYMBOL on a symbol outside [0, vocab).
 * Counts advance for exactly the tokens that narrowed the interval, so a stopped stream's state
 * and counts stay a consistent pair.  Everything else as for the table coders.
 * ---------------------------------------------------------------------------------- */
#define LAC_ADAPTIVE_MAX_VOCAB 4096

int lac_ac_encode_adaptive(int64_t *d_counts, int32_t vocab, int64_t inc, const int32_t *d_syms, int64_t sym_stride,
                           int64_t n_streams, int64_t T, const int32_t *d_ntok, lac_enc_state *d_state,
                           uint8_t *d_out, int64_t out_stride, int finish, int prec, void *stream);
int lac_ac_decode_adaptive(int64_t *d_counts, int32_t vocab, int64_t inc, int64_t n_streams, int64_t T,
                           const int32_t *d_ntok, lac_dec_state *d_state, const uint8_t *d_bytes,
                           const int64_t *d_offsets, int32_t *d_syms, int64_t sym_stride, int prec, void *stream);
int lac_acs_encode_adaptive(int64_t *d_counts, int32_t vocab, int64_t inc, const int32_t *d_syms, int64_t sym_stride,
                            int64_t n_streams, int64_t T, const int32_t *d_ntok, lac_enc_state *d_state,
                            uint8_t *d_out, int64_t out_stride, int finish, int prec, void *stream);
int lac_acs_decode_adaptive(int64_t *d_counts, int32_t vocab, int64_t inc, int64_t n_streams, int64_t T,
                            const int32_t *d_ntok, lac_dec_state *d_state, const uint8_t *d_bytes,
                            const int64_t *d_offsets, int32_t *d_syms, int64_t sym_stride, int prec, void *stream);

/* ------------------------------------------------------------------------------------
 * (e) batch-invariant model kernels: the layers of a Llama-style decoder (llama_compress.LlamaModel with
 * batch_invariant=True).  bf16 activations and weights, fp32 accumulation, row-major tensors.
 *
 * Invariance contract: the bits of output row r depend only on row r's inputs, the weights and, for attention,
 * the KV cache up to that row's position.  They never depend on M, on the number of query positions a launch
 * covers, or on which CTA (or which row of a tile) computes the row.  So a prefill launch over T_blk positions
 * of S streams (M = T_blk * S, row t * S + s) reproduces, bit for bit, the rows a per-token step computes with
 * M = S.
 *
 * Activations are position-major: row r = t * S + s is stream s at position base + t, where base = *d_pos when
 * d_pos (device, one int64) is given -- the per-token step, so one CUDA graph serves every position -- and p0
 * otherwise.  The KV cache is [S, kv_heads, max_len, hd] bf16; qkv rows are [heads | kv_heads | kv_heads] x hd.
 * A launch with S = n streams may run on the first n streams of a larger cache (they are a prefix of it).
 * ---------------------------------------------------------------------------------- */
#define LAC_MODEL_OUT_BF16 0      /* y = bf16(x @ w) */
#define LAC_MODEL_OUT_BF16_ADD 1  /* y = bf16(res + bf16(x @ w)); y may be res */
#define LAC_MODEL_OUT_F32 2       /* y = x @ w in fp32 (the logits) */

/* Y[M, N] = X[M, K] @ W[K, N] on tcgen05 (TMA ring, accumulator in tensor memory), tile 128 x 128 x 64 (M <= 128:
 * 128 x 64 x 64 with a deeper ring when N / 64 CTAs fit one wave; the same bits per row), K in one ascending pass.
 * N a multiple of 128 and K a multiple of 64 (every CONFIGS geometry); other shapes return LAC_E_ARG.  All pointers
 * 16-byte aligned. */
int lac_model_gemm(const void *d_x, const void *d_w, int64_t M, int32_t N, int32_t K, int epilogue,
                   const void *d_res, void *d_y, void *stream);
/* y = bf16(x * rsqrt(mean(x^2) + eps)) per row; dim a multiple of 256. */
int lac_model_rmsnorm(const void *d_x, int64_t rows, int32_t dim, float eps, void *d_y, void *stream);
/* Rotate-half RoPE of the q and k heads of every qkv row in place, from the [max_len, hd] bf16 tables, and write
 * k and v to the cache at the row's position.  rows a multiple of n_streams. */
int lac_model_rope_kv(void *d_qkv, int64_t rows, int32_t n_streams, int32_t heads, int32_t kv_heads, int32_t hd,
                      const void *d_cos, const void *d_sin, const int64_t *d_pos, int64_t p0, void *d_kc,
                      void *d_vc, int32_t max_len, void *stream);
/* y[r, j] = bf16(bf16(silu(h[r, j])) * h[r, ffn + j]) for h [rows, 2 * ffn]. */
int lac_model_swiglu(const void *d_h, int64_t rows, int32_t ffn, void *d_y, void *stream);
/* Causal GQA attention of n_q query positions per stream (the roped q of qkv) over the KV cache, hd 64 or 128:
 * out [n_q * S, heads * hd].  Each query visits 64-key blocks from slot 0 in order, fp32 online softmax with
 * exp2, and skips per row the blocks past its position. */
int lac_model_attention(const void *d_qkv, int32_t n_streams, int32_t n_q, int32_t heads, int32_t kv_heads,
                        int32_t hd, const int64_t *d_pos, int64_t p0, const void *d_kc, const void *d_vc,
                        int32_t max_len, void *d_out, void *stream);

/* ------------------------------------------------------------------------------------
 * Host-buffer convenience calls (what bench.py's `e2e` times): pinned or pageable HOST
 * buffers in, HOST buffers out, copies + kernels + synchronisation inside.  The logits go to the current
 * device in <= 256 MB pieces over two staging buffers and two streams, so the copy of piece k + 1 overlaps the
 * kernels of piece k; the call is PCIe-bound (4 * vocab bytes per token each way).
 * ---------------------------------------------------------------------------------- */

/* Encode n_streams x T tokens from host logits [n_streams, T, vocab] and host symbols
 * [n_streams, T].  h_out: n_streams * out_stride bytes; h_nbits: n_streams stream lengths. */
int lac_encode_logits_host(const float *h_logits, const int32_t *h_syms, int64_t n_streams, int64_t T,
                           int32_t vocab, uint8_t *h_out, int64_t out_stride, uint64_t *h_nbits, int prec);

/* Decode them back.  h_offsets: n_streams + 1 byte offsets into h_bytes (checked: start at 0, non-decreasing).
 * Returns LAC_E_STREAM when a stream was truncated / foreign. */
int lac_decode_logits_host(const float *h_logits, int64_t n_streams, int64_t T, int32_t vocab,
                           const uint8_t *h_bytes, const int64_t *h_offsets, int32_t *h_syms, int prec);

#ifdef __cplusplus
}
#endif
#endif /* LAC_B200_H */
