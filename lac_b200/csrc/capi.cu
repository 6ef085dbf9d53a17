// capi.cu -- extern "C" entry points of liblac_b200.so (include/lac_b200.h).
// Argument checking, launch, error text.  No CPU compute path exists here: every entry
// point either launches CUDA work or fails with LAC_E_CUDA.
#include <cstdarg>
#include <cstdio>
#include <cstring>
#include <mutex>
#include <string>
#include <cuda_runtime.h>

#include "launch.h"
#include "lq32.cuh"

namespace lac {
cudaError_t launch_status_or(const void* state, int64_t n, int stride_words, int status_word, uint32_t* d_or,
                             cudaStream_t st);
}

namespace {

thread_local std::string g_err;

int fail(int code, const char* fmt, ...) {
    char buf[512];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof buf, fmt, ap);
    va_end(ap);
    g_err = buf;
    return code;
}
int cuda_fail(cudaError_t e, const char* what) {
    return fail(LAC_E_CUDA, "%s: %s", what, cudaGetErrorString(e));
}
#define CK(call, what)                                  \
    do {                                                \
        cudaError_t e__ = (call);                       \
        if (e__ != cudaSuccess) return cuda_fail(e__, what); \
    } while (0)

bool prec_ok(int prec, int lo) { return prec >= lo && prec <= 60; }

int check_vocab(int32_t vocab) {
    if (vocab < 1 || vocab > lac::max_vocab())
        return fail(LAC_E_ARG, "vocab %d out of range [1, %d]", vocab, lac::max_vocab());
    return LAC_OK;
}
bool ws_ok(const void* ws, int64_t ws_bytes) { return ws_bytes >= 0 && (ws || ws_bytes == 0); }

}  // namespace

extern "C" {

int lac_abi_version(void) { return LAC_ABI_VERSION; }
const char* lac_last_error(void) { return g_err.c_str(); }

int lac_device_info(int* sm_count, int* cc_major, int* cc_minor, int64_t* hbm_bytes) {
    int dev = 0;
    CK(cudaGetDevice(&dev), "cudaGetDevice");
    cudaDeviceProp p;
    CK(cudaGetDeviceProperties(&p, dev), "cudaGetDeviceProperties");
    if (sm_count) *sm_count = p.multiProcessorCount;
    if (cc_major) *cc_major = p.major;
    if (cc_minor) *cc_minor = p.minor;
    if (hbm_bytes) *hbm_bytes = (int64_t)p.totalGlobalMem;
    return LAC_OK;
}

int64_t lac_workspace_bytes(int64_t rows, int32_t vocab) {
    if (rows < 0 || vocab < 1 || vocab > lac::max_vocab()) return 0;
    const int parts = lq::parts_of(vocab);
    const int64_t chunk = lac::summ_chunk_rows(parts);
    return (int64_t)lac::summ_bytes(rows < chunk ? (rows < 1 ? 1 : rows) : chunk, parts);
}

int lac_cdf_build_f32(const float* d_logits, int64_t rows, int32_t vocab, int64_t row_stride, uint32_t* d_cum,
                      void* d_ws, int64_t ws_bytes, void* stream) {
    if (!d_logits || !d_cum || rows < 0 || row_stride < vocab || !ws_ok(d_ws, ws_bytes))
        return fail(LAC_E_ARG, "lac_cdf_build_f32: bad argument");
    if (int rc = check_vocab(vocab)) return rc;
    CK(lac::launch_build(d_logits, rows, vocab, row_stride, d_cum, d_ws, (size_t)ws_bytes, (cudaStream_t)stream),
       "lac_cdf_build_f32");
    return LAC_OK;
}

int lac_cdf_lookup_f32(const float* d_logits, int64_t rows, int32_t vocab, int64_t row_stride, const int32_t* d_syms,
                       uint32_t* d_pairs, uint32_t* d_status, void* d_ws, int64_t ws_bytes, void* stream) {
    if (!d_logits || !d_syms || !d_pairs || rows < 0 || row_stride < vocab || !ws_ok(d_ws, ws_bytes))
        return fail(LAC_E_ARG, "lac_cdf_lookup_f32: bad argument");
    if (int rc = check_vocab(vocab)) return rc;
    if ((uintptr_t)d_pairs & 7) return fail(LAC_E_ARG, "lac_cdf_lookup_f32: d_pairs must be 8-byte aligned");
    CK(lac::launch_lookup(d_logits, rows, vocab, row_stride, d_syms, d_pairs, d_status, d_ws, (size_t)ws_bytes,
                          (cudaStream_t)stream),
       "lac_cdf_lookup_f32");
    return LAC_OK;
}

int lac_enc_init(lac_enc_state* d_state, int64_t n_streams, int prec, void* stream) {
    if (!d_state || n_streams < 0 || !prec_ok(prec, 2)) return fail(LAC_E_ARG, "lac_enc_init: bad argument");
    CK(lac::launch_enc_init(d_state, n_streams, prec, (cudaStream_t)stream), "lac_enc_init");
    return LAC_OK;
}

int lac_dec_init(lac_dec_state* d_state, int64_t n_streams, int prec, const uint8_t* d_bytes,
                 const int64_t* d_offsets, void* stream) {
    if (!d_state || !d_bytes || !d_offsets || n_streams < 0 || !prec_ok(prec, 2))
        return fail(LAC_E_ARG, "lac_dec_init: bad argument");
    CK(lac::launch_dec_init(d_state, n_streams, prec, d_bytes, d_offsets, (cudaStream_t)stream), "lac_dec_init");
    return LAC_OK;
}

int lac_ac_encode_pairs(const uint32_t* d_pairs, int64_t n_streams, int64_t T, int64_t stream_stride,
                        int64_t tok_stride, const int32_t* d_ntok, lac_enc_state* d_state, uint8_t* d_out,
                        int64_t out_stride, int finish, int prec, void* stream) {
    if ((!d_pairs && T > 0) || !d_state || !d_out || n_streams < 0 || T < 0 || out_stride < 1)
        return fail(LAC_E_ARG, "lac_ac_encode_pairs: bad argument");
    if (!prec_ok(prec, 34)) return fail(LAC_E_ARG, "lac_ac_encode_pairs: prec %d outside [34, 60]", prec);
    if ((uintptr_t)d_pairs & 7) return fail(LAC_E_ARG, "lac_ac_encode_pairs: d_pairs must be 8-byte aligned");
    CK(lac::launch_encode_pairs(d_pairs, n_streams, T, stream_stride, tok_stride, d_ntok, 0, d_state, d_out,
                                out_stride, finish, prec, (cudaStream_t)stream),
       "lac_ac_encode_pairs");
    return LAC_OK;
}

int lac_ac_encode_logits_f32(const float* d_logits, int64_t n_streams, int64_t T, int64_t stream_stride,
                             int64_t tok_stride, int32_t vocab, const int32_t* d_syms, int64_t sym_stride,
                             const int32_t* d_ntok, lac_enc_state* d_state, uint8_t* d_out, int64_t out_stride,
                             int finish, int prec, void* d_ws, int64_t ws_bytes, void* stream) {
    if (((!d_logits || !d_syms) && T > 0) || !d_state || !d_out || n_streams < 0 || T < 0 || out_stride < 1 ||
        !ws_ok(d_ws, ws_bytes))
        return fail(LAC_E_ARG, "lac_ac_encode_logits_f32: bad argument");
    if (!prec_ok(prec, 34)) return fail(LAC_E_ARG, "lac_ac_encode_logits_f32: prec %d outside [34, 60]", prec);
    if (int rc = check_vocab(vocab)) return rc;
    CK(lac::launch_encode_logits(d_logits, n_streams, T, stream_stride, tok_stride, vocab, d_syms, sym_stride, d_ntok,
                                 d_state, d_out, out_stride, finish, prec, d_ws, (size_t)ws_bytes, (cudaStream_t)stream),
       "lac_ac_encode_logits_f32");
    return LAC_OK;
}

int lac_ac_decode_logits_f32(const float* d_logits, int64_t n_streams, int64_t T, int64_t stream_stride,
                             int64_t tok_stride, int32_t vocab, const int32_t* d_ntok, lac_dec_state* d_state,
                             const uint8_t* d_bytes, const int64_t* d_offsets, int32_t* d_syms, int64_t sym_stride,
                             int prec, void* d_ws, int64_t ws_bytes, void* stream) {
    if ((!d_logits && T > 0) || !d_state || !d_bytes || !d_offsets || (!d_syms && T > 0) || n_streams < 0 || T < 0 ||
        !ws_ok(d_ws, ws_bytes))
        return fail(LAC_E_ARG, "lac_ac_decode_logits_f32: bad argument");
    if (!prec_ok(prec, 34)) return fail(LAC_E_ARG, "lac_ac_decode_logits_f32: prec %d outside [34, 60]", prec);
    if (int rc = check_vocab(vocab)) return rc;
    CK(lac::launch_decode(d_logits, n_streams, T, stream_stride, tok_stride, vocab, d_ntok, d_state, d_bytes,
                          d_offsets, d_syms, sym_stride, prec, d_ws, (size_t)ws_bytes, (cudaStream_t)stream),
       "lac_ac_decode_logits_f32");
    return LAC_OK;
}

int lac_enc_status(const lac_enc_state* d_state, int64_t n_streams, uint32_t* d_or, void* stream) {
    if (!d_state || !d_or || n_streams < 0) return fail(LAC_E_ARG, "lac_enc_status: bad argument");
    CK(lac::launch_status_or(d_state, n_streams, (int)(sizeof(lac_enc_state) / 4), 6, d_or, (cudaStream_t)stream),
       "lac_enc_status");
    return LAC_OK;
}
int lac_dec_status(const lac_dec_state* d_state, int64_t n_streams, uint32_t* d_or, void* stream) {
    if (!d_state || !d_or || n_streams < 0) return fail(LAC_E_ARG, "lac_dec_status: bad argument");
    CK(lac::launch_status_or(d_state, n_streams, (int)(sizeof(lac_dec_state) / 4), 8, d_or, (cudaStream_t)stream),
       "lac_dec_status");
    return LAC_OK;
}

int lac_ac_encode_uniform(const int32_t* d_syms, int64_t n_streams, int64_t T, int64_t sym_stride,
                          const int32_t* d_ntok, int32_t n_symbols, lac_enc_state* d_state, uint8_t* d_out,
                          int64_t out_stride, int finish, int prec, void* stream) {
    if ((!d_syms && T > 0) || !d_state || !d_out || n_streams < 0 || T < 0 || out_stride < 1 || n_symbols < 1)
        return fail(LAC_E_ARG, "lac_ac_encode_uniform: bad argument");
    if (!prec_ok(prec, 2)) return fail(LAC_E_ARG, "lac_ac_encode_uniform: prec %d outside [2, 60]", prec);
    CK(lac::launch_table_encode(lac::Uniform{n_symbols}, d_syms, sym_stride, n_streams, T, d_ntok, d_state, d_out,
                                out_stride, finish ? lac::kFlushAc : lac::kFlushNone, prec, (cudaStream_t)stream),
       "lac_ac_encode_uniform");
    return LAC_OK;
}

int lac_ac_decode_uniform(int64_t n_streams, int64_t T, const int32_t* d_ntok, int32_t n_symbols,
                          lac_dec_state* d_state, const uint8_t* d_bytes, const int64_t* d_offsets, int32_t* d_syms,
                          int64_t sym_stride, int prec, void* stream) {
    if (!d_state || !d_bytes || !d_offsets || (!d_syms && T > 0) || n_streams < 0 || T < 0 || n_symbols < 1)
        return fail(LAC_E_ARG, "lac_ac_decode_uniform: bad argument");
    if (!prec_ok(prec, 2)) return fail(LAC_E_ARG, "lac_ac_decode_uniform: prec %d outside [2, 60]", prec);
    CK(lac::launch_table_decode(lac::Uniform{n_symbols}, n_streams, T, d_ntok, d_state, d_bytes, d_offsets, d_syms,
                                sym_stride, prec, (cudaStream_t)stream),
       "lac_ac_decode_uniform");
    return LAC_OK;
}

int lac_ac_encode_tables(const int64_t* d_dist, int32_t vocab, int64_t stream_stride, int64_t tok_stride,
                         const int64_t* d_minp, int64_t minp_stream_stride, int64_t minp_tok_stride,
                         const int32_t* d_syms, int64_t sym_stride, int64_t n_streams, int64_t T,
                         const int32_t* d_ntok, lac_enc_state* d_state, uint8_t* d_out, int64_t out_stride, int finish,
                         int prec, int flags, void* stream) {
    if (!d_dist || !d_minp || (!d_syms && T > 0) || !d_state || !d_out || vocab < 1 || n_streams < 0 || T < 0 ||
        out_stride < 1)
        return fail(LAC_E_ARG, "lac_ac_encode_tables: bad argument");
    if (!prec_ok(prec, 2)) return fail(LAC_E_ARG, "lac_ac_encode_tables: prec %d outside [2, 60]", prec);
    const lac::Cdf m{vocab, d_dist, stream_stride, tok_stride, d_minp, minp_stream_stride, minp_tok_stride, flags};
    CK(lac::launch_table_encode(m, d_syms, sym_stride, n_streams, T, d_ntok, d_state, d_out, out_stride,
                                finish ? lac::kFlushAc : lac::kFlushNone, prec, (cudaStream_t)stream),
       "lac_ac_encode_tables");
    return LAC_OK;
}

int lac_ac_decode_tables(const int64_t* d_dist, int32_t vocab, int64_t stream_stride, int64_t tok_stride,
                         const int64_t* d_minp, int64_t minp_stream_stride, int64_t minp_tok_stride,
                         int64_t n_streams, int64_t T, const int32_t* d_ntok, lac_dec_state* d_state,
                         const uint8_t* d_bytes, const int64_t* d_offsets, int32_t* d_syms, int64_t sym_stride,
                         int prec, int flags, void* stream) {
    if (!d_dist || !d_minp || !d_state || !d_bytes || !d_offsets || !d_syms || vocab < 1 || n_streams < 0 || T < 0)
        return fail(LAC_E_ARG, "lac_ac_decode_tables: bad argument");
    if (!prec_ok(prec, 2)) return fail(LAC_E_ARG, "lac_ac_decode_tables: prec %d outside [2, 60]", prec);
    const lac::Cdf m{vocab, d_dist, stream_stride, tok_stride, d_minp, minp_stream_stride, minp_tok_stride, flags};
    CK(lac::launch_table_decode(m, n_streams, T, d_ntok, d_state, d_bytes, d_offsets, d_syms, sym_stride, prec,
                                (cudaStream_t)stream),
       "lac_ac_decode_tables");
    return LAC_OK;
}

int lac_acs_encode_tables(const uint64_t* d_cdf, int32_t vocab, int64_t stream_stride, int64_t tok_stride,
                          const int32_t* d_syms, int64_t sym_stride, int64_t n_streams, int64_t T,
                          const int32_t* d_ntok, lac_enc_state* d_state, uint8_t* d_out, int64_t out_stride, int finish,
                          int prec, void* stream) {
    if (!d_cdf || (!d_syms && T > 0) || !d_state || !d_out || vocab < 1 || n_streams < 0 || T < 0 || out_stride < 1)
        return fail(LAC_E_ARG, "lac_acs_encode_tables: bad argument");
    if (!prec_ok(prec, 2)) return fail(LAC_E_ARG, "lac_acs_encode_tables: prec %d outside [2, 60]", prec);
    // finish 1: flush_compress (the reference's), 2: the safe termination, anything else: no flush
    const int flush = finish == 1 ? lac::kFlushCompress : (finish == 2 ? lac::kFlushAc : lac::kFlushNone);
    CK(lac::launch_table_encode(lac::Acs{vocab, d_cdf, stream_stride, tok_stride}, d_syms, sym_stride, n_streams, T,
                                d_ntok, d_state, d_out, out_stride, flush, prec, (cudaStream_t)stream),
       "lac_acs_encode_tables");
    return LAC_OK;
}

int lac_acs_decode_tables(const uint64_t* d_cdf, int32_t vocab, int64_t stream_stride, int64_t tok_stride,
                          int64_t n_streams, int64_t T, const int32_t* d_ntok, lac_dec_state* d_state,
                          const uint8_t* d_bytes, const int64_t* d_offsets, int32_t* d_syms, int64_t sym_stride,
                          int prec, void* stream) {
    if (!d_cdf || !d_state || !d_bytes || !d_offsets || !d_syms || vocab < 1 || n_streams < 0 || T < 0)
        return fail(LAC_E_ARG, "lac_acs_decode_tables: bad argument");
    if (!prec_ok(prec, 2)) return fail(LAC_E_ARG, "lac_acs_decode_tables: prec %d outside [2, 60]", prec);
    CK(lac::launch_table_decode(lac::Acs{vocab, d_cdf, stream_stride, tok_stride}, n_streams, T, d_ntok, d_state,
                                d_bytes, d_offsets, d_syms, sym_stride, prec, (cudaStream_t)stream),
       "lac_acs_decode_tables");
    return LAC_OK;
}

namespace {
// what the four adaptive entry points check before any CUDA call
int check_adaptive(const char* fn, const int64_t* d_counts, int32_t vocab, int64_t inc, int prec) {
    if (!d_counts || vocab < 1 || vocab > LAC_ADAPTIVE_MAX_VOCAB || inc < 0) return fail(LAC_E_ARG, "%s: bad argument", fn);
    if (!prec_ok(prec, 2)) return fail(LAC_E_ARG, "%s: prec %d outside [2, 60]", fn, prec);
    return LAC_OK;
}
}  // namespace

int lac_ac_encode_adaptive(int64_t* d_counts, int32_t vocab, int64_t inc, const int32_t* d_syms, int64_t sym_stride,
                           int64_t n_streams, int64_t T, const int32_t* d_ntok, lac_enc_state* d_state,
                           uint8_t* d_out, int64_t out_stride, int finish, int prec, void* stream) {
    if ((!d_syms && T > 0) || !d_state || !d_out || n_streams < 0 || T < 0 || out_stride < 1)
        return fail(LAC_E_ARG, "lac_ac_encode_adaptive: bad argument");
    if (int rc = check_adaptive("lac_ac_encode_adaptive", d_counts, vocab, inc, prec)) return rc;
    CK(lac::launch_table_encode(lac::Adaptive{vocab, d_counts, inc}, d_syms, sym_stride, n_streams, T, d_ntok, d_state,
                                d_out, out_stride, finish ? lac::kFlushAc : lac::kFlushNone, prec,
                                (cudaStream_t)stream),
       "lac_ac_encode_adaptive");
    return LAC_OK;
}

int lac_ac_decode_adaptive(int64_t* d_counts, int32_t vocab, int64_t inc, int64_t n_streams, int64_t T,
                           const int32_t* d_ntok, lac_dec_state* d_state, const uint8_t* d_bytes,
                           const int64_t* d_offsets, int32_t* d_syms, int64_t sym_stride, int prec, void* stream) {
    if (!d_state || !d_bytes || !d_offsets || !d_syms || n_streams < 0 || T < 0)
        return fail(LAC_E_ARG, "lac_ac_decode_adaptive: bad argument");
    if (int rc = check_adaptive("lac_ac_decode_adaptive", d_counts, vocab, inc, prec)) return rc;
    CK(lac::launch_table_decode(lac::Adaptive{vocab, d_counts, inc}, n_streams, T, d_ntok, d_state, d_bytes, d_offsets,
                                d_syms, sym_stride, prec, (cudaStream_t)stream),
       "lac_ac_decode_adaptive");
    return LAC_OK;
}

int lac_acs_encode_adaptive(int64_t* d_counts, int32_t vocab, int64_t inc, const int32_t* d_syms, int64_t sym_stride,
                            int64_t n_streams, int64_t T, const int32_t* d_ntok, lac_enc_state* d_state,
                            uint8_t* d_out, int64_t out_stride, int finish, int prec, void* stream) {
    if ((!d_syms && T > 0) || !d_state || !d_out || n_streams < 0 || T < 0 || out_stride < 1)
        return fail(LAC_E_ARG, "lac_acs_encode_adaptive: bad argument");
    if (int rc = check_adaptive("lac_acs_encode_adaptive", d_counts, vocab, inc, prec)) return rc;
    // finish 1: flush_compress (the reference's), 2: the safe termination, anything else: no flush
    const int flush = finish == 1 ? lac::kFlushCompress : (finish == 2 ? lac::kFlushAc : lac::kFlushNone);
    CK(lac::launch_table_encode(lac::AcsAdaptive{vocab, d_counts, inc}, d_syms, sym_stride, n_streams, T, d_ntok,
                                d_state, d_out, out_stride, flush, prec, (cudaStream_t)stream),
       "lac_acs_encode_adaptive");
    return LAC_OK;
}

int lac_acs_decode_adaptive(int64_t* d_counts, int32_t vocab, int64_t inc, int64_t n_streams, int64_t T,
                            const int32_t* d_ntok, lac_dec_state* d_state, const uint8_t* d_bytes,
                            const int64_t* d_offsets, int32_t* d_syms, int64_t sym_stride, int prec, void* stream) {
    if (!d_state || !d_bytes || !d_offsets || !d_syms || n_streams < 0 || T < 0)
        return fail(LAC_E_ARG, "lac_acs_decode_adaptive: bad argument");
    if (int rc = check_adaptive("lac_acs_decode_adaptive", d_counts, vocab, inc, prec)) return rc;
    CK(lac::launch_table_decode(lac::AcsAdaptive{vocab, d_counts, inc}, n_streams, T, d_ntok, d_state, d_bytes,
                                d_offsets, d_syms, sym_stride, prec, (cudaStream_t)stream),
       "lac_acs_decode_adaptive");
    return LAC_OK;
}

// ------------------------------------------------------------------ host-buffer calls
namespace {

struct DevBuf {
    void* p = nullptr;
    size_t n = 0;
    int reserve(size_t bytes) {
        if (bytes <= n) return LAC_OK;
        if (p) cudaFree(p);
        p = nullptr;
        n = 0;
        cudaError_t e = cudaMalloc(&p, bytes);
        if (e != cudaSuccess) return cuda_fail(e, "cudaMalloc");
        n = bytes;
        return LAC_OK;
    }
};

// One context per device ordinal: its streams, events and buffers belong to that device only.
struct HostCtx {
    std::mutex mu;
    bool ready = false;
    cudaStream_t st[2] = {nullptr, nullptr};
    cudaEvent_t done[2] = {nullptr, nullptr};  // kernels of the last piece on st[q]
    DevBuf logits[2], ws[2], syms, state, out, offs, bytes, flag;
    int ensure() {
        if (ready) return LAC_OK;
        for (int q = 0; q < 2; q++) {
            CK(cudaStreamCreateWithFlags(&st[q], cudaStreamNonBlocking), "cudaStreamCreate");
            CK(cudaEventCreateWithFlags(&done[q], cudaEventDisableTiming), "cudaEventCreate");
        }
        ready = true;
        return LAC_OK;
    }
};
constexpr int kMaxDevices = 64;
HostCtx g_host[kMaxDevices];

int host_ctx(HostCtx** ctx) {
    int dev = 0;
    CK(cudaGetDevice(&dev), "cudaGetDevice");
    if (dev < 0 || dev >= kMaxDevices) return fail(LAC_E_CUDA, "device ordinal %d not supported", dev);
    *ctx = &g_host[dev];
    return LAC_OK;
}

constexpr size_t kPieceBytes = size_t(256) << 20;  // logits staged to the device in <= 256 MB pieces, double-buffered

// The [n_streams, T] grid cut into pieces of contiguous logits: whole streams when a stream fits a piece, else
// token ranges of one stream.
struct Pieces {
    int64_t ns, tn;  // streams per piece, tokens per piece
    Pieces(int64_t n_streams, int64_t T, size_t row_bytes) {
        int64_t rows = (int64_t)(kPieceBytes / row_bytes);
        if (rows < 1) rows = 1;
        if (T <= rows) {
            ns = rows / T;
            if (ns > n_streams) ns = n_streams;
            tn = T;
        } else {
            ns = 1;
            tn = rows;
        }
    }
};

}  // namespace

// ---- (e) batch-invariant model kernels
int lac_model_gemm(const void* d_x, const void* d_w, int64_t M, int32_t N, int32_t K, int epilogue,
                   const void* d_res, void* d_y, void* stream) {
    if (!d_x || !d_w || !d_y || epilogue < LAC_MODEL_OUT_BF16 || epilogue > LAC_MODEL_OUT_F32 ||
        (epilogue == LAC_MODEL_OUT_BF16_ADD && !d_res) || (((uintptr_t)d_x | (uintptr_t)d_w | (uintptr_t)d_y |
                                                             (uintptr_t)d_res) & 15))
        return fail(LAC_E_ARG, "lac_model_gemm: bad argument");
    if (!lac::model_gemm_shape_ok(M, N, K))
        return fail(LAC_E_ARG, "lac_model_gemm: unsupported shape M=%lld N=%d K=%d (N %% 128 == 0, K %% 64 == 0, M >= 1)",
                    (long long)M, N, K);
    CK(lac::launch_model_gemm(d_x, d_w, M, N, K, epilogue, d_res, d_y, (cudaStream_t)stream), "lac_model_gemm");
    return LAC_OK;
}

int lac_model_rmsnorm(const void* d_x, int64_t rows, int32_t dim, float eps, void* d_y, void* stream) {
    if (!d_x || !d_y || rows < 0 || dim < 256 || dim % 256 || !(eps >= 0.f) || (((uintptr_t)d_x | (uintptr_t)d_y) & 15))
        return fail(LAC_E_ARG, "lac_model_rmsnorm: bad argument (dim %d must be a positive multiple of 256)", dim);
    if (rows == 0) return LAC_OK;
    CK(lac::launch_model_rmsnorm(d_x, rows, dim, eps, d_y, (cudaStream_t)stream), "lac_model_rmsnorm");
    return LAC_OK;
}

int lac_model_rope_kv(void* d_qkv, int64_t rows, int32_t n_streams, int32_t heads, int32_t kv_heads, int32_t hd,
                      const void* d_cos, const void* d_sin, const int64_t* d_pos, int64_t p0, void* d_kc, void* d_vc,
                      int32_t max_len, void* stream) {
    if (!d_qkv || !d_cos || !d_sin || !d_kc || !d_vc || n_streams < 1 || rows < 0 || rows % n_streams ||
        kv_heads < 1 || heads < kv_heads || heads % kv_heads || hd < 2 || hd % 2 || max_len < 1 || p0 < 0 ||
        (!d_pos && p0 + rows / n_streams > max_len))
        return fail(LAC_E_ARG, "lac_model_rope_kv: bad argument");
    if (rows == 0) return LAC_OK;
    CK(lac::launch_model_rope_kv(d_qkv, rows, n_streams, heads, kv_heads, hd, d_cos, d_sin, d_pos, p0, d_kc, d_vc,
                                 max_len, (cudaStream_t)stream),
       "lac_model_rope_kv");
    return LAC_OK;
}

int lac_model_swiglu(const void* d_h, int64_t rows, int32_t ffn, void* d_y, void* stream) {
    if (!d_h || !d_y || rows < 0 || ffn < 1) return fail(LAC_E_ARG, "lac_model_swiglu: bad argument");
    if (rows == 0) return LAC_OK;
    CK(lac::launch_model_swiglu(d_h, rows, ffn, d_y, (cudaStream_t)stream), "lac_model_swiglu");
    return LAC_OK;
}

int lac_model_attention(const void* d_qkv, int32_t n_streams, int32_t n_q, int32_t heads, int32_t kv_heads, int32_t hd,
                        const int64_t* d_pos, int64_t p0, const void* d_kc, const void* d_vc, int32_t max_len,
                        void* d_out, void* stream) {
    if (!d_qkv || !d_kc || !d_vc || !d_out || n_streams < 1 || n_q < 0 || kv_heads < 1 || heads < kv_heads ||
        heads % kv_heads || heads / kv_heads > 64 || max_len < 1 || p0 < 0 || (!d_pos && p0 + n_q > max_len) ||
        (((uintptr_t)d_qkv | (uintptr_t)d_kc | (uintptr_t)d_vc | (uintptr_t)d_out) & 15))
        return fail(LAC_E_ARG, "lac_model_attention: bad argument");
    if (hd != 64 && hd != 128) return fail(LAC_E_ARG, "lac_model_attention: head dim %d is not 64 or 128", hd);
    if (n_q == 0) return LAC_OK;
    CK(lac::launch_model_attention(d_qkv, n_streams, n_q, heads, kv_heads, hd, d_pos, p0, d_kc, d_vc, max_len, d_out,
                                   (cudaStream_t)stream),
       "lac_model_attention");
    return LAC_OK;
}

int lac_encode_logits_host(const float* h_logits, const int32_t* h_syms, int64_t n_streams, int64_t T,
                           int32_t vocab, uint8_t* h_out, int64_t out_stride, uint64_t* h_nbits, int prec) {
    if ((T > 0 && (!h_logits || !h_syms)) || !h_out || !h_nbits || n_streams < 0 || T < 0 || out_stride < 1)
        return fail(LAC_E_ARG, "lac_encode_logits_host: bad argument");
    if (!prec_ok(prec, 34)) return fail(LAC_E_ARG, "lac_encode_logits_host: prec %d outside [34, 60]", prec);
    if (int rc = check_vocab(vocab)) return rc;
    if (n_streams == 0) return LAC_OK;
    HostCtx* c = nullptr;
    if (int rc = host_ctx(&c)) return rc;
    std::lock_guard<std::mutex> lk(c->mu);
    if (int rc = c->ensure()) return rc;
    const size_t row_bytes = (size_t)vocab * 4;
    const Pieces pc(n_streams, T > 0 ? T : 1, row_bytes);
    const int64_t piece_rows = pc.ns * pc.tn;
    if (T > 0) {
        for (int q = 0; q < 2; q++) {
            if (int rc = c->logits[q].reserve((size_t)piece_rows * row_bytes)) return rc;
            if (int rc = c->ws[q].reserve((size_t)lac_workspace_bytes(piece_rows, vocab))) return rc;
        }
        if (int rc = c->syms.reserve((size_t)n_streams * (size_t)T * 4)) return rc;
    }
    if (int rc = c->state.reserve((size_t)n_streams * sizeof(lac_enc_state))) return rc;
    if (int rc = c->out.reserve((size_t)n_streams * (size_t)out_stride)) return rc;
    lac_enc_state* dstate = (lac_enc_state*)c->state.p;
    cudaStream_t s0 = c->st[0];
    if (T > 0) CK(cudaMemcpyAsync(c->syms.p, h_syms, (size_t)n_streams * (size_t)T * 4, cudaMemcpyHostToDevice, s0), "H2D syms");
    CK(lac::launch_enc_init(dstate, n_streams, prec, s0), "enc_init");
    CK(cudaEventRecord(c->done[0], s0), "event");
    CK(cudaStreamWaitEvent(c->st[1], c->done[0], 0), "wait");
    if (T == 0) {
        CK(lac::launch_encode_logits(nullptr, n_streams, 0, 0, 0, vocab, nullptr, 0, nullptr, dstate,
                                     (uint8_t*)c->out.p, out_stride, 1, prec, nullptr, 0, s0),
           "encode (flush only)");
        CK(cudaEventRecord(c->done[0], s0), "event");
    }
    int k = 0;
    for (int64_t sb = 0; sb < n_streams && T > 0; sb += pc.ns) {
        const int64_t ns = n_streams - sb < pc.ns ? n_streams - sb : pc.ns;
        for (int64_t t0 = 0; t0 < T; t0 += pc.tn, k++) {
            const int64_t tn = T - t0 < pc.tn ? T - t0 : pc.tn;
            const int q = k & 1;
            // the copy of piece k overlaps the kernels of piece k - 1 (other stream); its kernels wait for them
            // (a stream cut into token pieces carries its coder state from piece to piece)
            CK(cudaMemcpyAsync(c->logits[q].p, h_logits + (sb * T + t0) * (int64_t)vocab, (size_t)(ns * tn) * row_bytes,
                               cudaMemcpyHostToDevice, c->st[q]),
               "H2D logits");
            CK(cudaStreamWaitEvent(c->st[q], c->done[q ^ 1], 0), "wait");
            CK(lac::launch_encode_logits((const float*)c->logits[q].p, ns, tn, tn * (int64_t)vocab, vocab, vocab,
                                         (const int32_t*)c->syms.p + sb * T + t0, T, nullptr, dstate + sb,
                                         (uint8_t*)c->out.p + sb * out_stride, out_stride, t0 + tn >= T, prec,
                                         c->ws[q].p, c->ws[q].n, c->st[q]),
               "encode");
            CK(cudaEventRecord(c->done[q], c->st[q]), "event");
        }
    }
    CK(cudaStreamWaitEvent(s0, c->done[1], 0), "wait");
    CK(cudaStreamWaitEvent(s0, c->done[0], 0), "wait");
    CK(cudaMemcpyAsync(h_out, c->out.p, (size_t)n_streams * (size_t)out_stride, cudaMemcpyDeviceToHost, s0), "D2H bytes");
    std::string tmp((size_t)n_streams * sizeof(lac_enc_state), '\0');
    CK(cudaMemcpyAsync(&tmp[0], dstate, tmp.size(), cudaMemcpyDeviceToHost, s0), "D2H state");
    CK(cudaStreamSynchronize(s0), "sync");
    CK(cudaStreamSynchronize(c->st[1]), "sync");
    const lac_enc_state* hs = (const lac_enc_state*)tmp.data();
    int rc = LAC_OK;
    for (int64_t s = 0; s < n_streams; s++) {
        h_nbits[s] = hs[s].nbits;
        if (hs[s].status & LAC_ST_CAP) rc = fail(LAC_E_CAP, "stream %lld: output capacity exceeded", (long long)s);
        else if (hs[s].status & LAC_ST_SYMBOL) rc = fail(LAC_E_SYMBOL, "stream %lld: symbol outside [0, %d)", (long long)s, vocab);
        else if (hs[s].status) rc = fail(LAC_E_ARG, "stream %lld: status %u", (long long)s, hs[s].status);
    }
    return rc;
}

int lac_decode_logits_host(const float* h_logits, int64_t n_streams, int64_t T, int32_t vocab,
                           const uint8_t* h_bytes, const int64_t* h_offsets, int32_t* h_syms, int prec) {
    if ((T > 0 && (!h_logits || !h_syms)) || !h_bytes || !h_offsets || n_streams < 0 || T < 0)
        return fail(LAC_E_ARG, "lac_decode_logits_host: bad argument");
    if (!prec_ok(prec, 34)) return fail(LAC_E_ARG, "lac_decode_logits_host: prec %d outside [34, 60]", prec);
    if (int rc = check_vocab(vocab)) return rc;
    if (n_streams == 0 || T == 0) return LAC_OK;
    if (h_offsets[0] != 0) return fail(LAC_E_ARG, "lac_decode_logits_host: offsets must start at 0");
    for (int64_t s = 0; s < n_streams; s++)
        if (h_offsets[s + 1] < h_offsets[s])
            return fail(LAC_E_ARG, "lac_decode_logits_host: offsets decrease at stream %lld", (long long)s);
    HostCtx* c = nullptr;
    if (int rc = host_ctx(&c)) return rc;
    std::lock_guard<std::mutex> lk(c->mu);
    if (int rc = c->ensure()) return rc;
    const size_t row_bytes = (size_t)vocab * 4;
    const Pieces pc(n_streams, T, row_bytes);
    const int64_t piece_rows = pc.ns * pc.tn;
    const size_t total_bytes = (size_t)h_offsets[n_streams];
    for (int q = 0; q < 2; q++) {
        if (int rc = c->logits[q].reserve((size_t)piece_rows * row_bytes)) return rc;
        if (int rc = c->ws[q].reserve((size_t)lac_workspace_bytes(piece_rows, vocab))) return rc;
    }
    if (int rc = c->bytes.reserve(total_bytes + 16)) return rc;
    if (int rc = c->offs.reserve((size_t)(n_streams + 1) * 8)) return rc;
    if (int rc = c->state.reserve((size_t)n_streams * sizeof(lac_dec_state))) return rc;
    if (int rc = c->syms.reserve((size_t)n_streams * (size_t)T * 4)) return rc;
    if (int rc = c->flag.reserve(16)) return rc;
    cudaStream_t s0 = c->st[0];
    CK(cudaMemcpyAsync(c->bytes.p, h_bytes, total_bytes, cudaMemcpyHostToDevice, s0), "H2D bytes");
    CK(cudaMemcpyAsync(c->offs.p, h_offsets, (size_t)(n_streams + 1) * 8, cudaMemcpyHostToDevice, s0), "H2D offsets");
    lac_dec_state* dstate = (lac_dec_state*)c->state.p;
    CK(lac::launch_dec_init(dstate, n_streams, prec, (const uint8_t*)c->bytes.p, (const int64_t*)c->offs.p, s0), "dec_init");
    CK(cudaEventRecord(c->done[0], s0), "event");
    CK(cudaStreamWaitEvent(c->st[1], c->done[0], 0), "wait");
    int k = 0;
    for (int64_t sb = 0; sb < n_streams; sb += pc.ns) {
        const int64_t ns = n_streams - sb < pc.ns ? n_streams - sb : pc.ns;
        for (int64_t t0 = 0; t0 < T; t0 += pc.tn, k++) {
            const int64_t tn = T - t0 < pc.tn ? T - t0 : pc.tn;
            const int q = k & 1;
            CK(cudaMemcpyAsync(c->logits[q].p, h_logits + (sb * T + t0) * (int64_t)vocab, (size_t)(ns * tn) * row_bytes,
                               cudaMemcpyHostToDevice, c->st[q]),
               "H2D logits");
            CK(cudaStreamWaitEvent(c->st[q], c->done[q ^ 1], 0), "wait");
            CK(lac::launch_decode((const float*)c->logits[q].p, ns, tn, tn * (int64_t)vocab, vocab, vocab, nullptr,
                                  dstate + sb, (const uint8_t*)c->bytes.p, (const int64_t*)c->offs.p + sb,
                                  (int32_t*)c->syms.p + sb * T + t0, T, prec, c->ws[q].p, c->ws[q].n, c->st[q]),
               "decode");
            CK(cudaEventRecord(c->done[q], c->st[q]), "event");
        }
    }
    CK(cudaStreamWaitEvent(s0, c->done[1], 0), "wait");
    CK(cudaStreamWaitEvent(s0, c->done[0], 0), "wait");
    CK(lac::launch_status_or(dstate, n_streams, (int)(sizeof(lac_dec_state) / 4), 8, (uint32_t*)c->flag.p, s0), "status");
    uint32_t st_or = 0;
    CK(cudaMemcpyAsync(h_syms, c->syms.p, (size_t)n_streams * (size_t)T * 4, cudaMemcpyDeviceToHost, s0), "D2H syms");
    CK(cudaMemcpyAsync(&st_or, c->flag.p, 4, cudaMemcpyDeviceToHost, s0), "D2H status");
    CK(cudaStreamSynchronize(s0), "sync");
    CK(cudaStreamSynchronize(c->st[1]), "sync");
    if (st_or & LAC_ST_TRUNC) return fail(LAC_E_STREAM, "lac_decode_logits_host: truncated or foreign bitstream");
    if (st_or) return fail(LAC_E_ARG, "lac_decode_logits_host: decoder status %u", st_or);
    return LAC_OK;
}

}  // extern "C"
