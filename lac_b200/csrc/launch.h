// launch.h -- host-side declarations shared by the .cu files of liblac_b200.so.
#pragma once
#include <cstddef>
#include <cstdint>
#include <cuda_runtime.h>

#include "../../include/lac_b200.h"

namespace lac {

// device scratch of one call: the caller's workspace or a stream-ordered allocation
struct Scratch {
    void* p;
    bool owned;
};
cudaError_t scratch_get(Scratch* sc, size_t bytes, void* ws, size_t ws_bytes, cudaStream_t st);
cudaError_t scratch_put(Scratch* sc, cudaStream_t st);

int sm_count();
int max_vocab();
int path_for(const float* p, int V, int64_t s0, int64_t s1, int* parts);  // load width: 4, 1 (or -1: unsupported)
int64_t summ_chunk_rows(int parts);
int64_t summ_rows_for(int64_t want, int parts, const void* ws, size_t ws_bytes);
size_t summ_bytes(int64_t rows, int parts);       // scratch per launch: row summaries + (lo, hi) pairs
size_t summ_only_bytes(int64_t rows, int parts);  // offset of the pairs inside it
cudaError_t launch_summary(const float* base, int64_t n_outer, int64_t T, int64_t so, int64_t st_, int V, int parts,
                           int vec, int keep_l2, uint64_t* summ, cudaStream_t st);
cudaError_t launch_pairs(const float* logits, int64_t n, int64_t T, int64_t so, int64_t st_, int V, int parts, int vec,
                         const uint64_t* summ, const int32_t* syms, int64_t sym_stride, uint32_t* pairs,
                         uint32_t* status, cudaStream_t st);

// instantiate MACRO(CL) for the run-time number of parts (1 .. 8)
#define LAC_BY_PARTS(parts, MACRO) \
    switch (parts) {               \
        case 1: MACRO(1); break;   \
        case 2: MACRO(2); break;   \
        case 3: MACRO(3); break;   \
        case 4: MACRO(4); break;   \
        case 5: MACRO(5); break;   \
        case 6: MACRO(6); break;   \
        case 7: MACRO(7); break;   \
        default: MACRO(8); break;  \
    }

// cdf_kernels.cu
cudaError_t launch_lookup(const float*, int64_t, int, int64_t, const int32_t*, uint32_t*, uint32_t*, void*, size_t,
                          cudaStream_t);
cudaError_t launch_build(const float*, int64_t, int, int64_t, uint32_t*, void*, size_t, cudaStream_t);
// decode_kernels.cu
cudaError_t launch_decode(const float*, int64_t, int64_t, int64_t, int64_t, int, const int32_t*, lac_dec_state*,
                          const uint8_t*, const int64_t*, int32_t*, int64_t, int, void*, size_t, cudaStream_t);
cudaError_t launch_dec_init(lac_dec_state*, int64_t, int, const uint8_t*, const int64_t*, cudaStream_t);
// coder_kernels.cu
cudaError_t launch_enc_init(lac_enc_state*, int64_t, int, cudaStream_t);
cudaError_t launch_encode_pairs(const uint32_t*, int64_t, int64_t, int64_t, int64_t, const int32_t*, int64_t,
                                lac_enc_state*, uint8_t*, int64_t, int, int, cudaStream_t);
cudaError_t launch_encode_logits(const float*, int64_t, int64_t, int64_t, int64_t, int, const int32_t*, int64_t,
                                 const int32_t*, lac_enc_state*, uint8_t*, int64_t, int, int, void*, size_t,
                                 cudaStream_t);

// table_coders.cu: the table models, symbols [0, n_symbols), and how many threads code one stream (1 or 32)
struct Uniform {  // Predictor(n)
    static constexpr int kEncLanes = 1, kDecLanes = 1;
    int n_symbols;
};
struct Cdf {  // CDFPredictor: table (s, t) at dist + s * ss + t * ts, its minp at minp[s * mss + t * mts]
    static constexpr int kEncLanes = 32, kDecLanes = 32;
    int n_symbols;
    const int64_t* dist;
    int64_t ss, ts;
    const int64_t* minp;
    int64_t mss, mts;
    int flags;
};
struct Acs {  // ACSampler: table (s, t) at cdf + s * ss + t * ts
    static constexpr int kEncLanes = 1, kDecLanes = 32;
    int n_symbols;
    const uint64_t* cdf;
    int64_t ss, ts;
};
// Adaptive count models, prob(s) = counts[s] and counts[sym] += inc after every token; the counts of stream s at
// counts + s * n_symbols (n_symbols <= LAC_ADAPTIVE_MAX_VOCAB), read at the start of a call and written back at its end
struct Adaptive {  // CDFPredictor semantics (ProbPredictor under A_to_bin / A_from_bin)
    static constexpr int kEncLanes = 32, kDecLanes = 32;
    int n_symbols;
    int64_t* counts;
    int64_t inc;
};
struct AcsAdaptive {  // ACSampler semantics
    static constexpr int kEncLanes = 32, kDecLanes = 32;
    int n_symbols;
    int64_t* counts;
    int64_t inc;
};
// how an encode call ends a stream: A_to_bin.flush (coder::ac_flush) or ACSampler's flush_compress
enum TableFlush { kFlushNone, kFlushAc, kFlushCompress };
template <class Model>
cudaError_t launch_table_encode(const Model&, const int32_t* syms, int64_t sym_stride, int64_t n, int64_t T,
                                const int32_t* ntok, lac_enc_state*, uint8_t* out, int64_t out_stride, int flush,
                                int P, cudaStream_t);
template <class Model>
cudaError_t launch_table_decode(const Model&, int64_t n, int64_t T, const int32_t* ntok, lac_dec_state*,
                                const uint8_t* bytes, const int64_t* offsets, int32_t* syms, int64_t sym_stride,
                                int P, cudaStream_t);

// model_kernels.cu
bool model_gemm_shape_ok(int64_t M, int N, int K);
cudaError_t launch_model_gemm(const void* x, const void* w, int64_t M, int N, int K, int epi, const void* res, void* y,
                              cudaStream_t st);
cudaError_t launch_model_rmsnorm(const void* x, int64_t rows, int dim, float eps, void* y, cudaStream_t st);
cudaError_t launch_model_rope_kv(void* qkv, int64_t rows, int S, int H, int KV, int hd, const void* cosb,
                                 const void* sinb, const int64_t* d_pos, int64_t p0, void* kc, void* vc, int max_len,
                                 cudaStream_t st);
cudaError_t launch_model_swiglu(const void* h, int64_t rows, int F, void* y, cudaStream_t st);
cudaError_t launch_model_attention(const void* qkv, int S, int n_q, int H, int KV, int hd, const int64_t* d_pos,
                                   int64_t p0, const void* kc, const void* vc, int max_len, void* out,
                                   cudaStream_t st);

}  // namespace lac
