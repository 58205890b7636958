// Interface of gemm_tc.cu (tcgen05 GEMM with fused epilogues) to the rest of the library.
#pragma once
#include "xb_common.cuh"

enum { EPI_F32 = 0, EPI_BF16OUT = 5, EPI_CONV3_BWD = 7 };

struct GemmParams {
    int M = 0, N = 0, K = 0;       // logical problem (rows of A that are valid, columns = rows of B, depth)
    int split_k = 1;               // EPI_F32: K slices (gridDim.z) whose partial tiles are ADDED to a zeroed output
    const float *bias = nullptr;   // (N) fp32
    void *out = nullptr;
    int ldo = 0;                   // output row pitch in elements
    int T = 0, NB = 0;             // EPI_CONV3_BWD: rows are (chunk, t), dy is stored at (t, chunk)
    // training backward (EPI_CONV3_BWD: recomputed conv3 pre-activation -> its gradient)
    const void *dy = nullptr;      // (T, NB, 768) bf16: gradient w.r.t. the stem output
};

// TMA descriptor of a rank-n tensor (2 <= n <= 5): dims / box in elements (innermost first), strides in BYTES for
// dimensions 1 .. n-1; elem_bytes 2 (16-bit payload) or 4 (fp32).  With CU_TENSOR_MAP_SWIZZLE_128B the innermost box
// extent must span 128 bytes.
int xb_make_tmap_nd(xb_handle *h, CUtensorMap *out, const void *base, int rank, int elem_bytes, const uint64_t *dims,
                    const uint64_t *strides_bytes, const uint32_t *box, CUtensorMapSwizzle swizzle);
// the GEMM operand: rows x K 16-bit elements, row pitch ld elements, box 64 x 128, 128B swizzle
int xb_make_tmap_2d(xb_handle *h, CUtensorMap *out, const void *base, uint64_t rows, uint64_t K, uint64_t ld);

// lstm_bptt.cu: one step of back-propagation through time of an LSTM layer (programmatic dependent launches)
struct BpttMaps {
    CUtensorMap dz_rows;           // DZ as (T*N, 3072) bf16: the A operand dz_{t_next}
    CUtensorMap w_hhT;             // W_hh^T (768, 3072) bf16, 64-row boxes
    CUtensorMap saved;             // saved (768, N, 5, T) fp16 view, box {64, 128, 5, 1}
    CUtensorMap saved_c;           // same tensor, box {64, 128, 1, 1}: the cell state of the previous step
    CUtensorMap dz_out;            // DZ as (768, N, 4, T) bf16 view, box {64, 128, 4, 1}
};
struct BpttStep {
    int N = 0, t_cur = 0, t_prev = -1, t_next = -1;      // t_next < 0: first BPTT step of the layer (no recurrent term)
    const void *dy = nullptr;      // (T, N, 768) bf16
    float *dcstate = nullptr;      // (N, 768) fp32
};
int xb_bptt_make_maps(xb_handle *h, BpttMaps *m, const void *dz, const void *w_hhT, const void *saved, int T, int N);
int xb_bptt_step_launch(xb_handle *h, const BpttMaps &m, const BpttStep &p, bool dependent, cudaStream_t s);
// conv3_gemm.cu: weight-stationary persistent GEMM of the stem's third convolution
int xb_conv3_launch(xb_handle *h, const void *col, const void *w3, const float *bias, void *out_tnc, int T, int N, cudaStream_t s);
int xb_gemm_launch(xb_handle *h, int epi, const CUtensorMap &tmA, const CUtensorMap &tmB, const GemmParams &p,
                   cudaStream_t s, bool bf16_operands = false);
