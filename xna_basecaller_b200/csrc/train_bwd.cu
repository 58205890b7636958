// Training step of the encoder (BASELINE configs[4] "fwd_bwd"): forward that keeps what the backward needs, and the
// backward from d loss / d scores to the gradients of all 28 parameter tensors.
//
// Reference: Trainer.train_one_step (bonito/training.py:91-117): scores = model(data); loss = ctc_loss(scores, targets);
// scaler.scale(loss).backward() -- torch autograd through LinearCRFEncoder (nn.py:112-133), five torch.nn.LSTM layers
// (nn.py:176-235, directions crf/model.py:152-154), Permute and the three Convolutions (nn.py:57-68).  The loss and its
// gradient w.r.t. the scores are xb_ctc_crf_loss_fwd / _bwd; this file carries that gradient down to the weights.
//
// Forward (xb_encoder_fwd_train): the inference kernels, with every layer's input kept (x[0..5], (T,N,768) fp16) and the
// persistent LSTM kernel in its SAVE form: it also stores the activated gates i, f, g, o and the cell state c of every
// step ((T,N,5,768) fp16 per layer), so that back-propagation through time needs no recomputation.
//
// Backward (xb_encoder_bwd).  Gradients travel as bfloat16 (the range of fp16 is too narrow for unscaled gradients: the
// reference needs a GradScaler for the same reason), products accumulate in fp32 on the tensor cores, weight gradients
// are written in fp32.
//   head     dz = dS[non-blank] * scale * (1 - tanh^2) from the stored scores;  dW = dz^T x5;  db = colsum dz;  dy5 = dz W
//   LSTM l   T launches of the BPTT step kernel (lstm_bptt.cu), one per time step in reverse forward order, chained with
//            programmatic dependent launches: dh_t = dz_{next} W_hh + dy_t, then the cell backward -> DZ[t] (T*N, 3072)
//            and the running dc;  dW_ih = DZ^T x_l,  dW_hh = DZ^T h_prev (time-shifted view of the layer output),
//            db = colsum DZ,  dy_{l-1} = DZ W_ih.   The K = T*N contractions run on K-major transposed copies
//            (transpose16v_kernel), which also take every bias gradient's column sum on the way.
//   conv3    pre-activation recomputed from the im2col rows (EPI_CONV3_BWD) -> d pre;  dW3 = d pre^T col;  db3;
//            d col = d pre W3 -> col2im -> conv2 / conv1 backward (conv_stem_bwd kernels below).
// Measured at N = 512, T = 800 (profiles/r02_config5_train_step_v5.json): 154 ms per training step, of which the 4000 BPTT
// steps take ~69 ms (17.3 us each: ~10 us of main loop bound by one SM's L2 ingest of its 1.15 MB of operands, the rest
// epilogue and the kernel hand-over), the K = T*N weight-gradient GEMMs ~20 ms (wgrad_gemm.cu) and the forward ~25 ms.
//
// Dropout (xb_encoder_fwd_train_dropout; mask contract in xb_dropout.cuh).  Nothing is stored: every pass that needs a mask
// regenerates it from (seed, site, element index).
//   sites 0, 1  conv12_im2col's masked form in the forward and in the backward's recomputation of the rows; conv2_bwd_kernel
//               masks its recomputed conv1 output (site 0), the incoming conv2 gradient (site 1) and the conv1 gradient
//               it scatters (site 0).
//   site 2      applied in place to x[0] (the conv3 backward recomputes its pre-activation from the rows, so the
//               undropped x[0] is never needed again); the gradient w.r.t. x[0] is masked before EPI_CONV3_BWD.
//   sites 3..6  x[l+1] keeps the undropped output of LSTM l (dW_hh of layer l reads it through the time-shifted view);
//               layer l+1's input projection reads a dropped copy in the scratch buffer xd.  The backward transposes x[l+1]
//               twice: plainly into XT (for dW_hh of layer l) and through the mask into xd (for dW_ih of layer l+1),
//               and masks dy (the gradient w.r.t. the dropped input) before the BPTT of layer l consumes it.
// With every p = 0 none of these launches happens and the step is bit for bit the step without dropout.
#include "xb_common.cuh"
#include "xb_dropout.cuh"
#include "xb_gemm.cuh"

struct xb_train_ws {
    int cap_N = 0, cap_T = 0;      // capacity
    int N = 0, T = 0;              // shape of the last forward
    void *x[6] = {};               // x[0] stem output, x[l+1] output of LSTM l: (T,N,768) fp16
    void *saved[5] = {};           // (T,N,5,768) fp16
    void *DZ = nullptr, *DZT = nullptr;          // (TN,3072) / (3072,TN) bf16
    void *XT[2] = {};              // (768,TN) bf16
    void *dy[2] = {};              // (TN,768) bf16
    void *dzh = nullptr, *dzhT = nullptr;        // (TN,HP) / (HP,TN) bf16, HP = padded head rows
    void *dpre = nullptr, *dpreT = nullptr;      // conv3: (TN,768) / (768,TN) bf16 (aliases of DZ / DZT)
    void *colT = nullptr;          // (320,TN) bf16: transposed im2col rows
    void *dcol = nullptr;          // (TN,320) bf16
    float *dcstate = nullptr;      // (N,768)
    float *dc2 = nullptr;          // (N, L, 16) fp32: gradient w.r.t. the conv2 output (post-activation)
    float *dc1 = nullptr;          // (N, L, 4) fp32
    void *xd = nullptr;            // dropout sites 3..6 only: forward (T,N,768) fp16 dropped copy of the next layer's input;
                                   // backward (768,TN) bf16 transposed dropped input of the layer being differentiated
    xb_dropout drop;               // (p, seed) of the last forward
};

namespace {

// dropout of a 16-bit tensor whose element index is its flat offset (sites 2..6): eight elements per iteration; in == out
// is allowed
template <bool BF16>
__global__ void __launch_bounds__(256) dropout16_kernel(const uint4 *in, uint4 *out, size_t n8, const xb_dropout drop, int site) {
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n8; i += (size_t)gridDim.x * blockDim.x)
        out[i] = xb_dropout8<BF16>(drop, site, i * 8, in[i]);
}

__global__ void dropout_keep_kernel(const xb_dropout drop, int site, int64_t n, uint8_t *__restrict__ keep) {
    for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < n; e += (int64_t)gridDim.x * blockDim.x)
        keep[e] = xb_dropout_keep(drop, site, (uint64_t)e) ? 1 : 0;
}

// LinearCRFEncoder backward through scale * tanh and the blank expansion (nn.py:117-129): for head row j = c * n_base + b,
// score column c * NZ + 1 + b:  dz = dS * (scale - s^2 / scale).   dzh (TN, HP) bf16, padding columns zero.
__global__ void head_bwd_kernel(const float *__restrict__ dS, const float *__restrict__ scores, size_t rows, int n_base, int NZ,
                                int head_rows, int HP, int S, int expand, float scale, __nv_bfloat16 *__restrict__ dzh) {
    const size_t idx = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= rows * HP) return;
    const size_t r = idx / HP;
    const int j = (int)(idx % HP);
    float v = 0.0f;
    if (j < head_rows) {
        const int col = expand ? (j / n_base) * NZ + 1 + (j % n_base) : j;
        const float s = scores[r * S + col];
        v = dS[r * S + col] * (scale - s * s / scale);
    }
    dzh[idx] = __float2bfloat16_rn(v);
}

// ---- convolution stem backward below conv3 ---------------------------------------------------------------------
// d col (N*T, 320) bf16 -> gradient w.r.t. the conv2 OUTPUT a2 (N, L, 16) fp32 (col2im as a gather: position p of chunk b
// appears in window t at tap = p + 9 - 5 t, 0 <= tap < 19).
__global__ void col2im_kernel(const __nv_bfloat16 *__restrict__ dcol, int N, int T, int L, float *__restrict__ da2) {
    const size_t idx = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= (size_t)N * L * XB_C2_CH) return;
    const int ch = (int)(idx % XB_C2_CH);
    const int p = (int)((idx / XB_C2_CH) % L);
    const int b = (int)(idx / ((size_t)XB_C2_CH * L));
    float s = 0.0f;
    // 5 t - 9 <= p <= 5 t + 9
    int t_lo = (p - 9 + 4) / 5;
    if (p - 9 < 0) t_lo = 0;
    for (int t = t_lo; t < T && 5 * t - 9 <= p; t++) {
        const int tap = p + 9 - 5 * t;
        if (tap >= 0 && tap < XB_WINLEN) s += __bfloat162float(dcol[((size_t)b * T + t) * XB_CONV3_K + tap * XB_C2_CH + ch]);
    }
    da2[idx] = s;
}

__device__ __forceinline__ float swishf(float x) { return x / (1.0f + __expf(-x)); }
__device__ __forceinline__ float dswishf(float x) { const float sg = 1.0f / (1.0f + __expf(-x)); return sg * (1.0f + x * (1.0f - sg)); }

// conv2 backward: recomputes conv1 (and its swish) and the conv2 pre-activation from the signal, turns da2 into
// d pre2, accumulates dW2 (16,4,5), db2 (16) and scatters the gradient w.r.t. the conv1 output a1 into da1 (N, L, 4).
// One block per (chunk, tile of 256 positions); block-level reductions, then one atomicAdd per weight and block.
// DROP: conv2's input is the masked conv1 output (site 0) and da2 is the gradient w.r.t. the masked conv2 output (site 1).
template <bool DROP, typename SIG>
__global__ void __launch_bounds__(256)
conv2_bwd_kernel(const SIG *__restrict__ signal, int L, const float *__restrict__ w1, const float *__restrict__ b1,
                 const float *__restrict__ w2, const float *__restrict__ b2, const float *__restrict__ da2,
                 float *__restrict__ da1, float *__restrict__ dw2, float *__restrict__ db2, const xb_dropout drop) {
    constexpr int TP = 256;
    __shared__ float sx[TP + 8];          // signal positions p0-4 .. p0+TP+3
    __shared__ float a1[TP + 4][4];       // conv1 output (post swish) positions p0-2 .. p0+TP+1
    __shared__ float dp2[TP][16];         // d pre2
    __shared__ float sw1[20], sb1[4], sw2[320], sb2[16];
    const int b = blockIdx.y, p0 = blockIdx.x * TP, tid = threadIdx.x;
    const SIG *sig = signal + (size_t)b * L;
    for (int i = tid; i < 20; i += 256) sw1[i] = w1[i];
    for (int i = tid; i < 4; i += 256) sb1[i] = b1[i];
    for (int i = tid; i < 320; i += 256) sw2[i] = w2[i];
    for (int i = tid; i < 16; i += 256) sb2[i] = b2[i];
    for (int i = tid; i < TP + 8; i += 256) {
        const int p = p0 - 4 + i;
        sx[i] = (p >= 0 && p < L) ? (float)sig[p] : 0.0f;
    }
    __syncthreads();
    for (int i = tid; i < (TP + 4) * 4; i += 256) {
        const int pos = i >> 2, ch = i & 3, p = p0 - 2 + pos;
        float v = 0.0f;
        if (p >= 0 && p < L) {
            v = sb1[ch];
#pragma unroll
            for (int k = 0; k < 5; k++) v = fmaf(sw1[ch * 5 + k], sx[pos + k], v);
            v = swishf(v);
            if (DROP && drop.on(0)) v = xb_dropout_apply(drop, 0, ((uint64_t)b * 4 + ch) * L + p, v);
        }
        a1[pos][ch] = v;              // zero outside [0, L): conv2's zero padding
    }
    __syncthreads();
    // d pre2[p][o] = da2[p][o] * swish'(pre2[p][o])
    for (int i = tid; i < TP * 16; i += 256) {
        const int pos = i >> 4, o = i & 15, p = p0 + pos;
        float g = 0.0f;
        if (p < L) {
            float pre = sb2[o];
#pragma unroll
            for (int ci = 0; ci < 4; ci++)
#pragma unroll
                for (int k = 0; k < 5; k++) pre = fmaf(sw2[(o * 4 + ci) * 5 + k], a1[pos + k][ci], pre);
            g = da2[((size_t)b * L + p) * 16 + o];
            if (DROP && drop.on(1)) g = xb_dropout_apply(drop, 1, ((uint64_t)b * 16 + o) * L + p, g);
            g *= dswishf(pre);
        }
        dp2[pos][o] = g;
    }
    __syncthreads();
    // dW2[o][ci][k] = sum_p d pre2[p][o] * a1[p + k - 2][ci]; db2[o] = sum_p d pre2[p][o]   (336 outputs, one thread each + loop)
    for (int w = tid; w < 336; w += 256) {
        float s = 0.0f;
        if (w < 320) {
            const int o = w / 20, ci = (w / 5) % 4, k = w % 5;
            for (int pos = 0; pos < TP; pos++) s = fmaf(dp2[pos][o], a1[pos + k][ci], s);
            atomicAdd(dw2 + w, s);
        } else {
            const int o = w - 320;
            for (int pos = 0; pos < TP; pos++) s += dp2[pos][o];
            atomicAdd(db2 + o, s);
        }
    }
    // da1[q][ci] += sum_{o,k} w2[o][ci][k] * d pre2[q - k + 2][o]  (positions of this tile only; neighbours add their share)
    for (int i = tid; i < (TP + 4) * 4; i += 256) {
        const int pos = i >> 2, ci = i & 3, q = p0 - 2 + pos;
        if (q < 0 || q >= L) continue;
        float s = 0.0f;
#pragma unroll
        for (int k = 0; k < 5; k++) {
            const int pp = pos - k;               // tile-relative position of the conv2 output: q - k + 2 - p0
            if (pp >= 0 && pp < TP)
#pragma unroll
                for (int o = 0; o < 16; o++) s = fmaf(sw2[(o * 4 + ci) * 5 + k], dp2[pp][o], s);
        }
        if (DROP && drop.on(0)) s = xb_dropout_apply(drop, 0, ((uint64_t)b * 4 + ci) * L + q, s);
        atomicAdd(da1 + ((size_t)b * L + q) * 4 + ci, s);
    }
}

// conv1 backward: d pre1 = da1 * swish'(pre1); dW1 (4,1,5), db1 (4)
template <typename SIG>
__global__ void __launch_bounds__(256)
conv1_bwd_kernel(const SIG *__restrict__ signal, int L, const float *__restrict__ w1, const float *__restrict__ b1,
                 const float *__restrict__ da1, float *__restrict__ dw1, float *__restrict__ db1) {
    __shared__ float acc[24];
    const int b = blockIdx.y, tid = threadIdx.x;
    const SIG *sig = signal + (size_t)b * L;
    if (tid < 24) acc[tid] = 0.0f;
    __syncthreads();
    float loc[24];
#pragma unroll
    for (int i = 0; i < 24; i++) loc[i] = 0.0f;
    for (int p = blockIdx.x * 256 + tid; p < L; p += gridDim.x * 256) {
        float xs[5];
#pragma unroll
        for (int k = 0; k < 5; k++) { const int q = p + k - 2; xs[k] = (q >= 0 && q < L) ? (float)sig[q] : 0.0f; }
#pragma unroll
        for (int ch = 0; ch < 4; ch++) {
            float pre = b1[ch];
#pragma unroll
            for (int k = 0; k < 5; k++) pre = fmaf(w1[ch * 5 + k], xs[k], pre);
            const float g = da1[((size_t)b * L + p) * 4 + ch] * dswishf(pre);
#pragma unroll
            for (int k = 0; k < 5; k++) loc[ch * 5 + k] = fmaf(g, xs[k], loc[ch * 5 + k]);
            loc[20 + ch] += g;
        }
    }
#pragma unroll
    for (int i = 0; i < 24; i++) {
        float v = loc[i];
#pragma unroll
        for (int off = 16; off >= 1; off >>= 1) v += __shfl_xor_sync(0xffffffffu, v, off);
        if ((tid & 31) == 0) atomicAdd(&acc[i], v);
    }
    __syncthreads();
    if (tid < 20) atomicAdd(dw1 + tid, acc[tid]);
    else if (tid < 24) atomicAdd(db1 + tid - 20, acc[tid]);
}

// The three forms of the training step's transpositions (R, C) 16-bit -> (C, R) bf16:
//   TR_BF16_COLSUM  a bf16 gradient, plus the column sums of its first nsum columns (a bias gradient)
//   TR_F16          an fp16 activation
//   TR_F16_DROP     an fp16 activation masked by a dropout site
enum TrForm { TR_BF16_COLSUM, TR_F16, TR_F16_DROP };

// 64 x 64 tiles, 16-byte global loads and stores on both sides (R, C multiples of 8, 16-byte aligned buffers).  Two input
// rows are packed into one 32-bit word per column, so the transposed tile is written and read as words (pitch 33: the read
// side is conflict free, the write side two-way).  Each CTA walks a slab of row tiles; TR_BF16_COLSUM also accumulates the
// column sums of its slab and adds them to colsum_out once -- no separate column-sum pass over the same matrix.
// TR_F16_DROP: the input is masked by dropout site `site` (element index r * C + c) on the way in, rounded to fp16 as the
// forward's dropped copy was, then converted -- the transposed dropped copy without storing it.
template <TrForm FORM>
__global__ void __launch_bounds__(256) transpose16v_kernel(const uint16_t *__restrict__ in, int R, int C,
                                                           __nv_bfloat16 *__restrict__ out, float *__restrict__ colsum_out,
                                                           int nsum, const xb_dropout drop, int site) {
    constexpr bool IN_BF16 = FORM == TR_BF16_COLSUM, COLSUM = FORM == TR_BF16_COLSUM, DROP = FORM == TR_F16_DROP;
    __shared__ uint32_t tileT[64][33];
    const int t = threadIdx.x;
    const int c0 = blockIdx.x * 64;
    const int tiles = (R + 63) / 64, per = (tiles + gridDim.y - 1) / gridDim.y;
    const int tile_lo = blockIdx.y * per, tile_hi = min(tiles, tile_lo + per);
    const int cg = t & 7, rp = t >> 3;                 // load side: 8 columns cg*8.., rows 2*rp and 2*rp + 1
    const int oc = t >> 2, wq = t & 3;                 // store side: output row (input column) oc, words wq*8 .. wq*8 + 7
    float csum = 0.0f;
    auto to_bf16 = [](uint32_t v) -> uint32_t {        // two fp16 -> two bf16
        if (IN_BF16) return v;
        const float2 f = __half22float2(*reinterpret_cast<const __half2 *>(&v));
        const __nv_bfloat162 b = __floats2bfloat162_rn(f.x, f.y);
        return *reinterpret_cast<const uint32_t *>(&b);
    };
    for (int tile = tile_lo; tile < tile_hi; tile++) {
        const int r0 = tile * 64;
        {
            const int r = r0 + 2 * rp, c = c0 + cg * 8;
            uint4 a = make_uint4(0, 0, 0, 0), b = make_uint4(0, 0, 0, 0);
            if (c < C) {
                if (r < R) a = *reinterpret_cast<const uint4 *>(in + (size_t)r * C + c);
                if (r + 1 < R) b = *reinterpret_cast<const uint4 *>(in + (size_t)(r + 1) * C + c);
                if (DROP) {
                    if (r < R) a = xb_dropout8<false>(drop, site, (uint64_t)r * C + c, a);
                    if (r + 1 < R) b = xb_dropout8<false>(drop, site, (uint64_t)(r + 1) * C + c, b);
                }
            }
            const uint32_t av[4] = {to_bf16(a.x), to_bf16(a.y), to_bf16(a.z), to_bf16(a.w)};
            const uint32_t bv[4] = {to_bf16(b.x), to_bf16(b.y), to_bf16(b.z), to_bf16(b.w)};
#pragma unroll
            for (int j = 0; j < 4; j++) {              // word (column, row pair) = {row 2rp (low half), row 2rp + 1 (high half)}
                tileT[cg * 8 + 2 * j][rp] = __byte_perm(av[j], bv[j], 0x5410);
                tileT[cg * 8 + 2 * j + 1][rp] = __byte_perm(av[j], bv[j], 0x7632);
            }
        }
        __syncthreads();
        {
            uint32_t w[8];
#pragma unroll
            for (int k = 0; k < 8; k++) w[k] = tileT[oc][wq * 8 + k];
            const int c = c0 + oc, r = r0 + wq * 16;
            if (c < C) {
                __nv_bfloat16 *o = out + (size_t)c * R + r;
                if (r < R) *reinterpret_cast<uint4 *>(o) = make_uint4(w[0], w[1], w[2], w[3]);
                if (r + 8 < R) *reinterpret_cast<uint4 *>(o + 8) = make_uint4(w[4], w[5], w[6], w[7]);
            }
            if (COLSUM) {
#pragma unroll
                for (int k = 0; k < 8; k++) {           // rows past R were loaded as zeros
                    const float2 f = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162 *>(&w[k]));
                    csum += f.x + f.y;
                }
            }
        }
        __syncthreads();
    }
    if (COLSUM) {
        csum += __shfl_xor_sync(0xffffffffu, csum, 1);
        csum += __shfl_xor_sync(0xffffffffu, csum, 2);
        if (wq == 0 && c0 + oc < nsum) atomicAdd(colsum_out + c0 + oc, csum);
    }
}

// in (R, C) -> out (C, R) bf16 in one of the forms of TrForm.  TR_BF16_COLSUM: colsum_out[0 .. nsum) = the sums of the
// first nsum columns (zeroed here).  TR_F16_DROP: masked by dropout site `site` of *drop.
int transpose_to_bf16(xb_handle *h, TrForm form, const void *in, int R, int C, void *out, cudaStream_t s,
                      float *colsum_out = nullptr, int nsum = 0, const xb_dropout *drop = nullptr, int site = 0) {
    const uint16_t *src = reinterpret_cast<const uint16_t *>(in);
    __nv_bfloat16 *dst = reinterpret_cast<__nv_bfloat16 *>(out);
    xb_stage_timer tm(h, XB_ST_TRAIN_TRANSPOSE, s);
    if (R % 8 || C % 8 || (reinterpret_cast<uintptr_t>(in) & 15) || (reinterpret_cast<uintptr_t>(out) & 15))
        return xb_fail(h, XB_ERR_ARG, "transposition of (%d, %d): rows must be multiples of 8 and buffers 16-byte aligned", R, C);
    const int tiles = (R + 63) / 64, ctiles = (C + 63) / 64;
    int slabs = (h->num_sms * 12 + ctiles - 1) / ctiles;  // ~12 CTAs per SM over the whole grid
    if (slabs > tiles) slabs = tiles;
    if (form == TR_BF16_COLSUM) XB_CUDA(h, cudaMemsetAsync(colsum_out, 0, (size_t)nsum * sizeof(float), s));
    auto k = form == TR_BF16_COLSUM ? transpose16v_kernel<TR_BF16_COLSUM>
             : form == TR_F16       ? transpose16v_kernel<TR_F16>
                                    : transpose16v_kernel<TR_F16_DROP>;
    k<<<dim3(ctiles, slabs), 256, 0, s>>>(src, R, C, dst, colsum_out, nsum, drop ? *drop : xb_dropout(), site);
    XB_LAUNCH_CHECK(h);
    return XB_OK;
}

// in (n 16-bit elements, n % 8 == 0, flat index = element index of the site) -> out, masked by dropout site `site`
int dropout16(xb_handle *h, const void *in, void *out, size_t n, bool bf16, const xb_dropout &drop, int site, cudaStream_t s) {
    const size_t n8 = n / 8;
    const unsigned blocks = (unsigned)std::min<size_t>((n8 + 255) / 256, (size_t)h->num_sms * 16);
    const uint4 *src = reinterpret_cast<const uint4 *>(in);
    uint4 *dst = reinterpret_cast<uint4 *>(out);
    if (bf16) dropout16_kernel<true><<<blocks, 256, 0, s>>>(src, dst, n8, drop, site);
    else dropout16_kernel<false><<<blocks, 256, 0, s>>>(src, dst, n8, drop, site);
    XB_LAUNCH_CHECK(h);
    return XB_OK;
}

// D (M, N) = A (M, K) B (N, K)^T on bf16 operands; out fp32 (EPI_F32) or bf16 (EPI_BF16OUT)
int gemm_bf16(xb_handle *h, int epi, const void *A, int M, int lda, const void *B, int Nn, int ldb, int K, void *out, int ldo,
              cudaStream_t s) {
    CUtensorMap tmA, tmB;
    if (int rc = xb_make_tmap_2d(h, &tmA, A, (uint64_t)M, (uint64_t)K, (uint64_t)lda)) return rc;
    if (int rc = xb_make_tmap_2d(h, &tmB, B, (uint64_t)Nn, (uint64_t)K, (uint64_t)ldb)) return rc;
    GemmParams p;
    p.M = M; p.N = Nn; p.K = K; p.out = out; p.ldo = ldo;
    xb_stage_timer tm(h, epi == EPI_F32 ? XB_ST_TRAIN_WGRAD : XB_ST_TRAIN_XGRAD, s);
    if (epi == EPI_F32) {
        // weight gradients: few output tiles, K = T*N deep -- slice K until the grid covers the SMs (partials added in L2)
        const int tiles = ((M + 127) / 128) * ((Nn + 127) / 128), kb = (K + 63) / 64;
        int split = tiles >= h->num_sms ? 1 : (2 * h->num_sms) / tiles;
        if (split > kb / 8) split = kb / 8 > 0 ? kb / 8 : 1;
        if (split > 1) {
            p.split_k = split;
            XB_CUDA(h, cudaMemsetAsync(out, 0, (size_t)M * ldo * sizeof(float), s));
        }
    }
    return xb_gemm_launch(h, epi, tmA, tmB, p, s, true);
}

}  // namespace

// Every buffer the workspace owns, with its size at the workspace's capacity: train_ws allocates this list and
// xb_train_free frees it.  dpre / dpreT are not in it (aliases of DZ / DZT).
struct ws_buffer { void **p; size_t bytes; };
static std::vector<ws_buffer> ws_buffers(const xb_handle *h, xb_train_ws *w) {
    const size_t TN = (size_t)w->cap_T * w->cap_N, F = XB_FEATURES, HP = h->head_rows_padded;
    const size_t NL = (size_t)w->cap_N * w->cap_T * XB_STRIDE;
    std::vector<ws_buffer> b;
    for (void *&p : w->x) b.push_back({&p, TN * F * 2});
    for (void *&p : w->saved) b.push_back({&p, TN * 5 * F * 2});
    for (void *&p : w->XT) b.push_back({&p, TN * F * 2});
    for (void *&p : w->dy) b.push_back({&p, TN * F * 2});
    b.insert(b.end(), {{&w->DZ, TN * XB_GATES * 2}, {&w->DZT, TN * XB_GATES * 2}, {&w->dzh, TN * HP * 2}, {&w->dzhT, TN * HP * 2},
                       {&w->colT, TN * XB_CONV3_K * 2}, {&w->dcol, TN * XB_CONV3_K * 2},
                       {reinterpret_cast<void **>(&w->dcstate), (size_t)w->cap_N * F * 4},
                       {reinterpret_cast<void **>(&w->dc2), NL * XB_C2_CH * 4},
                       {reinterpret_cast<void **>(&w->dc1), NL * 4 * 4},
                       {&w->xd, TN * F * 2}});
    return b;
}

void xb_train_free(xb_handle *h) {
    xb_train_ws *w = h->train;
    if (!w) return;
    for (const ws_buffer &b : ws_buffers(h, w))
        if (*b.p) cudaFree(*b.p);
    delete w;
    h->train = nullptr;
}

// with_xd: also the scratch copy xd, which only a forward with an active LSTM dropout site needs (kept once allocated)
static int train_ws(xb_handle *h, int N, int T, bool with_xd) {
    if (!(h->flags & XB_FLAG_TRAIN)) return xb_fail(h, XB_ERR_STATE, "the handle was created without XB_FLAG_TRAIN");
    if (h->train && (h->train->cap_N < N || h->train->cap_T < T)) xb_train_free(h);
    if (!h->train) { h->train = new xb_train_ws(); h->train->cap_N = N; h->train->cap_T = T; }
    xb_train_ws *w = h->train;
    for (const ws_buffer &b : ws_buffers(h, w))
        if (b.p != &w->xd || with_xd)
            if (int rc = xb_alloc(h, b.p, b.bytes)) return rc;
    w->dpre = w->DZ;            // conv3's (TN,768) gradients reuse the LSTM buffers (the LSTM layers are done by then)
    w->dpreT = w->DZT;
    return XB_OK;
}

// Model.forward in training (training.py:100): scores (T, N, C*NZ) fp32, activations and LSTM step state kept in the handle;
// p (host, XB_DROPOUT_SITES; NULL = none) and seed: the dropout of rnn_encoder(drop_rate_bottom=...)
static int encoder_fwd_train(xb_handle *h, const void *signal, int sig_dtype, int N, int L, const float *p, uint64_t seed,
                             float *scores, void *stream) {
    if (!h) return xb_fail(nullptr, XB_ERR_ARG, "NULL handle");
    XB_REQUIRE(h, signal && scores, "NULL buffer");
    xb_dropout drop;
    if (int rc = xb_dropout_init(h, &drop, p, seed)) return rc;
    XB_REQUIRE(h, L > 0 && L % XB_STRIDE == 0, "chunk length %d must be a positive multiple of the stride %d", L, XB_STRIDE);
    XB_REQUIRE(h, (h->loaded & 127) == 127, "weights have not been loaded (xb_load_weights)");
    const int T = L / XB_STRIDE;
    XB_REQUIRE(h, T <= h->max_T && N <= h->max_N && N > 0, "T=%d N=%d exceed the handle capacity", T, N);
    // N % 8: the K = T*N contractions read K-major transposed copies through TMA -- their row pitch (T*N 16-bit elements)
    // must be a multiple of 16 bytes, and so must the byte offset of dW_hh's time shift (N elements along such a row:
    // an unaligned box start raises an illegal-instruction error, measured with N = 7)
    XB_REQUIRE(h, N % 8 == 0, "the training path needs a batch that is a multiple of 8 (16-byte TMA alignment of the time-shifted "
                              "operand views); got %d", N);
    XB_CUDA(h, cudaSetDevice(h->device));
    if (int rc = train_ws(h, N, T, drop.active >> 3)) return rc;    // a dropped LSTM output needs the scratch copy xd
    xb_train_ws *w = h->train;
    const size_t TNF = (size_t)T * N * XB_FEATURES;
    w->N = N; w->T = T;
    w->drop = drop;
    cudaStream_t s = reinterpret_cast<cudaStream_t>(stream);
    if (int rc = xb_conv_stem_fwd_dropout(h, signal, sig_dtype, N, L, w->x[0], &drop, stream)) return rc;
    if (drop.on(2)) { if (int rc = dropout16(h, w->x[0], w->x[0], TNF, false, drop, 2, s)) return rc; }
    for (int l = 0; l < 5; l++) {
        const xb_lstm_weights &lw = h->lstm[l];
        const void *in = (l > 0 && drop.on(l + 2)) ? w->xd : w->x[l];
        if (int rc = xb_inproj_launch(h, in, lw.w_ih, lw.bias, h->gates, T * N, s)) return rc;
        if (int rc = xb_lstm_recurrence_persistent(h, l, w->x[l + 1], T, N, (l % 2) == 0, s, w->saved[l])) return rc;
        if (l < 4 && drop.on(l + 3)) { if (int rc = dropout16(h, w->x[l + 1], w->xd, TNF, false, drop, l + 3, s)) return rc; }
    }
    return xb_crf_head_fwd(h, w->x[5], scores, T, N, stream);
}

// ---- the three stages of xb_encoder_bwd.  Each reads the gradient w.r.t. its output and writes the gradient w.r.t. its
// input (the stem: only parameter gradients); the workspace buffers they share are described in xb_train_ws.

// CRF head: dscores -> grads[26], grads[27] and dy_out = d x5 (T,N,768) bf16.  Leaves x5 transposed in XT[1] for layer 4.
static int head_bwd(xb_handle *h, xb_train_ws *w, const float *scores, const float *dscores, float *const *grads, void *dy_out,
                    cudaStream_t s) {
    const int TN = w->T * w->N, F = XB_FEATURES, HP = h->head_rows_padded, S = h->C * h->NZ;
    const size_t n = (size_t)TN * HP;
    {
        xb_stage_timer tm(h, XB_ST_TRAIN_HEAD_CONV, s);
        head_bwd_kernel<<<(unsigned)((n + 255) / 256), 256, 0, s>>>(dscores, scores, (size_t)TN, h->n_base, h->NZ, h->head_rows,
                                                                  HP, h->expand_blanks ? S : h->head_rows, h->expand_blanks,
                                                                  h->scale, reinterpret_cast<__nv_bfloat16 *>(w->dzh));
        XB_LAUNCH_CHECK(h);
    }
    // + db = colsum dz over the head_rows real columns
    if (int rc = transpose_to_bf16(h, TR_BF16_COLSUM, w->dzh, TN, HP, w->dzhT, s, grads[27], h->head_rows)) return rc;
    if (int rc = transpose_to_bf16(h, TR_F16, w->x[5], TN, F, w->XT[1], s)) return rc;
    if (int rc = gemm_bf16(h, EPI_F32, w->dzhT, h->head_rows, TN, w->XT[1], F, TN, TN, grads[26], F, s)) return rc;
    return gemm_bf16(h, EPI_BF16OUT, w->dzh, TN, HP, h->head_wT, F, HP, HP, dy_out, F, s);
}

// LSTM layer l: dy_in = d (output of layer l) -> grads[6 + 4l .. 9 + 4l] and dy_out = d (input of layer l), both (T,N,768)
// bf16.  XT[(l+1) & 1] must hold the transposed output of layer l; leaves the transposed input in XT[l & 1].
static int lstm_layer_bwd(xb_handle *h, xb_train_ws *w, int l, const void *dy_in, void *dy_out, float *const *grads,
                          cudaStream_t s) {
    const int N = w->N, T = w->T, TN = T * N, F = XB_FEATURES;
    const xb_dropout &drop = w->drop;
    const xb_lstm_weights &lw = h->lstm[l];
    const bool reverse = (l % 2) == 0;
    BpttMaps maps;
    if (int rc = xb_bptt_make_maps(h, &maps, w->DZ, lw.w_hhT, w->saved[l], T, N)) return rc;
    {
    xb_stage_timer tm_bptt(h, XB_ST_TRAIN_BPTT, s);
    for (int i = 0; i < T; i++) {                       // forward ran t = (reverse ? T-1 .. 0 : 0 .. T-1); walk it backwards
        const int t = reverse ? i : T - 1 - i;
        const int t_next = reverse ? t - 1 : t + 1;     // the step the forward ran AFTER t (its dz feeds dh_t); i == 0: none
        const int t_prev = reverse ? t + 1 : t - 1;     // the step the forward ran BEFORE t (its c is c_prev)
        BpttStep p;
        p.N = N; p.t_cur = t;
        p.t_next = (i == 0) ? -1 : t_next;
        p.t_prev = (t_prev >= 0 && t_prev < T) ? t_prev : -1;
        p.dy = dy_in; p.dcstate = w->dcstate;
        if (int rc = xb_bptt_step_launch(h, maps, p, /*dependent=*/i > 0, s)) return rc;
    }
    }
    float *g_wih = grads[6 + 4 * l], *g_whh = grads[7 + 4 * l], *g_bih = grads[8 + 4 * l], *g_bhh = grads[9 + 4 * l];
    // + db = colsum DZ
    if (int rc = transpose_to_bf16(h, TR_BF16_COLSUM, w->DZ, TN, XB_GATES, w->DZT, s, g_bih, XB_GATES)) return rc;
    XB_CUDA(h, cudaMemcpyAsync(g_bhh, g_bih, XB_GATES * sizeof(float), cudaMemcpyDeviceToDevice, s));
    if (int rc = transpose_to_bf16(h, TR_F16, w->x[l], TN, F, w->XT[l & 1], s)) return rc;
    // layer l > 0 read the dropped copy of x[l] (site l + 2): dW_ih takes that, transposed through the mask into xd
    const bool drop_in = l > 0 && drop.on(l + 2);
    if (drop_in) { if (int rc = transpose_to_bf16(h, TR_F16_DROP, w->x[l], TN, F, w->xd, s, nullptr, 0, &drop, l + 2)) return rc; }
    // dW_ih = DZ^T x_l and dW_hh = sum over the steps that had a predecessor of dz_t (x) h_prev (a time shift of N columns
    // between DZ^T and Y^T), one launch over 128 x 256 tiles (wgrad_gemm.cu)
    {
        xb_stage_timer tm(h, XB_ST_TRAIN_WGRAD, s);
        if (int rc = xb_lstm_wgrad_launch(h, w->DZT, drop_in ? w->xd : w->XT[l & 1], w->XT[(l + 1) & 1], T, N, reverse, g_wih,
                                          g_whh, s)) return rc;
    }
    if (int rc = gemm_bf16(h, EPI_BF16OUT, w->DZ, TN, XB_GATES, lw.w_ihT, F, XB_GATES, XB_GATES, dy_out, F, s)) return rc;
    // gradient w.r.t. the dropped input -> w.r.t. the output of the layer below (l == 0: the conv3 output, site 2)
    if (drop.on(l + 2)) { if (int rc = dropout16(h, dy_out, dy_out, (size_t)TN * F, true, drop, l + 2, s)) return rc; }
    return XB_OK;
}

// conv2 and conv1 backward of the stem (SIG: the signal's element type): w->dc2 -> grads[0 .. 3], through w->dc1
template <typename SIG>
static int conv12_bwd(xb_handle *h, xb_train_ws *w, const void *signal, float *const *grads, cudaStream_t s) {
    const int N = w->N, L = w->T * XB_STRIDE;
    const xb_dropout &drop = w->drop;
    const SIG *sig = reinterpret_cast<const SIG *>(signal);
    auto conv2 = drop.on(0) || drop.on(1) ? conv2_bwd_kernel<true, SIG> : conv2_bwd_kernel<false, SIG>;
    conv2<<<dim3((L + 255) / 256, N), 256, 0, s>>>(sig, L, h->conv1_w, h->conv1_b, h->conv2_w, h->conv2_b, w->dc2, w->dc1,
                                                  grads[2], grads[3], drop);
    XB_LAUNCH_CHECK(h);
    conv1_bwd_kernel<SIG><<<dim3(4, N), 256, 0, s>>>(sig, L, h->conv1_w, h->conv1_b, w->dc1, grads[0], grads[1]);
    XB_LAUNCH_CHECK(h);
    return XB_OK;
}

// convolution stem: dy_in = d x0 (T,N,768) bf16 -> grads[0 .. 5]
static int stem_bwd(xb_handle *h, xb_train_ws *w, const void *signal, int sig_dtype, const void *dy_in, float *const *grads,
                    cudaStream_t s) {
    const int N = w->N, T = w->T, TN = T * N, F = XB_FEATURES, L = T * XB_STRIDE;
    if (int rc = xb_conv12_im2col(h, signal, sig_dtype, N, L, s, &w->drop)) return rc;   // im2col rows of this batch into h->c2
    CUtensorMap tmA, tmB;
    if (int rc = xb_make_tmap_2d(h, &tmA, h->c2, (uint64_t)TN, XB_CONV3_K, XB_CONV3_K)) return rc;
    if (int rc = xb_make_tmap_2d(h, &tmB, h->conv3_w, F, XB_CONV3_K, XB_CONV3_K)) return rc;
    GemmParams p;
    p.M = TN; p.N = F; p.K = XB_CONV3_K; p.bias = h->conv3_b; p.out = w->dpre; p.ldo = F; p.T = T; p.NB = N; p.dy = dy_in;
    {
        xb_stage_timer tm(h, XB_ST_TRAIN_HEAD_CONV, s);
        if (int rc = xb_gemm_launch(h, EPI_CONV3_BWD, tmA, tmB, p, s, false)) return rc;
    }
    // + db3 = colsum d pre
    if (int rc = transpose_to_bf16(h, TR_BF16_COLSUM, w->dpre, TN, F, w->dpreT, s, grads[5], F)) return rc;
    if (int rc = transpose_to_bf16(h, TR_F16, h->c2, TN, XB_CONV3_K, w->colT, s)) return rc;
    // dW3 in im2col column order (768, 320): the caller drops the 16 padding columns and permutes to (768, 16, 19)
    if (int rc = gemm_bf16(h, EPI_F32, w->dpreT, F, TN, w->colT, XB_CONV3_K, TN, TN, grads[4], XB_CONV3_K, s)) return rc;
    if (int rc = gemm_bf16(h, EPI_BF16OUT, w->dpre, TN, F, h->conv3_wT, XB_CONV3_K, F, F, w->dcol, XB_CONV3_K, s)) return rc;
    xb_stage_timer tm(h, XB_ST_TRAIN_HEAD_CONV, s);
    const size_t n2 = (size_t)N * L * XB_C2_CH;
    col2im_kernel<<<(unsigned)((n2 + 255) / 256), 256, 0, s>>>(reinterpret_cast<const __nv_bfloat16 *>(w->dcol), N, T, L, w->dc2);
    XB_LAUNCH_CHECK(h);
    XB_CUDA(h, cudaMemsetAsync(w->dc1, 0, (size_t)N * L * 4 * sizeof(float), s));
    XB_CUDA(h, cudaMemsetAsync(grads[2], 0, 320 * sizeof(float), s));
    XB_CUDA(h, cudaMemsetAsync(grads[3], 0, 16 * sizeof(float), s));
    XB_CUDA(h, cudaMemsetAsync(grads[0], 0, 20 * sizeof(float), s));
    XB_CUDA(h, cudaMemsetAsync(grads[1], 0, 4 * sizeof(float), s));
    return sig_dtype == XB_SIG_F32 ? conv12_bwd<float>(h, w, signal, grads, s) : conv12_bwd<int16_t>(h, w, signal, grads, s);
}

extern "C" {

int xb_encoder_fwd_train(xb_handle *h, const void *signal, int sig_dtype, int N, int L, float *scores, void *stream) {
    return encoder_fwd_train(h, signal, sig_dtype, N, L, nullptr, 0, scores, stream);
}

int xb_encoder_fwd_train_dropout(xb_handle *h, const void *signal, int sig_dtype, int N, int L, const float *p, uint64_t seed,
                                 float *scores, void *stream) {
    return encoder_fwd_train(h, signal, sig_dtype, N, L, p, seed, scores, stream);
}

int xb_dropout_keep(uint64_t seed, int site, float p, int64_t n, uint8_t *keep, void *stream) {
    if (site < 0 || site >= XB_DROPOUT_SITES) return xb_fail(nullptr, XB_ERR_ARG, "dropout site %d out of range", site);
    if (n < 0 || (n > 0 && !keep)) return xb_fail(nullptr, XB_ERR_ARG, "bad keep buffer");
    float ps[XB_DROPOUT_SITES] = {};
    ps[site] = p;
    xb_dropout drop;
    if (int rc = xb_dropout_init(nullptr, &drop, ps, seed)) return rc;
    if (n == 0) return XB_OK;
    int dev = 0, sms = 0;
    XB_CUDA(nullptr, cudaGetDevice(&dev));
    XB_CUDA(nullptr, cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
    const unsigned blocks = (unsigned)std::min<int64_t>((n + 255) / 256, (int64_t)sms * 16);
    dropout_keep_kernel<<<blocks, 256, 0, reinterpret_cast<cudaStream_t>(stream)>>>(drop, site, n, keep);
    XB_CUDA(nullptr, cudaGetLastError());
    return XB_OK;
}

// Backward of the last xb_encoder_fwd_train.  signal / scores: the buffers of that forward; dscores (T,N,C*NZ) fp32.
// grads: XB_NUM_WEIGHTS fp32 device tensors in xb_load_weights' order and the reference's layouts, except
// encoder.2.conv.weight, whose gradient is written as (768, 320) = [out][tap * 16 + in] (im2col column order, the last 16
// columns are padding; the caller reshapes to (768, 16, 19)).
int xb_encoder_bwd(xb_handle *h, const void *signal, int sig_dtype, const float *scores, const float *dscores, float *const *grads,
                   int n_tensors, void *stream) {
    return xb_encoder_bwd_stages(h, 6, 0, signal, sig_dtype, scores, dscores, nullptr, nullptr, grads, n_tensors, stream);
}

// Stages top .. bottom of the same backward (6 head, 5 .. 1 LSTM layers 4 .. 0, 0 stem); include/xna_basecaller.h.
int xb_encoder_bwd_stages(xb_handle *h, int top, int bottom, const void *signal, int sig_dtype, const float *scores,
                          const float *dscores, const void *dy_top, void *dy_bottom, float *const *grads, int n_tensors,
                          void *stream) {
    if (!h) return xb_fail(nullptr, XB_ERR_ARG, "NULL handle");
    XB_REQUIRE(h, h->train && h->train->T > 0, "xb_encoder_bwd needs a preceding xb_encoder_fwd_train");
    XB_REQUIRE(h, 0 <= bottom && bottom <= top && top <= 6, "bad stage range %d .. %d (need 6 >= top >= bottom >= 0)", top, bottom);
    XB_REQUIRE(h, grads && n_tensors == XB_NUM_WEIGHTS, "bad arguments");
    XB_REQUIRE(h, top < 6 || (scores && dscores), "the head stage needs scores and dscores");
    XB_REQUIRE(h, top == 6 || (dy_top && (reinterpret_cast<uintptr_t>(dy_top) & 15) == 0),
               "stage %d needs dy_top, 16-byte aligned", top);
    XB_REQUIRE(h, bottom == 0 || (dy_bottom && (reinterpret_cast<uintptr_t>(dy_bottom) & 15) == 0),
               "stage %d needs dy_bottom, 16-byte aligned", bottom);
    XB_REQUIRE(h, bottom > 0 || signal, "the stem stage needs the signal");
    XB_REQUIRE(h, bottom > 0 || sig_dtype == XB_SIG_F32 || sig_dtype == XB_SIG_I16, "the backward reads fp32 or int16 signal");
    // parameter tensors of stage k: 6 -> 26, 27; k in 1..5 (LSTM layer k-1) -> 4k+2 .. 4k+5; 0 -> 0 .. 5
    for (int k = bottom; k <= top; k++) {
        const int lo = k == 6 ? 26 : k == 0 ? 0 : 4 * k + 2, hi = k == 6 ? 27 : 4 * k + 5;
        for (int i = lo; i <= hi; i++) XB_REQUIRE(h, grads[i] != nullptr, "gradient tensor %d is NULL", i);
    }
    if (h->train->drop.active && !(top == 6 && bottom == 0))
        return xb_fail(h, XB_ERR_UNSUPPORTED, "the last forward applied dropout: only the whole backward (stages 6 .. 0) runs");
    XB_CUDA(h, cudaSetDevice(h->device));
    xb_train_ws *w = h->train;
    cudaStream_t s = reinterpret_cast<cudaStream_t>(stream);
    // stage k's outgoing gradient: dy_bottom for the last stage, else the workspace buffer the next stage reads
    const void *dy = dy_top;
    if (top == 6) {
        void *out = bottom == 6 ? dy_bottom : w->dy[1];
        if (int rc = head_bwd(h, w, scores, dscores, grads, out, s)) return rc;
        dy = out;
    } else if (top >= 1) {
        // layer top-1 reads its own output transposed, which the stage above it leaves behind in a chained backward
        const int l = top - 1;
        if (int rc = transpose_to_bf16(h, TR_F16, w->x[l + 1], w->T * w->N, XB_FEATURES, w->XT[(l + 1) & 1], s)) return rc;
    }
    for (int k = std::min(top, 5); k >= std::max(bottom, 1); k--) {
        const int l = k - 1;
        void *out = k == bottom ? dy_bottom : w->dy[l & 1];
        if (int rc = lstm_layer_bwd(h, w, l, dy, out, grads, s)) return rc;
        dy = out;
    }
    if (bottom == 0) return stem_bwd(h, w, signal, sig_dtype, dy, grads, s);
    return XB_OK;
}

}  // extern "C"
