// One step of back-propagation through time of an LSTM layer (the backward of bonito/nn.py:189-193's torch.nn.LSTM),
// tcgen05 + TMA, sm_100a.  The training step launches it T times per layer, walking the forward's order backwards:
//
//   dh_t   = dz_{t_next} W_hh  +  dy_t                       (M = chunks, N = 768 hidden units, K = 3072 gate rows)
//   dc     = dh o (1 - tanh^2 c) + dc_next;   do = dh tanh c;   di = dc g;   dg = dc i;   df = dc c_prev;   dc_prev = dc f
//   dz_t   = (di i(1-i), df f(1-f), dg (1-g^2), do o(1-o))    -> DZ[t], bf16, the reference's gate-row order
//
// Each CTA owns a [128 chunks x 64 hidden units] tile of dh (grid 12 x ceil(N/128): 48 CTAs at N = 512).
//   * Everything a step needs that does NOT depend on the previous step -- the saved gates i, f, g, o, c of step t, the
//     cell state of step t_prev, W_hh's first tiles, dy_t -- is fetched BEFORE griddepcontrol.wait: the kernels are chained
//     with programmatic dependent launches, so that fetch (and the prologue: barriers, TMEM allocation, descriptor
//     prefetch) runs while the previous step is still computing on other SMs.  Only dz_{t_next} (A operand) and the carried
//     cell gradient are read after the wait.
//   * The saved state arrives by TMA as [gate][chunk][64 units] blocks with the 128-byte swizzle: thread = chunk (the TMEM
//     lane of the accumulator) reads its row 16 bytes at a time without bank conflicts, instead of the row-strided global
//     loads of the tile-GEMM epilogue this kernel replaces (57 us per step).
//   * dz is written in place over the staged gates and leaves as one TMA tensor store, clipped by the tensor map at the
//     batch edge.
//
// Where a step's 17.8 us go (globaltimer stamps of one CTA, N = 512, mid-layer; the kernel is resident ~35 us = two steps
// before it is needed): previous step's dz store complete -> +1.4 us griddepcontrol.wait returns -> +0.9 us first A tile in
// shared memory -> +11.4 us main loop (48 K blocks, 1.15 MB through one SM's L2 port) -> +2.6..3.6 us cell backward -> +1.5 us
// dz staged, TMA store issued and drained.  Sixteen epilogue warps with the MUFU tanh shortened the cell backward by 1 us
// on that CTA's clock without moving the step time (69.2 against 69.3 ms per backward); eight warps and tanhf stay.
//
// Warp roles (384 threads): warp 0 = TMA producer, warp 1 = MMA issuer, warp 2 = TMEM allocator, warps 4..11 = cell
// backward (warp w: TMEM lane quadrant w % 4, hidden units 32 * ((w - 4) / 4) .. + 31 of the tile).
#include "xb_common.cuh"
#include "xb_ptx.cuh"
#include "xb_gemm.cuh"

#include <cuda_bf16.h>
#include <cuda_fp16.h>

using namespace xbptx;

namespace {

constexpr int BM = 128, BU = 64, BK = 64;
constexpr int A_BYTES = BM * BK * 2, B_BYTES = BU * BK * 2, STAGE_BYTES = A_BYTES + B_BYTES;
constexpr int STAGES = 5;                                   // 120 KB in flight per SM: the main loop is bound by the L2 -> SM round trip
constexpr int GATE_BYTES = BM * 128;                        // one [128 chunks][64 units] 16-bit block
constexpr int OFF_SAVED = STAGES * STAGE_BYTES;             // i, f, g, o, c blocks; dz overwrites the first four
constexpr int OFF_CPREV = OFF_SAVED + 5 * GATE_BYTES;
constexpr int OFF_BAR = OFF_CPREV + GATE_BYTES;
constexpr int SMEM_BYTES = OFF_BAR + 256 + 1024 /*align slack*/;
constexpr int THREADS = 384;
static_assert(OFF_SAVED % 1024 == 0 && SMEM_BYTES <= 232448, "shared memory plan");

struct StepParams {
    int N, t_cur, t_prev, a_row, first;
    const __nv_bfloat16 *dy;
    float *dcstate;
};

__device__ __forceinline__ void unpack8h(const uint4 &raw, float (&o)[8]) {
    const __half2 *h2 = reinterpret_cast<const __half2 *>(&raw);
#pragma unroll
    for (int j = 0; j < 4; j++) {
        const float2 f = __half22float2(h2[j]);
        o[2 * j] = f.x;
        o[2 * j + 1] = f.y;
    }
}
__device__ __forceinline__ uint4 pack8b(const float (&v)[8]) {
    uint4 raw;
    __nv_bfloat162 *b2 = reinterpret_cast<__nv_bfloat162 *>(&raw);
#pragma unroll
    for (int j = 0; j < 4; j++) b2[j] = __floats2bfloat162_rn(v[2 * j], v[2 * j + 1]);
    return raw;
}

__global__ void __launch_bounds__(THREADS, 1)
lstm_bptt_step_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB,
                      const __grid_constant__ CUtensorMap tmS, const __grid_constant__ CUtensorMap tmC,
                      const __grid_constant__ CUtensorMap tmZ, const StepParams p) {
    extern __shared__ uint8_t smem_raw[];
    uint8_t *smem = reinterpret_cast<uint8_t *>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
    uint64_t *full = reinterpret_cast<uint64_t *>(smem + OFF_BAR);
    uint64_t *empty = full + STAGES;
    uint64_t *tmem_full = empty + STAGES;
    uint64_t *state_full = tmem_full + 1;
    uint32_t *tmem_holder = reinterpret_cast<uint32_t *>(state_full + 1);

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int u0 = blockIdx.x * BU, m0 = blockIdx.y * BM;
    const int kblocks = p.first ? 0 : XB_GATES / BK;

    if (warp == 0 && lane == 0) {
        prefetch_tmap(&tmA);
        prefetch_tmap(&tmB);
        prefetch_tmap(&tmS);
        prefetch_tmap(&tmC);
        prefetch_tmap(&tmZ);
    }
    if (warp == 1 && lane == 0) {
        for (int s = 0; s < STAGES; s++) {
            mbar_init(&full[s], 1);
            mbar_init(&empty[s], 1);
        }
        mbar_init(tmem_full, 1);
        mbar_init(state_full, 1);
        fence_barrier_init();
    }
    if (warp == 2) {
        tmem_alloc(tmem_holder, BU);
        tmem_relinquish();
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_holder;
    griddep_launch_dependents();             // the next step may start its own prologue and state fetch on idle SMs

    if (warp == 0) {
        if (elect_one()) {
            mbar_expect_tx(state_full, (p.t_prev >= 0 ? 6 : 5) * GATE_BYTES);
            tma_load_4d(smem + OFF_SAVED, &tmS, state_full, u0, m0, 0, p.t_cur);
            if (p.t_prev >= 0) tma_load_4d(smem + OFF_CPREV, &tmC, state_full, u0, m0, 4, p.t_prev);
            const int npre = kblocks < STAGES ? kblocks : STAGES;
            for (int kb = 0; kb < npre; kb++) {                 // weights: not produced by the previous step
                mbar_expect_tx(&full[kb], STAGE_BYTES);
                tma_load_2d(smem + kb * STAGE_BYTES + A_BYTES, &tmB, &full[kb], kb * BK, u0);
            }
            griddep_wait();                                     // dz_{t_next} is complete and visible from here on
            for (int kb = 0; kb < npre; kb++) tma_load_2d(smem + kb * STAGE_BYTES, &tmA, &full[kb], kb * BK, p.a_row + m0);
            for (int kb = npre; kb < kblocks; kb++) {
                const int s = kb % STAGES;
                mbar_wait(&empty[s], ((kb / STAGES) & 1) ^ 1);
                mbar_expect_tx(&full[s], STAGE_BYTES);
                uint8_t *sa = smem + s * STAGE_BYTES;
                tma_load_2d(sa, &tmA, &full[s], kb * BK, p.a_row + m0);
                tma_load_2d(sa + A_BYTES, &tmB, &full[s], kb * BK, u0);
            }
        }
    } else if (warp == 1) {
        constexpr uint32_t idesc = umma_idesc_f16(1u, BM, BU);
        for (int kb = 0; kb < kblocks; kb++) {
            const int s = kb % STAGES;
            mbar_wait(&full[s], (kb / STAGES) & 1);
            tc_fence_after();
            if (elect_one()) {
                const uint32_t a_addr = smem_u32(smem + s * STAGE_BYTES);
                const uint32_t b_addr = a_addr + A_BYTES;
#pragma unroll
                for (int k = 0; k < BK / 16; k++)
                    mma_f16_ss(tmem_base, umma_desc_sw128(a_addr + k * 32), umma_desc_sw128(b_addr + k * 32), idesc, (kb | k) != 0);
                mma_commit(&empty[s]);
                if (kb == kblocks - 1) mma_commit(tmem_full);
            }
            __syncwarp();
        }
    } else if (warp >= 4) {
        const int q = warp & 3, half = (warp - 4) >> 2;
        const int r = q * 32 + lane;                           // tile row = chunk = TMEM lane
        const int m = m0 + r;
        const bool row_ok = m < p.N;
        const int uh = u0 + half * 32;                         // first hidden unit of this thread
        // gradient from the layer above: independent of the previous step
        uint4 dyraw[4];
        {
            const uint4 *src = reinterpret_cast<const uint4 *>(p.dy + ((size_t)p.t_cur * p.N + (row_ok ? m : 0)) * XB_FEATURES + uh);
#pragma unroll
            for (int j = 0; j < 4; j++) dyraw[j] = row_ok ? __ldg(src + j) : make_uint4(0, 0, 0, 0);
        }
        griddep_wait();
        float *dcs = p.dcstate + (size_t)(row_ok ? m : 0) * XB_FEATURES + uh;
        float4 dcin[8];
#pragma unroll
        for (int j = 0; j < 8; j++)
            dcin[j] = (row_ok && !p.first) ? *reinterpret_cast<const float4 *>(dcs + 4 * j) : make_float4(0.f, 0.f, 0.f, 0.f);
        uint32_t acc[32];
        if (kblocks > 0) {
            mbar_wait(tmem_full, 0);
            tc_fence_after();
            tmem_ld_32x32b_x32(tmem_base + ((uint32_t)(q * 32) << 16) + half * 32, acc);
            tmem_ld_wait();
        } else {
#pragma unroll
            for (int j = 0; j < 32; j++) acc[j] = 0u;
        }
        mbar_wait(state_full, 0);
        const uint32_t row_addr = smem_u32(smem + OFF_SAVED) + r * 128;
        const uint32_t cprev_addr = smem_u32(smem + OFF_CPREV) + r * 128;
#pragma unroll
        for (int j8 = 0; j8 < 4; j8++) {
            const uint32_t swz = (uint32_t)(((half * 4 + j8) ^ (r & 7)) << 4);      // 128B swizzle: 16-byte chunk ^ (row mod 8)
            float gi[8], gf[8], gg[8], go[8], cc[8], cprev[8], dyv[8];
            unpack8h(lds_v4(row_addr + 0 * GATE_BYTES + swz), gi);
            unpack8h(lds_v4(row_addr + 1 * GATE_BYTES + swz), gf);
            unpack8h(lds_v4(row_addr + 2 * GATE_BYTES + swz), gg);
            unpack8h(lds_v4(row_addr + 3 * GATE_BYTES + swz), go);
            unpack8h(lds_v4(row_addr + 4 * GATE_BYTES + swz), cc);
            if (p.t_prev >= 0) unpack8h(lds_v4(cprev_addr + swz), cprev);
            else {
#pragma unroll
                for (int j = 0; j < 8; j++) cprev[j] = 0.0f;
            }
            {
                const __nv_bfloat162 *b2 = reinterpret_cast<const __nv_bfloat162 *>(&dyraw[j8]);
#pragma unroll
                for (int j = 0; j < 4; j++) { const float2 f = __bfloat1622float2(b2[j]); dyv[2 * j] = f.x; dyv[2 * j + 1] = f.y; }
            }
            const float dci[8] = {dcin[2 * j8].x, dcin[2 * j8].y, dcin[2 * j8].z, dcin[2 * j8].w,
                                  dcin[2 * j8 + 1].x, dcin[2 * j8 + 1].y, dcin[2 * j8 + 1].z, dcin[2 * j8 + 1].w};
            float dzi[8], dzf[8], dzg[8], dzo[8], dcp[8];
#pragma unroll
            for (int j = 0; j < 8; j++) {
                const float dh = __uint_as_float(acc[8 * j8 + j]) + dyv[j];
                const float tc = tanhf(cc[j]);
                const float dc = dh * go[j] * (1.0f - tc * tc) + dci[j];
                dzo[j] = dh * tc * go[j] * (1.0f - go[j]);
                dzi[j] = dc * gg[j] * gi[j] * (1.0f - gi[j]);
                dzg[j] = dc * gi[j] * (1.0f - gg[j] * gg[j]);
                dzf[j] = dc * cprev[j] * gf[j] * (1.0f - gf[j]);
                dcp[j] = dc * gf[j];
            }
            sts_v4(row_addr + 0 * GATE_BYTES + swz, pack8b(dzi));
            sts_v4(row_addr + 1 * GATE_BYTES + swz, pack8b(dzf));
            sts_v4(row_addr + 2 * GATE_BYTES + swz, pack8b(dzg));
            sts_v4(row_addr + 3 * GATE_BYTES + swz, pack8b(dzo));
            if (row_ok) {
                *reinterpret_cast<float4 *>(dcs + 8 * j8) = make_float4(dcp[0], dcp[1], dcp[2], dcp[3]);
                *reinterpret_cast<float4 *>(dcs + 8 * j8 + 4) = make_float4(dcp[4], dcp[5], dcp[6], dcp[7]);
            }
        }
        fence_proxy_async();                                    // generic-proxy writes of dz -> visible to the TMA store
        named_bar_sync(1, 256);
        if (warp == 4 && elect_one()) {
            tma_store_4d(&tmZ, smem_u32(smem + OFF_SAVED), u0, m0, 0, p.t_cur);     // rows >= N are clipped by the map
            bulk_commit_group();
            bulk_wait_group0();
        }
        tc_fence_before();
    }
    __syncthreads();
    if (warp == 2) {
        tc_fence_after();
        tmem_dealloc(tmem_base, BU);
    }
}

}  // namespace

int xb_bptt_make_maps(xb_handle *h, BpttMaps *m, const void *dz, const void *w_hhT, const void *saved, int T, int N) {
    const uint64_t F = XB_FEATURES, G = XB_GATES;
    if (int rc = xb_make_tmap_2d(h, &m->dz_rows, dz, (uint64_t)T * N, G, G)) return rc;
    {
        const uint64_t dims[2] = {G, F}, st[1] = {G * 2};
        const uint32_t box[2] = {BK, BU};
        if (int rc = xb_make_tmap_nd(h, &m->w_hhT, w_hhT, 2, 2, dims, st, box, CU_TENSOR_MAP_SWIZZLE_128B)) return rc;
    }
    {
        const uint64_t dims[4] = {F, (uint64_t)N, 5, (uint64_t)T};
        const uint64_t st[3] = {5 * F * 2, F * 2, (uint64_t)N * 5 * F * 2};
        const uint32_t box5[4] = {64, BM, 5, 1}, box1[4] = {64, BM, 1, 1};
        if (int rc = xb_make_tmap_nd(h, &m->saved, saved, 4, 2, dims, st, box5, CU_TENSOR_MAP_SWIZZLE_128B)) return rc;
        if (int rc = xb_make_tmap_nd(h, &m->saved_c, saved, 4, 2, dims, st, box1, CU_TENSOR_MAP_SWIZZLE_128B)) return rc;
    }
    {
        const uint64_t dims[4] = {F, (uint64_t)N, 4, (uint64_t)T};
        const uint64_t st[3] = {G * 2, F * 2, (uint64_t)N * G * 2};
        const uint32_t box[4] = {64, BM, 4, 1};
        if (int rc = xb_make_tmap_nd(h, &m->dz_out, dz, 4, 2, dims, st, box, CU_TENSOR_MAP_SWIZZLE_128B)) return rc;
    }
    return XB_OK;
}

int xb_bptt_step_launch(xb_handle *h, const BpttMaps &m, const BpttStep &p, bool dependent, cudaStream_t s) {
    if (int rc = xb_smem_attr(h, lstm_bptt_step_kernel, SMEM_BYTES)) return rc;
    StepParams sp;
    sp.N = p.N; sp.t_cur = p.t_cur; sp.t_prev = p.t_prev;
    sp.first = p.t_next < 0;
    sp.a_row = sp.first ? 0 : p.t_next * p.N;
    sp.dy = reinterpret_cast<const __nv_bfloat16 *>(p.dy);
    sp.dcstate = p.dcstate;
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(XB_FEATURES / BU, (p.N + BM - 1) / BM);
    cfg.blockDim = dim3(THREADS);
    cfg.dynamicSmemBytes = SMEM_BYTES;
    cfg.stream = s;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr;
    cfg.numAttrs = dependent ? 1 : 0;       // the first step of a layer serialises fully behind the kernels before it
    XB_CUDA(h, cudaLaunchKernelEx(&cfg, lstm_bptt_step_kernel, m.dz_rows, m.w_hhT, m.saved, m.saved_c, m.dz_out, sp));
    return XB_OK;
}
