// Persistent-weight bidirectional LSTM recurrence on tcgen05 (Clair3_P's LSTM1 / LSTM2,
// clair3/model.py:96-107,132-133; torch nn.LSTM semantics: gate rows i,f,g,o, h0 = c0 = 0, the reverse direction
// walks t = 32..0 and both directions are concatenated per time step).
//
// One CTA owns (two sub-tiles of NB candidate sites) x (one direction) for all 33 steps.  The gate GEMM is issued
// "swapped": the recurrent weight matrix is the UMMA A operand (gate rows -> the 128 TMEM lanes, one 128-row block per
// gate), the activations [x_t ; h_{t-1}] of a sub-tile's NB sites are the B operand (sites -> TMEM columns).  So
//   * the whole weight matrix stays on chip for the 33 steps (160 KB LSTM1; LSTM2: 160 KB in shared memory + its fifth
//     row block as a TMEM-resident A operand), loaded once per CTA from a host-packed SWIZZLE_NONE K-major image;
//   * epilogue thread r owns hidden unit r: it reads its i,f,g,o pre-activations for every site of the sub-tile from four
//     TMEM column ranges of its own lane, keeps the cell state c[NB] in fp32 registers for the whole sequence, and writes
//     h_t (fp16) back into the B-operand buffer for step t+1 - no cross-thread exchange, no grid-wide sync;
//   * the two sub-tiles ping-pong: while warpgroup 0 runs the sigma/tanh/cell epilogue of sub-tile 0 (MUFU-bound), the
//     MMA warp issues the gate GEMM of sub-tile 1, and vice versa, so the tensor pipe and the MUFU pipe overlap.
//     Measured on B200: a 128xNx16 tcgen05.mma costs ~44 cycles for any N <= 64 (65 at N=128, 128 at N=256), so the
//     per-step tensor time is fixed (40-50 MMAs) and wide sub-tiles amortise it.
//
// LSTM1 (H=128): K = 48 + 128.  The 48 x columns are [hi(x) (18) | 1 | lo(x) (18) | 0...]: the raw counts are unbounded integers
// (the reference's GPU branch does not rescale depth, clair3/CallVariantsFromCffi.py:299-353), fp16 is exact only to 2048, so
// every count is split as x = hi + lo with hi = fp16(x) and lo = fp16(x - hi) - exact for |x| <= 67 552 (hi stops at 65 504) -
// and W_ih multiplies both parts (fp32 accumulate: the same result as an exact-input product).  Column 18 is a constant 1 that
// carries b_ih + b_hh, so the x projection and the bias are fused into the same MMAs.  
// LSTM2 (H=160, input 256): the input projection W_ih*h1 (+bias) is a separate big GEMM
// (proj_tc.cu) that leaves fp16 pre-gates in the thread-friendly layout pgT[dir][t][subtile][blk][row][NB]; this kernel
// keeps only W_hh on chip (K = 160).  Units 0..127 are lane-aligned in row blocks 0..3; units 128..159 live in a fifth
// block laid out [i(32) f(32) g(32) o(32)] whose activated gates cross warps through a small shared-memory exchange.
// The sigmoid gates' rows are pre-halved on the host so sigma(x) = 0.5*tanh(x/2)+0.5 is one MUFU + one FMA.
//
// h_t leaves the CTA as 16-byte chunks copied from the operand buffer while the next step's MMAs run.
#include <type_traits>

#include "c3b_internal.h"
#include "ptx.cuh"

namespace {

constexpr int kWgThreads = 128;                // one epilogue warpgroup = one thread per TMEM lane
// block = 2 sub-tiles x WG epilogue warpgroups + the MMA warp (WG = 2: the two warpgroups of a sub-tile split its sites,
// so twice as many warps hide the epilogue's TMEM / MUFU / shared-memory latencies: the epilogue is latency-bound)

struct LstmDev {
    const op_t *w_img;             // [dir][NBLK][K/8][128][8]
    const op_t *xs;                // LSTM1 input  [33][Bp][48]: hi | 1 | lo columns
    const __half *pg;              // LSTM2 pre-gates pgT[dir][33][Bp/NB][5][128][NB]
    op_t *hout;                    // tile-major k-group-planar: LSTM1 h1 (rows t*Bp+b, 32 k-groups); LSTM2 h2 (rows b, 1320 k-groups)
    int bp;                        // padded batch
    long long *trace;              // optional [33][4] clock64 stamps of CTA (0,0) thread 0 (debug option "lstm_trace")
};

__device__ __forceinline__ void lstm_cell8(const float *gi, const float *gf, const float *gg, const float *go, float *c,
                                           float *h) {
#pragma unroll
    for (int i = 0; i < 8; ++i) {
        const float iv = ptx::sigmoid_prehalved(gi[i]);
        const float fv = ptx::sigmoid_prehalved(gf[i]);
        const float gv = ptx::tanh_approx(gg[i]);
        const float ov = ptx::sigmoid_prehalved(go[i]);
        c[i] = fmaf(fv, c[i], iv * gv);
        h[i] = ov * ptx::tanh_approx(c[i]);
    }
}

// Packed variant: the four gate activations and tanh(c) of two neighbouring sites share one MUFU op each
// (tanh.approx.f16x2: 2.5 MUFU ops per cell instead of 5 - the SFU is what bounds the fp32 epilogue); i*g and o*tanh(c) are packed
// fp16 multiplies, the cell state and its update stay fp32.  Returns h as four packed (site, site+1) fp16 pairs.
__device__ __forceinline__ uint32_t pack_f16x2(float lo, float hi) {
    uint32_t r;
    asm("cvt.rn.f16x2.f32 %0, %1, %2;" : "=r"(r) : "f"(hi), "f"(lo));
    return r;
}
__device__ __forceinline__ uint32_t tanh_f16x2(uint32_t x) {
    uint32_t r;
    asm("tanh.approx.f16x2 %0, %1;" : "=r"(r) : "r"(x));
    return r;
}
__device__ __forceinline__ uint32_t sigm_f16x2(uint32_t xh) {      // sigma of a pre-halved argument pair: 0.5 * tanh(xh) + 0.5
    uint32_t r;
    const uint32_t half2 = 0x38003800u;
    asm("fma.rn.f16x2 %0, %1, %2, %2;" : "=r"(r) : "r"(tanh_f16x2(xh)), "r"(half2));
    return r;
}
__device__ __forceinline__ uint32_t mul_f16x2(uint32_t a, uint32_t b) {
    uint32_t r;
    asm("mul.rn.f16x2 %0, %1, %2;" : "=r"(r) : "r"(a), "r"(b));
    return r;
}
__device__ __forceinline__ void lstm_cell8_h2(const float *gi, const float *gf, const float *gg, const float *go, float *c,
                                              uint32_t *hp) {
#pragma unroll
    for (int i = 0; i < 8; i += 2) {
        const uint32_t iv = sigm_f16x2(pack_f16x2(gi[i], gi[i + 1]));
        const uint32_t gv = tanh_f16x2(pack_f16x2(gg[i], gg[i + 1]));
        const uint32_t ig = mul_f16x2(iv, gv);
        const uint32_t fv = sigm_f16x2(pack_f16x2(gf[i], gf[i + 1]));
        const float2 f2 = __half22float2(*reinterpret_cast<const __half2 *>(&fv));
        const float2 g2 = __half22float2(*reinterpret_cast<const __half2 *>(&ig));
        c[i] = fmaf(f2.x, c[i], g2.x);
        c[i + 1] = fmaf(f2.y, c[i + 1], g2.y);
        const uint32_t ov = sigm_f16x2(pack_f16x2(go[i], go[i + 1]));
        hp[i >> 1] = mul_f16x2(ov, tanh_f16x2(pack_f16x2(c[i], c[i + 1])));
    }
}

// Element offset of the 8-unit group `kgh` of site `b` at time t in the layer's output, TILE-MAJOR k-group-planar
// [row tile of 128][k-groups][128 rows][8] (c3b_tile_major_offset): LSTM1 -> h1 (row = t*bp + b, 32 k-groups: dir*16 + kgh),
// LSTM2 -> h2 (row = b, 1320 k-groups: t*40 + dir*20 + kgh = the flatten order of clair3/model.py:135).
template <bool LAYER2>
__device__ __forceinline__ size_t h_out_offset(int t, int dir, int kgh, int b, int bp) {
    return LAYER2 ? c3b_tile_major_offset((size_t)b, t * 40 + dir * 20 + kgh, 1320)
                  : c3b_tile_major_offset((size_t)t * bp + b, dir * 16 + kgh, 32);
}

__device__ __forceinline__ void unpack_half8(const uint4 &v, float *f) {
    const __half2 *hp = reinterpret_cast<const __half2 *>(&v);
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        const float2 t = __half22float2(hp[i]);
        f[2 * i] = t.x;
        f[2 * i + 1] = t.y;
    }
}

template <int NB, bool LAYER2, bool MUFU16, int WG>
__global__ void __launch_bounds__(2 * 128 * WG + 32, 1) lstm_tc_kernel(const LstmDev p) {
    constexpr int kGroupThreads = kWgThreads * WG;  // threads working on one sub-tile
    constexpr int kBlockThreads = 2 * kGroupThreads + 32;
    constexpr int kMmaWarp = 8 * WG;
    constexpr int NBH = NB / WG;                    // sites per epilogue thread
    static_assert(NBH % 8 == 0, "each warpgroup takes whole 8-site chunks");
    constexpr int H = LAYER2 ? 160 : 128;
    constexpr int KX = LAYER2 ? 0 : C3B_X1_COLS;
    constexpr int K = KX + H;                       // 176 (LSTM1) | 160 (LSTM2)
    constexpr int kBlkBytes = (K / 8) * 128 * 16;   // one 128-row weight block: [K/8][128][8] fp16
    static_assert(K % 16 == 0, "whole UMMA k-steps");
    constexpr int NBLK = LAYER2 ? 5 : 4;            // accumulator row blocks
    constexpr int NBLK_S = 4;                       // row blocks whose weights live in shared memory
    constexpr uint32_t LBO_B = (NB + 1) * 16;       // padded: conflict-free h stores
    constexpr uint32_t B_BYTES = (K / 8) * LBO_B;
    constexpr uint32_t ACC_COLS = 2 * NBLK * NB;    // two sub-tiles
    constexpr uint32_t WT_COLS = LAYER2 ? 80 : 0;   // LSTM2 tail block weights as a TMEM A operand (K=160 -> 80 columns)
    constexpr uint32_t NEED = ACC_COLS + WT_COLS;
    constexpr uint32_t TCOLS = NEED <= 32 ? 32 : NEED <= 64 ? 64 : NEED <= 128 ? 128 : NEED <= 256 ? 256 : 512;
    static_assert(NEED <= 512, "TMEM budget");

    extern __shared__ __align__(128) uint8_t smem[];
    __shared__ uint64_t w_bar, acc_bar[2], ready_bar[2];
    __shared__ uint32_t tmem_base_smem;
    uint8_t *w_smem = smem;
    uint8_t *b_smem0 = smem + NBLK_S * kBlkBytes;
    float *xch0 = reinterpret_cast<float *>(b_smem0 + 2 * B_BYTES);     // LAYER2 only: [2][NB][128]

    const int tid = threadIdx.x;
    const int warp = tid >> 5;
    const int lane = tid & 31;
    const int dir = blockIdx.y;
    const uint32_t w_addr = ptx::smem_u32(w_smem);
    const uint32_t b_addr0 = ptx::smem_u32(b_smem0);

    if (tid == 0) {
        ptx::mbar_init(&w_bar, 1);
        for (int s = 0; s < 2; ++s) {
            ptx::mbar_init(&acc_bar[s], 1);
            ptx::mbar_init(&ready_bar[s], 1);
        }
        ptx::fence_barrier_init();
    }
    if (warp == kMmaWarp) ptx::tmem_alloc<TCOLS>(&tmem_base_smem);
    for (uint32_t i = tid * 16; i < 2 * B_BYTES; i += kBlockThreads * 16)
        *reinterpret_cast<uint4 *>(b_smem0 + i) = make_uint4(0, 0, 0, 0);
    ptx::tc_fence_before();
    __syncthreads();
    ptx::tc_fence_after();
    const uint32_t tmem_base = tmem_base_smem;

    if (tid == 0) {
        ptx::mbar_arrive_expect_tx(&w_bar, NBLK_S * kBlkBytes);
        const char *src = reinterpret_cast<const char *>(p.w_img) + (size_t)dir * NBLK * kBlkBytes;
#pragma unroll
        for (int m = 0; m < NBLK_S; ++m) ptx::bulk_g2s(w_addr + m * kBlkBytes, src + (size_t)m * kBlkBytes, kBlkBytes, &w_bar);
    }

    const uint32_t idesc = ptx::umma_idesc_f16(128, NB);
    if (warp == kMmaWarp) {
        // ===================================================== MMA warp: alternate between the two sub-tiles.
        // ONE elected thread runs the whole 33-step loop, barrier waits included (tcgen05.mma issue does not run ahead of the
        // tensor pipe: a per-step elect / reconvergence / __syncwarp and 64-bit descriptor rebuilds between MMAs were pipe idle
        // time - measured 68 cycles per MMA against the 48-cycle floor of a 128 x NB x 16 MMA).  Descriptors: constant high
        // words, low words advanced by 32-bit adds on the start-address field (shared memory < 256 KB: no carry).
        ptx::mbar_wait(&w_bar, 0);
        if (ptx::elect_one()) {
            const uint64_t a_d0 = ptx::umma_desc_nosw(w_addr, 2048, 128), b_d0 = ptx::umma_desc_nosw(b_addr0, LBO_B, 128);
            const uint32_t a_lo0 = (uint32_t)a_d0, a_hi = (uint32_t)(a_d0 >> 32);
            const uint32_t b_lo0 = (uint32_t)b_d0, b_hi = (uint32_t)(b_d0 >> 32);
            constexpr uint32_t a_kstep = (2u * 2048u) >> 4, a_mstep = (uint32_t)kBlkBytes >> 4;
            constexpr uint32_t b_kstep = (2u * LBO_B) >> 4, b_sstep = B_BYTES >> 4;
            for (int step = 0; step < C3B_T; ++step) {
#pragma unroll
                for (int s = 0; s < 2; ++s) {
                    ptx::mbar_wait(&ready_bar[s], (uint32_t)step & 1u);
                    ptx::tc_fence_after();
                    const uint32_t d0 = tmem_base + (uint32_t)(s * NBLK * NB);
                    uint32_t b_lo = b_lo0 + (uint32_t)s * b_sstep, a_lo = a_lo0, wt_col = tmem_base + ACC_COLS;
                    // k loop rolled (a fully unrolled one makes ptxas park every descriptor in vector registers and pay R2UR /
                    // spill moves between MMAs); its body is four or five MMAs and three uniform adds
#pragma unroll 1
                    for (int ks = 0; ks < K / 16; ++ks) {
                        const uint64_t b_desc = ((uint64_t)b_hi << 32) | (uint64_t)b_lo;
                        const uint32_t acc = ks > 0 ? 1u : 0u;
#pragma unroll
                        for (int m = 0; m < NBLK_S; ++m)
                            ptx::umma_f16(d0 + m * NB, ((uint64_t)a_hi << 32) | (uint64_t)(a_lo + (uint32_t)m * a_mstep), b_desc, idesc, acc);
                        if (LAYER2) ptx::umma_f16_ts(d0 + 4 * NB, wt_col, b_desc, idesc, acc);
                        a_lo += a_kstep;
                        b_lo += b_kstep;
                        wt_col += 8;
                    }
                    ptx::umma_commit(&acc_bar[s]);
                }
            }
        }
        __syncwarp();
    }

    // ========================================================= epilogue warpgroup `sub` (0 or 1)
    if (warp != kMmaWarp) {
    const int sub = (warp >> 2) & 1;                // warps [0,4) sub 0, [4,8) sub 1, then (WG = 2) the second halves
    const int half = warp >> 3;                     // which NBH-site half of the sub-tile this warpgroup owns
    const int q = warp & 3;                         // TMEM lane quadrant
    const int wt = tid & 127;                       // thread index in the warpgroup = TMEM lane = hidden unit
    const int gt = wt + 128 * half;                 // thread index among the sub-tile's kGroupThreads
    const int j0h = half * (NBH / 8);               // first 8-site chunk of this warpgroup
    const int subtile = blockIdx.x * 2 + sub;       // index of this NB-site sub-tile in the padded batch
    const int b0 = subtile * NB;
    uint8_t *b_smem = b_smem0 + sub * B_BYTES;
    float *xch = xch0 + sub * NB * 128;
    const uint32_t lane_taddr = tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(sub * NBLK * NB);
    const int ntl = p.bp / NB;
    const uint32_t bar_id = 1 + sub;

    if (LAYER2 && sub == 0 && half == 0) {
        // tail-block weights (units 128..159) -> TMEM columns [ACC_COLS, ACC_COLS+80): thread = row, 16 halves per k-step
        const op_t *wt_img = p.w_img + ((size_t)dir * NBLK + 4) * (kBlkBytes / 2);
#pragma unroll 1
        for (int ks = 0; ks < K / 16; ++ks) {
            const uint4 v0 = *reinterpret_cast<const uint4 *>(wt_img + ((size_t)(2 * ks) * 128 + wt) * 8);
            const uint4 v1 = *reinterpret_cast<const uint4 *>(wt_img + ((size_t)(2 * ks + 1) * 128 + wt) * 8);
            uint32_t r[8] = {v0.x, v0.y, v0.z, v0.w, v1.x, v1.y, v1.z, v1.w};
            ptx::tmem_st8(tmem_base + ((uint32_t)(q * 32) << 16) + ACC_COLS + ks * 8, r);
        }
        ptx::tmem_st_wait();
    }

    float c[NBH];
#pragma unroll
    for (int i = 0; i < NBH; ++i) c[i] = 0.f;
    float c_tail[LAYER2 ? NBH / 4 : 1];
#pragma unroll
    for (int i = 0; i < (LAYER2 ? NBH / 4 : 1); ++i) c_tail[i] = 0.f;

    int t_prev = 0;
    for (int step = 0; step < C3B_T; ++step) {
        const int t = dir ? (C3B_T - 1 - step) : step;

        if constexpr (!LAYER2) {
            // stage x_0: xs[t][b0+n][0..47] -> operand k-groups 0..5.  Later steps find x_t already there: it was fetched into
            // registers while the previous step's MMAs ran and stored once they had finished reading the operand buffer (below) -
            // a global load on the step's critical path cost ~700 cycles of L2 latency per step.
            if (step == 0) {
                for (int idx = gt; idx < NB * (KX / 8); idx += kGroupThreads) {
                    const int n = idx / (KX / 8), kg = idx % (KX / 8);
                    const uint4 v = *reinterpret_cast<const uint4 *>(p.xs + ((size_t)t * p.bp + b0 + n) * KX + kg * 8);
                    *reinterpret_cast<uint4 *>(b_smem + kg * LBO_B + n * 16) = v;
                }
            }
        }
        ptx::fence_proxy_async_smem();
        ptx::tc_fence_before();
        // S1: every thread of the warpgroup has written its h_t / x_t and finished its TMEM reads.  The barrier (not just
        // per-thread mbarrier arrivals) matters: the copy-out below reads 16-byte chunks of h written by OTHER threads.
        ptx::named_bar_sync(bar_id, kGroupThreads);
        if (gt == 0) ptx::mbar_arrive(&ready_bar[sub]);
        const bool tr = p.trace != nullptr && tid == 0 && blockIdx.x == 0 && blockIdx.y == 0;
        if (tr) p.trace[step * 4 + 0] = clock64();
        if (tr) p.trace[step * 4 + 1] = clock64();

        // LSTM1: fetch x_{t+1} now (in flight while the MMAs run), store it after the accumulator barrier
        constexpr int XN = LAYER2 ? 1 : (NB * (KX / 8) + kGroupThreads - 1) / kGroupThreads;
        uint4 xnext[XN];
        if constexpr (!LAYER2) {
            if (step + 1 < C3B_T) {
                const int tn = dir ? t - 1 : t + 1;
#pragma unroll
                for (int i = 0; i < XN; ++i) {
                    const int idx = gt + i * kGroupThreads;
                    if (idx < NB * (KX / 8))
                        xnext[i] = *reinterpret_cast<const uint4 *>(p.xs + ((size_t)tn * p.bp + b0 + idx / (KX / 8)) * KX + (idx % (KX / 8)) * 8);
                }
            }
        }
        // while the MMAs run: ship h_{t_prev} (still in the operand buffer) to global memory
        if (step > 0) {
            for (int idx = gt; idx < NB * (H / 8); idx += kGroupThreads) {
                const int kgh = idx / NB, n = idx % NB;           // consecutive threads -> consecutive sites: 16 B x NB runs
                const uint4 v = *reinterpret_cast<const uint4 *>(b_smem + (KX / 8 + kgh) * LBO_B + n * 16);
                op_t *dst = p.hout + h_out_offset<LAYER2>(t_prev, dir, kgh, b0 + n, p.bp);
                *reinterpret_cast<uint4 *>(dst) = v;
            }
        }
        // LSTM2: prefetch this step's pre-gates (fp16, NB contiguous values per (block,row))
        uint4 pgv[LAYER2 ? 5 : 1][LAYER2 ? NBH / 8 : 1];
        if (LAYER2) {
            const __half *pgp = p.pg + ((((size_t)(dir * C3B_T + t) * ntl + subtile) * 5) * 128 + wt) * NB;
#pragma unroll
            for (int m = 0; m < 5; ++m)
#pragma unroll
                for (int j = 0; j < NBH / 8; ++j)
                    pgv[m][j] = *reinterpret_cast<const uint4 *>(pgp + (size_t)m * 128 * NB + (j0h + j) * 8);
            // the pre-gate tensor (86 MB per 1024 sites) streams from HBM: pull the NEXT step's lines into L2 now so the
            // loads above find them there one step later
            if (step + 1 < C3B_T) {
                const int tn = dir ? t - 1 : t + 1;
                const __half *pgn = p.pg + ((((size_t)(dir * C3B_T + tn) * ntl + subtile) * 5) * 128 + wt) * NB;
#pragma unroll
                for (int m = 0; m < 5; ++m)
#pragma unroll
                    for (int j = 0; j < (NB * 2 + 127) / 128; ++j)
                        asm volatile("prefetch.global.L2 [%0];" ::"l"(pgn + (size_t)m * 128 * NB + j * 64));
            }
        }

        ptx::mbar_wait(&acc_bar[sub], (uint32_t)step & 1u);
        ptx::tc_fence_after();
        if (tr) p.trace[step * 4 + 2] = clock64();
        ptx::named_bar_sync(bar_id, kGroupThreads);                         // S2: the sub-tile's threads are done reading h_{t_prev}
        if constexpr (!LAYER2) {
            if (step + 1 < C3B_T) {       // this step's MMAs have completed: the x columns of the operand buffer may take x_{t+1}
#pragma unroll
                for (int i = 0; i < XN; ++i) {
                    const int idx = gt + i * kGroupThreads;
                    if (idx < NB * (KX / 8)) *reinterpret_cast<uint4 *>(b_smem + (idx % (KX / 8)) * LBO_B + (idx / (KX / 8)) * 16) = xnext[i];
                }
            }
        }

        if (LAYER2) {
            // tail block (units 128..159): warp q holds gate q; activate and publish to the exchange buffer
#pragma unroll
            for (int j = 0; j < NBH / 8; ++j) {
                float v[8], pgf[8];
                ptx::tmem_ld8(lane_taddr + 4 * NB + (j0h + j) * 8, v);
                ptx::tmem_ld_wait();
                unpack_half8(pgv[4][j], pgf);
#pragma unroll
                for (int i = 0; i < 8; ++i) {
                    const float x = v[i] + pgf[i];
                    const float a = (q == 2) ? ptx::tanh_approx(x) : ptx::sigmoid_prehalved(x);
                    xch[((j0h + j) * 8 + i) * 128 + wt] = a;
                }
            }
            ptx::named_bar_sync(bar_id, kGroupThreads);
        }

        // main blocks: thread = hidden unit `wt`, 8 sites at a time
#pragma unroll
        for (int j = 0; j < NBH / 8; ++j) {
            float gi[8], gf[8], gg[8], go[8], h[8];
            ptx::tmem_ld8(lane_taddr + 0 * NB + (j0h + j) * 8, gi);
            ptx::tmem_ld8(lane_taddr + 1 * NB + (j0h + j) * 8, gf);
            ptx::tmem_ld8(lane_taddr + 2 * NB + (j0h + j) * 8, gg);
            ptx::tmem_ld8(lane_taddr + 3 * NB + (j0h + j) * 8, go);
            ptx::tmem_ld_wait();
            if (LAYER2) {
                float pf[8];
                unpack_half8(pgv[0][j], pf);
#pragma unroll
                for (int i = 0; i < 8; ++i) gi[i] += pf[i];
                unpack_half8(pgv[1][j], pf);
#pragma unroll
                for (int i = 0; i < 8; ++i) gf[i] += pf[i];
                unpack_half8(pgv[2][j], pf);
#pragma unroll
                for (int i = 0; i < 8; ++i) gg[i] += pf[i];
                unpack_half8(pgv[3][j], pf);
#pragma unroll
                for (int i = 0; i < 8; ++i) go[i] += pf[i];
            }
            // h[n][unit] -> operand buffer (fp16), element (n, k = KX + wt)
            const uint32_t kcol = KX + wt;
            uint8_t *dst = b_smem + (kcol >> 3) * LBO_B + (kcol & 7) * 2;
            if (MUFU16) {
                uint32_t hp[4];
                lstm_cell8_h2(gi, gf, gg, go, &c[j * 8], hp);
#pragma unroll
                for (int i = 0; i < 4; ++i) {
                    *reinterpret_cast<uint16_t *>(dst + ((j0h + j) * 8 + 2 * i) * 16) = (uint16_t)(hp[i] & 0xffffu);
                    *reinterpret_cast<uint16_t *>(dst + ((j0h + j) * 8 + 2 * i + 1) * 16) = (uint16_t)(hp[i] >> 16);
                }
            } else {
                lstm_cell8(gi, gf, gg, go, &c[j * 8], h);
#pragma unroll
                for (int i = 0; i < 8; ++i) *reinterpret_cast<op_t *>(dst + ((j0h + j) * 8 + i) * 16) = f2op(h[i]);
            }
        }

        if (LAYER2) {
            // tail cells: unit 128 + lane, sites n = q + 4*k of this warpgroup's half (their activations were published by
            // this same warpgroup, and the barrier above covers both)
#pragma unroll
            for (int k = 0; k < NBH / 4; ++k) {
                const int n = half * NBH + q + 4 * k;
                const float iv = xch[n * 128 + lane];
                const float fv = xch[n * 128 + 32 + lane];
                const float gv = xch[n * 128 + 64 + lane];
                const float ov = xch[n * 128 + 96 + lane];
                c_tail[k] = fmaf(fv, c_tail[k], iv * gv);
                const float hv = ov * ptx::tanh_approx(c_tail[k]);
                const uint32_t kcol = 128 + lane;
                *reinterpret_cast<op_t *>(b_smem + (kcol >> 3) * LBO_B + n * 16 + (kcol & 7) * 2) = f2op(hv);
            }
        }
        t_prev = t;
        if (tr) p.trace[step * 4 + 3] = clock64();
    }

    // last h
    ptx::named_bar_sync(bar_id, kGroupThreads);
    for (int idx = gt; idx < NB * (H / 8); idx += kGroupThreads) {
        const int kgh = idx / NB, n = idx % NB;
        const uint4 v = *reinterpret_cast<const uint4 *>(b_smem + (KX / 8 + kgh) * LBO_B + n * 16);
        op_t *dst = p.hout + h_out_offset<LAYER2>(t_prev, dir, kgh, b0 + n, p.bp);
        *reinterpret_cast<uint4 *>(dst) = v;
    }
    }   // epilogue warps

    // teardown: ONE barrier for every role (the MMA warp and the epilogue warps meet at the same __syncthreads)
    ptx::tc_fence_before();
    __syncthreads();
    if (warp == kMmaWarp) {
        ptx::tc_fence_after();
        ptx::tmem_dealloc<TCOLS>(tmem_base);
    }
}

template <typename T>
__device__ __forceinline__ float ingest_to_float(T v) { return (float)v; }

// Dense [batch][33][channels] tensor, or (starts != nullptr) 33-row windows of the per-column count matrix [n_cols][channels]
// (libclair3's plp_data.matrix; preprocess/CreateTensorPileupFromCffi.py:362-394 slices the same windows on the host, zero
// rows where a window overhangs the matrix) -> xs[t][bp][48] fp16 with columns [hi(x) | 1 | lo(x) | 0..]: hi = fp16(x)
// (saturating at +-65504), lo = fp16(x - hi), so hi + lo == x exactly for |x| <= 67 552; column `channels` = constant 1
// (LSTM1's bias column).
// tiled = 0: xs[t][bp][48] (lstm_tc_kernel); tiled = 1: xs2[t][bp/128][6 k-groups][128 sites][8] (the CTA-pair kernel bulk-copies one
// 12 KB run per step and 128-site tile)
template <typename T>
__global__ void ingest_pileup_tc_kernel(const T *__restrict__ x, const int64_t *__restrict__ starts, int64_t n_cols,
                                        op_t *__restrict__ xs, int64_t batch, int bp, int channels, int tiled) {
    // one thread per (t, site): six 16-byte stores
    const int64_t total = (int64_t)C3B_T * bp;
    for (int64_t tb = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; tb < total; tb += (int64_t)gridDim.x * blockDim.x) {
        const int b = (int)(tb % bp);
        const int t = (int)(tb / bp);
        bool have = b < batch;
        const T *src = x;
        if (have) {
            if (starts) {
                const int64_t row = starts[b] + t;
                have = row >= 0 && row < n_cols;
                src = x + row * channels;
            } else {
                src = x + ((int64_t)b * C3B_T + t) * channels;
            }
        }
        __align__(16) op_t v[C3B_X1_COLS];
        if (channels == 18) {
            // the reference's pileup shape (shared/param_p.py:32-36): every index is a compile-time constant, one load per count
            float xv[18];
#pragma unroll
            for (int c = 0; c < 18; ++c) xv[c] = have ? ingest_to_float(src[c]) : 0.f;
#pragma unroll
            for (int c = 0; c < 18; ++c) {
                const op_t hi = f2op_sat(xv[c]);
                v[c] = hi;
                v[19 + c] = f2op_sat(xv[c] - op2f(hi));
            }
            v[18] = f2op(1.f);
#pragma unroll
            for (int k = 37; k < C3B_X1_COLS; ++k) v[k] = f2op(0.f);
        } else {
#pragma unroll
            for (int k = 0; k < C3B_X1_COLS; ++k) {          // static indices: v stays in registers
                float f = (k == channels) ? 1.f : 0.f;
                if (have && k != channels && k <= 2 * channels) {
                    const float xvv = ingest_to_float(src[k < channels ? k : k - channels - 1]);
                    const op_t hi = f2op_sat(xvv);
                    f = k < channels ? op2f(hi) : xvv - op2f(hi);
                }
                v[k] = f2op_sat(f);
            }
        }
        if (tiled) {
            op_t *dst = xs + (((size_t)t * (bp >> 7) + (b >> 7)) * (C3B_X1_COLS / 8) * 128 + (b & 127)) * 8;
#pragma unroll
            for (int k = 0; k < C3B_X1_COLS / 8; ++k) *reinterpret_cast<uint4 *>(dst + (size_t)k * 128 * 8) = reinterpret_cast<const uint4 *>(v)[k];
        } else {
            uint4 *dst = reinterpret_cast<uint4 *>(xs + tb * C3B_X1_COLS);
#pragma unroll
            for (int k = 0; k < C3B_X1_COLS / 8; ++k) dst[k] = reinterpret_cast<const uint4 *>(v)[k];
        }
    }
}

template <int NB, bool LAYER2, bool MUFU16, int WG>
int launch_lstm_impl(const LstmDev &p, cudaStream_t s) {
    constexpr int K = (LAYER2 ? 0 : C3B_X1_COLS) + (LAYER2 ? 160 : 128);
    const size_t smem = (size_t)4 * (K / 8) * 2048 + 2 * (K / 8) * (NB + 1) * 16 + (LAYER2 ? (size_t)2 * NB * 128 * 4 : 0);
    auto kern = lstm_tc_kernel<NB, LAYER2, MUFU16, WG>;
    C3B_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    dim3 grid(p.bp / (2 * NB), 2);
    c3b_note_grid((long long)grid.x * grid.y);
    kern<<<grid, 2 * 128 * WG + 32, smem, s>>>(p);
    C3B_CUDA(cudaGetLastError());
    return 0;
}

// wg = epilogue warpgroups per sub-tile (2 by default; 1 = the original layout, also used by the f16x2 MUFU variant)
template <int NB, bool LAYER2>
int launch_lstm(const LstmDev &p, bool mufu16, int wg, cudaStream_t s) {
    if (mufu16) return wg == 1 ? launch_lstm_impl<NB, LAYER2, true, 1>(p, s) : launch_lstm_impl<NB, LAYER2, true, 2>(p, s);
    return wg == 1 ? launch_lstm_impl<NB, LAYER2, false, 1>(p, s) : launch_lstm_impl<NB, LAYER2, false, 2>(p, s);
}

}  // namespace

int c3b_launch_ingest_pileup_tc(const void *x, int dtype, int channels, const int64_t *starts, int64_t n_cols, op_t *xs, int64_t batch,
                                int bp, int tiled, cudaStream_t s) {
    const int64_t total = (int64_t)C3B_T * bp;
    const int blocks = (int)((total + 127) / 128 < 2048 ? (total + 127) / 128 : 2048);
    c3b_note_grid(blocks);
    switch (dtype) {
        case C3B_DT_I8: ingest_pileup_tc_kernel<int8_t><<<blocks, 128, 0, s>>>((const int8_t *)x, starts, n_cols, xs, batch, bp, channels, tiled); break;
        case C3B_DT_I32: ingest_pileup_tc_kernel<int32_t><<<blocks, 128, 0, s>>>((const int32_t *)x, starts, n_cols, xs, batch, bp, channels, tiled); break;
        case C3B_DT_I64: ingest_pileup_tc_kernel<int64_t><<<blocks, 128, 0, s>>>((const int64_t *)x, starts, n_cols, xs, batch, bp, channels, tiled); break;
        case C3B_DT_F32: ingest_pileup_tc_kernel<float><<<blocks, 128, 0, s>>>((const float *)x, starts, n_cols, xs, batch, bp, channels, tiled); break;
        default: c3b_set_error("unsupported input dtype %d", dtype); return 1;
    }
    C3B_CUDA(cudaGetLastError());
    return 0;
}

// `tile` = sites per sub-tile (a CTA covers two sub-tiles).
int c3b_launch_lstm1_tc(const c3b_model *m, const TcPileupBuffers &b, int64_t batch, int tile, cudaStream_t s) {
    LstmDev p = {};
    p.w_img = m->lstm_tc[0][0].w_img;     // both directions are contiguous
    p.xs = b.xs;
    p.hout = b.h1;
    p.trace = (m->lstm_trace && m->trace_conv == 1) ? m->lstm_trace : nullptr;
    p.bp = b.bp;
    const_cast<c3b_model *>(m)->launches++;
    switch (tile) {
        case 16: return launch_lstm<16, false>(p, m->lstm_mufu16 != 0, m->lstm_wg, s);
        case 32: return launch_lstm<32, false>(p, m->lstm_mufu16 != 0, m->lstm_wg, s);
        case 64: return launch_lstm<64, false>(p, m->lstm_mufu16 != 0, m->lstm_wg, s);
    }
    c3b_set_error("lstm1: unsupported tile %d", tile);
    return 1;
}

int c3b_launch_lstm2_tc(const c3b_model *m, const TcPileupBuffers &b, int64_t batch, int tile, cudaStream_t s) {
    LstmDev p = {};
    p.w_img = m->lstm_tc[1][0].w_img;
    p.pg = b.pg;
    p.hout = b.h2;
    p.trace = (m->lstm_trace && m->trace_conv == 1) ? m->lstm_trace + C3B_T * 4 : nullptr;
    p.bp = b.bp;
    const_cast<c3b_model *>(m)->launches++;
    switch (tile) {
        case 16: return launch_lstm<16, true>(p, m->lstm_mufu16 != 0, m->lstm_wg, s);
        case 32: return launch_lstm<32, true>(p, m->lstm_mufu16 != 0, m->lstm_wg, s);
    }
    c3b_set_error("lstm2: unsupported tile %d", tile);
    return 1;
}
