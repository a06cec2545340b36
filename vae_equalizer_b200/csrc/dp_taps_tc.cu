// DP VAE step: BOTH tap-gradient correlations (dW and dh) on the 5th-generation tensor cores (tcgen05, accumulators in TMEM).
//
// OUTSIDE north_star's STATED DESIGN ("tensor cores are not used because the path is not a dense contraction"), accepted against the
// 1e-4 gradient tolerance and adopted on measurement (profiles/r02_tc_taps.txt); the default since r02, vaeq_dp_tc_taps(0) selects the
// CUDA-core kernels of dp_fast.cu.
//
// The correlations ARE a dense contraction once the symbol axis is cut into blocks of 16: for a per-symbol operand a(.) and a
// window operand w(.),
//     D[(row, i), (comp, n)] = sum_k a_row[16 k + i] * w_comp[16 k - 8 + n]         i < 16 (x 2 sample phases), n < 32
// is a plain GEMM over the block index k whose operands are the SoA rows as they lie in HBM, and the lag-b correlation is the sum
// of one diagonal (n = i + 8 + b) of D.  D is 128 x 128 per correlation and stays in TMEM for the WHOLE kernel (256 of the 512
// columns); the diagonals are summed once per CTA at the end.  40 % of the MMA flops are useful -- they are free: the CUDA-core
// kernels this replaces are bound by the FP32 pipe / register-file bandwidth (profiles/r02_fused_backward.txt), this one by HBM.
//   M side (128 = 4 components x 32):  dW: rx rows, 32 samples = 16 symbols x 2 phases per k;   dh: residual rows, phases interleaved
//   N side (128 = 4 components x 32):  dW: dL/dout window;                                      dh: E_q window
// fp32 accuracy with tf32 tensor cores: kind::tf32 TRUNCATES fp32 operands (measured, tools/tc_corr_bench.cu), so x = hi + lo with
// hi = trunc(x) exactly, and D += a b (hardware takes the hi parts) + a lo(b) + lo(a) b; the dropped lo lo term is 2^-22 relative.
// MN-major tf32 operands have ONE legal shared-memory layout (SWIZZLE_128B_BASE32B: 128-byte rows, 4 k-rows per atom, 32-byte chunks
// XORed with the k-row index); 16 converter warps build it (and the lo parts) straight from global memory: every thread owns one
// 16-byte chunk per array and tile, loaded one tile ahead into registers.  (Staging the rows with cp.async.bulk first was measured
// and dropped: the 20 one-to-two-kilobyte copies of a tile cost ~110 cycles EACH in the TMA unit, 127 us for the loads alone.)
// Reference: the dW / dh sums of loss.backward() through loss_function_shaping sf:115-129 and twoXtwoFIR.forward sf:500-518.
#include "dp_kernels.cuh"
#include "tma.cuh"   // mbarrier helpers

namespace vaeq {

constexpr int TC_NCV = 512;                                 // converter threads (16 warps)
constexpr int TC_NT = TC_NCV + 32;                          // + the MMA-issuing warp; one CTA per SM
constexpr int TC_KB = 16;                                   // symbols per k-row
constexpr int TC_NK = 16;                                   // k-rows per tile (two K = 8 MMA steps)
constexpr int TC_TS = TC_KB * TC_NK;                        // 256 symbols per tile
constexpr int TC_SH = 8;                                    // the window starts 8 symbols before the block (>= MH/2, 16-byte aligned)
constexpr int TC_OPB = 4 * TC_NK * 128;                     // bytes of one operand array: 4 components x 16 k-rows x 128 B
constexpr int TC_OS = 3;                                    // operand stages (conversion runs up to two tiles ahead of the MMAs)
constexpr int TC_DLD = 129;                                 // padded row length of the epilogue's copy of D

__device__ __forceinline__ uint64_t umma_desc_mn_tf32(uint32_t saddr, uint32_t lbo, uint32_t sbo) {
    // shared-memory matrix descriptor: start >> 4 | LBO >> 4 << 16 (stride between 32-element MN groups) | SBO >> 4 << 32 (stride
    // between groups of 4 k-rows) | version 1 << 46 | layout SWIZZLE_128B_BASE32B (1) << 61
    return (uint64_t)((saddr >> 4) & 0x3fff) | ((uint64_t)((lbo >> 4) & 0x3fff) << 16) | ((uint64_t)((sbo >> 4) & 0x3fff) << 32) | (1ull << 46) | (1ull << 61);
}
// instruction descriptor: D = f32 (1 << 4), A = B = tf32 (2 << 7, 2 << 10), both MN-major (bits 15, 16), N >> 3 << 17, M >> 4 << 24
constexpr uint32_t TC_IDESC = (1u << 4) | (2u << 7) | (2u << 10) | (1u << 15) | (1u << 16) | ((128u >> 3) << 17) | ((128u >> 4) << 24);
__device__ __forceinline__ void umma_tf32(uint32_t tmem_d, uint64_t da, uint64_t db, uint32_t acc) {
    asm volatile(
        "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n\t}\n" ::"r"(tmem_d),
        "l"(da), "l"(db), "r"(TC_IDESC), "r"(acc)
        : "memory");
}
__device__ __forceinline__ void umma_commit(uint64_t *bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ float tf32_lo(float x) {         // x - trunc_tf32(x), rounded to tf32
    const float r = x - __uint_as_float(__float_as_uint(x) & 0xffffe000u);
    uint32_t o;
    asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(o) : "f"(r));
    return __uint_as_float(o);
}
__device__ __forceinline__ void split_store(unsigned char *hi, unsigned char *lo, uint32_t off, float4 v) {
    *reinterpret_cast<float4 *>(hi + off) = v;
    *reinterpret_cast<float4 *>(lo + off) = make_float4(tf32_lo(v.x), tf32_lo(v.y), tf32_lo(v.z), tf32_lo(v.w));
}

template <int MH>
__global__ void __launch_bounds__(TC_NT, 1) k_dp_taps_tc(DpK p, int t_lo) {
    constexpr int M = 2 * MH + 1, HF = MH / 2;
    static_assert(MH % 2 == 0 && HF <= TC_SH, "tensor-core tap gradients need M_est = 1 (mod 4), M_est <= 33");
    extern __shared__ __align__(1024) unsigned char smem[];
    uint64_t *bars = reinterpret_cast<uint64_t *>(smem);    // conv_done[TC_OS], mma_done[TC_OS], fin
    uint32_t *tmem_slot = reinterpret_cast<uint32_t *>(smem + 128);
    unsigned char *ops = smem + 1024;                        // [TC_OS stages][8 arrays][TC_OPB]: rx hi/lo, e hi/lo, gy hi/lo, E_q hi/lo
    uint64_t *conv_done = bars, *mma_done = bars + TC_OS, *fin = bars + 2 * TC_OS;
    const int tid = threadIdx.x, wid = tid >> 5, lane = tid & 31;
    const int nt = p.ntiles;

    if (tid == 0) {
        for (int s = 0; s < TC_OS; ++s) {
            mbar_init(conv_done + s, TC_NCV);
            mbar_init(mma_done + s, 1);
        }
        mbar_init(fin, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (wid == 0) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], 256;" ::"r"(smem_u32(tmem_slot)) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    const uint32_t tmem = *tmem_slot;

    if (wid == TC_NCV / 32) {
        // ================= MMA warp (one lane issues): D += a b + a lo(b) + lo(a) b for both correlations, two K = 8 steps per tile =================
        int it = 0;
#pragma unroll 1
        for (int tile = blockIdx.x; tile < nt; tile += gridDim.x, ++it) {
            const int s = it % TC_OS;
            mbar_wait(conv_done + s, (it / TC_OS) & 1);
            if (lane == 0) {
                asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
                const uint32_t ob = smem_u32(ops + s * 8 * TC_OPB);
#pragma unroll
                for (int ks = 0; ks < TC_NK / 8; ++ks) {
#pragma unroll
                    for (int corr = 0; corr < 2; ++corr) {
                        const uint32_t a_hi = ob + (2 * corr) * TC_OPB + ks * 1024, b_hi = ob + (4 + 2 * corr) * TC_OPB + ks * 1024;
                        const uint64_t dah = umma_desc_mn_tf32(a_hi, TC_NK * 128, 512), dal = umma_desc_mn_tf32(a_hi + TC_OPB, TC_NK * 128, 512);
                        const uint64_t dbh = umma_desc_mn_tf32(b_hi, TC_NK * 128, 512), dbl = umma_desc_mn_tf32(b_hi + TC_OPB, TC_NK * 128, 512);
                        const uint32_t d = tmem + 128 * corr;
                        umma_tf32(d, dah, dbh, (it | ks) != 0);
                        umma_tf32(d, dah, dbl, 1);
                        umma_tf32(d, dal, dbh, 1);
                    }
                }
                umma_commit(mma_done + s);
            }
            __syncwarp();
        }
        if (lane == 0) umma_commit(fin);                     // arrives when every MMA issued above has completed
    } else {
        // ================= converters: global SoA rows -> swizzled MN-major operand arrays (+ lo parts) =================
        // thread = (component, k-row, 16-byte chunk q): rx samples 32 k + 4 q .. + 3 of k-row k; residual symbols 16 k + 2 q, + 1 of both
        // phases (interleaved like rx); window row k = positions 16 k - 8 + [0, 32) of the dL/dout / E_q rows.  A chunk lies entirely
        // inside or outside a row's valid range (all limits are multiples of 4); outside it is ZERO, never read: a NaN in
        // never-written scratch would poison D even against a zero.
        const int comp = tid >> 7, rem = tid & 127, k = rem >> 3, q = rem & 7;
        const uint32_t off = comp * (TC_NK * 128) + k * 128 + ((q * 16) ^ ((k & 3) << 5));
        const float *rx_row = p.rx + (int64_t)comp * p.ld_rx, *e0_row = p.erows + (int64_t)comp * p.B, *e1_row = p.erows + (int64_t)(4 + comp) * p.B;
        const float *gy_row = p.gyrows + (int64_t)comp * p.B, *eq_row = p.m1rows + (int64_t)comp * p.B;
        struct Chunk {
            float4 x, g, q;
            float2 ea, eb;
        };
        auto fetch = [&](int tile, Chunk &c) {
            const int64_t t0 = (int64_t)t_lo + (int64_t)tile * TC_TS;
            const int64_t ix = 2 * t0 + 32 * k + 4 * q, ie = t0 + 16 * k + 2 * q, iw = t0 - TC_SH + 16 * k + 4 * q;
            const float4 z4 = make_float4(0.f, 0.f, 0.f, 0.f);
            c.x = (ix >= 0 && ix < p.L) ? __ldg(reinterpret_cast<const float4 *>(rx_row + ix)) : z4;
            const bool ine = ie >= p.sym_lo && ie < p.sym_hi;
            c.ea = ine ? __ldg(reinterpret_cast<const float2 *>(e0_row + ie)) : make_float2(0.f, 0.f);
            c.eb = ine ? __ldg(reinterpret_cast<const float2 *>(e1_row + ie)) : make_float2(0.f, 0.f);
            c.g = (iw >= p.sym_lo && iw < p.sym_hi) ? __ldg(reinterpret_cast<const float4 *>(gy_row + iw)) : z4;
            c.q = (iw >= p.clo && iw < p.chi) ? __ldg(reinterpret_cast<const float4 *>(eq_row + iw)) : z4;
        };
        // the chunks of the NEXT tile are loaded into a second register set before this tile's stores and fence.  (Measured: two or three
        // tiles ahead raise the load-only rate from 4.0 to 4.3 TB/s but lower the kernel's: 117 -> 126-132 us, profiles/r02_tc_taps.txt.)
        Chunk cur, nxt;
        if ((int)blockIdx.x < nt) fetch(blockIdx.x, nxt);
        int it = 0;
#pragma unroll 1
        for (int tile = blockIdx.x; tile < nt; tile += gridDim.x, ++it) {
            const int s = it % TC_OS;
            unsigned char *op = ops + s * 8 * TC_OPB;
            cur = nxt;
            if (tile + (int)gridDim.x < nt) fetch(tile + gridDim.x, nxt);
            mbar_wait(mma_done + s, ((it / TC_OS) & 1) ^ 1);                 // the MMAs of tile it - TC_OS have read this stage's operand arrays
            split_store(op, op + TC_OPB, off, cur.x);
            split_store(op + 2 * TC_OPB, op + 3 * TC_OPB, off, make_float4(cur.ea.x, cur.eb.x, cur.ea.y, cur.eb.y));
            split_store(op + 4 * TC_OPB, op + 5 * TC_OPB, off, cur.g);
            split_store(op + 6 * TC_OPB, op + 7 * TC_OPB, off, cur.q);
            asm volatile("fence.proxy.async.shared::cta;" ::: "memory");     // generic-proxy stores -> visible to the tensor core's reads
            mbar_arrive(conv_done + s);
        }
    }
    mbar_wait(fin, 0);
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");

    // ---- epilogue (once per CTA): D -> shared memory, diagonal sums, complex combinations, this CTA's gradient partial ----
    float *Dsm = reinterpret_cast<float *>(smem + 1024);     // [2][128][TC_DLD]: the operand / raw stages are dead now
    float *Rsm = Dsm + 2 * 128 * TC_DLD;                     // [2][4][4][M]
    if (wid < 8) {
        const int q = wid & 3, corr = wid >> 2;              // warps w and w + 4 own the same 32 TMEM lanes: one correlation each
#pragma unroll 1
        for (int c0 = 0; c0 < 128; c0 += 32) {
            uint32_t v[32];
            const uint32_t taddr = tmem + ((uint32_t)(32 * q) << 16) + 128 * corr + c0;
            asm volatile(
                "tcgen05.ld.sync.aligned.32x32b.x32.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,%16,%17,%18,%19,%20,%21,%22,%23,%24,%25,%26,%27,%28,%29,%30,%31}, [%32];"
                : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), "=r"(v[8]), "=r"(v[9]), "=r"(v[10]),
                  "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15]), "=r"(v[16]), "=r"(v[17]), "=r"(v[18]), "=r"(v[19]), "=r"(v[20]),
                  "=r"(v[21]), "=r"(v[22]), "=r"(v[23]), "=r"(v[24]), "=r"(v[25]), "=r"(v[26]), "=r"(v[27]), "=r"(v[28]), "=r"(v[29]), "=r"(v[30]), "=r"(v[31])
                : "r"(taddr));
            asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
            float *row = Dsm + (corr * 128 + 32 * q + lane) * TC_DLD + c0;
#pragma unroll
            for (int j = 0; j < 32; ++j) row[j] = __uint_as_float(v[j]);
        }
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    if (wid == 0) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, 256;" ::"r"(tmem) : "memory");
    // R[corr][cM][cW][t] = sum_j D[32 cM + 2 j + ph][32 cW + j + 8 + HF - a],  tap index t = 2 a + ph
    for (int idx = tid; idx < 2 * 16 * M; idx += TC_NT) {
        const int t = idx % M, cw = (idx / M) & 3, cm = (idx / (4 * M)) & 3, corr = idx / (16 * M);
        const int ph = t & 1, a = t >> 1;
        const float *d = Dsm + (corr * 128 + 32 * cm + ph) * TC_DLD + 32 * cw + TC_SH + HF - a;
        float sum = 0.f;
#pragma unroll
        for (int j = 0; j < TC_KB; ++j) sum += d[2 * j * TC_DLD + j];
        Rsm[idx] = sum;
    }
    __syncthreads();
    float *dst = p.gpart + (int64_t)blockIdx.x * 16 * M;
    for (int idx = tid; idx < 16 * M; idx += TC_NT) {
        // gW entries (o, [Re<-i | Im<-i], t): components cM = 2 i + c (rx row), cW = 2 o + c (dL/dout row)
        //     Re = sum gyI xI + gyQ xQ,   Im = sum gyQ xI - gyI xQ
        // gh entries (chi, nu, c, t): cM = 2 chi + c (residual), cW = 2 nu + c (E_q)
        //     Re = sum eI qI + eQ qQ,     Im = sum eQ qI - eI qQ          (times 2 kappa_chi)
        const int t = idx % M;
        if (idx < 8 * M) {
            const int oc = idx / M, o = oc >> 2, cidx = (oc >> 1) & 1, i = oc & 1;
            const float *R = Rsm;                            // [cM][cW][t]
            const float v = cidx == 0 ? R[((2 * i) * 4 + 2 * o) * M + t] + R[((2 * i + 1) * 4 + 2 * o + 1) * M + t]
                                      : R[((2 * i) * 4 + 2 * o + 1) * M + t] - R[((2 * i + 1) * 4 + 2 * o) * M + t];
            dst[idx] = v;
        } else {
            const int r = idx - 8 * M, oc = r / M, chi = oc >> 2, nu = (oc >> 1) & 1, cidx = oc & 1;
            const float *R = Rsm + 16 * M;
            const float v = cidx == 0 ? R[((2 * chi) * 4 + 2 * nu) * M + t] + R[((2 * chi + 1) * 4 + 2 * nu + 1) * M + t]
                                      : R[((2 * chi + 1) * 4 + 2 * nu) * M + t] - R[((2 * chi) * 4 + 2 * nu + 1) * M + t];
            dst[idx] = 2.f * p.scal[DP_KAPPA_OFF + chi] * v;
        }
    }
}

template <int MH>
static int taps_tc_launch_t(DpK p, cudaStream_t st, int *nparts) {
    static SmemAttrCache set;
    const size_t sm = 1024 + (size_t)TC_OS * 8 * TC_OPB + 1024;
    static_assert(1024 + TC_OS * 8 * TC_OPB >= 1024 + (2 * 128 * TC_DLD + 2 * 16 * (2 * MH + 1)) * 4, "epilogue scratch");
    if (int rc = ensure_dyn_smem(k_dp_taps_tc<MH>, sm, set)) return rc;
    const int t_lo = max(0, p.sym_lo - 16), t_hi = min(p.B, p.sym_hi + 16);
    p.ntiles = (t_hi - t_lo + TC_TS - 1) / TC_TS;
    const int grid = min(sm_count(), p.ntiles);
    ktime_begin(VAEQ_K_DP_BWD2, st);
    k_dp_taps_tc<MH><<<grid, TC_NT, sm, st>>>(p, t_lo);
    ktime_end(VAEQ_K_DP_BWD2, st);
    VAEQ_LAUNCH_CHECK("k_dp_taps_tc");
    *nparts = grid;
    return VAEQ_OK;
}

// both tap-gradient correlations in one launch (after k_dp_bwd1_fast wrote the dL/dout rows); returns 0 if M_est does not qualify
int dp_taps_tc_launch(const DpK &p, cudaStream_t st, int *nparts, int *rc) {
    switch (p.mh) {
        case 12: *rc = taps_tc_launch_t<12>(p, st, nparts); return 1;
        case 6: *rc = taps_tc_launch_t<6>(p, st, nparts); return 1;
        case 4: *rc = taps_tc_launch_t<4>(p, st, nparts); return 1;
        case 2: *rc = taps_tc_launch_t<2>(p, st, nparts); return 1;
        default: return 0;
    }
}

}  // namespace vaeq
