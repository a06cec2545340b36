// DP VAE step, forward kernel with BOTH sliding-window contractions (the 2x2 butterfly FIR and the channel convolution D = h * E_q)
// on the 5th-generation tensor cores (tcgen05, accumulators in TMEM); the point-wise stage (soft demapper, moments, entropy, backward
// coefficients) is the one of dp_fast.cu, on the CUDA cores.  Same inputs, outputs and scratch rows as k_dp_fwd_fast.
//
// Outside north_star's stated design ("tensor cores are not used because the path is not a dense contraction"): the contraction IS
// dense once four consecutive symbols form one GEMM row.  With the window as a HANKEL operand -- overlapping rows of one flat
// shared-memory array, read through a K-major swizzled descriptor (validated in tools/tc_hankel_bench.cu: the hardware swizzles by
// ABSOLUTE shared-memory address, so a descriptor may start on any row and K may run on into the following rows) --
//     FIR:   Y[m][(i, o)] = sum_{c, j} X_c[8 m + j] * T[(c, j)][(i, o)],   T = W_real[o][c][j - 2 i - SH]     (m = block of 4 symbols,
//            X_c = rx row c exactly as it lies in HBM: 8 samples = 32 bytes per row -> SWIZZLE_32B, K = 4 rows x 32 samples)
//     D:     D[m][(ph, i, o)] = sum_{j, c} Q[4 m + j][c] * H[(j, c)][(ph, i, o)]                              (Q = E_q as {pI,pQ,pI,pQ}
//            per symbol: 4 symbols = 64 bytes per row -> SWIZZLE_64B, K = 16 positions x 4)
// no im2col matrix exists anywhere: rx lands by cp.async in the layout the tensor core reads.  TMEM lane m = 4 consecutive symbols =
// the thread that owns them in the point-wise stage, so tcgen05.ld hands every thread exactly its own y / D values.
// fp32 accuracy from tf32 tensor cores: kind::tf32 truncates its operands, so x = hi + lo with hi = the raw fp32 word and
// lo = tf32(x - trunc(x)); the tap tables carry [hi | lo] side by side in N, two MMAs per K step give (x_hi + x_lo)(w_hi + w_lo).
// One CTA of 4 independent 128-thread groups per SM (they share the 32 KB of tap tables; each group runs the tile loop of a
// k_dp_fwd_fast CTA with named barriers and its own mbarriers / TMEM columns), 174 KB of shared memory.
// The accumulator TRUNCATES every group of four products at its ulp (tools/tc_accum_bench.cu), so the MMAs are issued by growing magnitude (x_lo
// steps, outer taps, the K steps with the centre taps last) and the centre tap of each contraction stays in fp32 on the CUDA cores: the output
// error against float64 is then smaller than k_dp_fwd_fast's (profiles/r02c_tc_forward.txt).
// Tile pipeline of a group (default forward kernel of the fast path since r02c):
//   wait for this tile's rx rows (cp.async issued during the previous tile) -> derive x_lo -> barrier -> issue the FIR MMAs
//   -> residual e = D - rx of the PREVIOUS tile (TMEM + registers only) while they run -> centre tap, park this tile's rx samples in the spare
//   TMEM columns -> wait, read y -> point-wise stage, E_q hi | lo into the x_lo array -> barrier -> request the NEXT tile's rx rows into x_hi,
//   issue the D MMAs -> centre tap of D -> wait -> barrier.
// Reference: twoXtwoFIR.forward sf:500-527, loss_function_shaping sf:92-137.
#include <type_traits>
#include "dp_fast.cuh"
#include "tma.cuh"

namespace vaeq {

constexpr int FC_NG = 4;                          // groups per CTA
constexpr int FC_GT = 128;                        // threads per group = TMEM lanes = 4-symbol blocks per tile
constexpr int FC_NT = FC_NG * FC_GT;
constexpr int FC_XCH = 264;                       // 16-byte chunks per rx row of a tile's sample window (1056 samples)
constexpr int FC_XCB = 4352;                      // bytes between the component rows of an x array (multiple of 256 = SWIZZLE_32B period)
constexpr int FC_XB = 4 * FC_XCB;                 // bytes of one x array (hi or lo); the lo array is reused for E_q hi | lo
constexpr int FC_QB = 8704;                       // bytes of one E_q array (528 positions x 4 components, rounded up to the SWIZZLE_64B period)
static_assert(2 * FC_QB <= FC_XB && FC_QB % 512 == 0 && FC_QB >= 528 * 16, "E_q hi | lo live in the x_lo array");
static_assert(FT_TE == 4 * FC_GT, "a tile is 128 blocks of 4 symbols");

__device__ __forceinline__ uint64_t umma_desc(uint32_t saddr, uint32_t lbo, uint32_t sbo, uint32_t layout) {
    // start >> 4 | LBO >> 4 << 16 | SBO >> 4 << 32 | version 1 << 46 | base_offset 0 (absolute-address swizzle) | layout << 61
    return (uint64_t)((saddr >> 4) & 0x3fff) | ((uint64_t)((lbo >> 4) & 0x3fff) << 16) | ((uint64_t)((sbo >> 4) & 0x3fff) << 32) | (1ull << 46) |
           ((uint64_t)layout << 61);
}
constexpr uint32_t UMMA_SW_NONE = 0, UMMA_SW64 = 4, UMMA_SW32 = 6;
// instruction descriptor: D = f32, A = B = tf32, both K-major, N >> 3 << 17, M = 128
__host__ __device__ constexpr uint32_t umma_idesc_k(int N) { return (1u << 4) | (2u << 7) | (2u << 10) | ((uint32_t)(N >> 3) << 17) | ((128u >> 4) << 24); }
__device__ __forceinline__ void umma_tf32_k(uint32_t tmem_d, uint64_t da, uint64_t db, uint32_t idesc, uint32_t acc) {
    asm volatile(
        "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n\t}\n" ::"r"(tmem_d),
        "l"(da), "l"(db), "r"(idesc), "r"(acc)
        : "memory");
}
__device__ __forceinline__ void umma_commit_to(uint64_t *bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ float tf32_lo_part(float x) {    // x - trunc_tf32(x), rounded to tf32 (the hardware would truncate it)
    const float r = x - __uint_as_float(__float_as_uint(x) & 0xffffe000u);
    uint32_t o;
    asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(o) : "f"(r));
    return __uint_as_float(o);
}
// tcgen05.ld is asynchronous: the destination registers are valid after tcgen05.wait::ld.  tmem_ld16_issue only issues the load; tmem_ld16_wait
// is the wait, with the 16 registers as read-write operands so that the compiler sees every consumer depend on it (several loads can then be
// in flight under what is, in time, one wait: the second and third wait of a batch return at once)
__device__ __forceinline__ void tmem_ld16_issue(uint32_t taddr, float (&v)[16]) {
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15}, [%16];"
                 : "=f"(v[0]), "=f"(v[1]), "=f"(v[2]), "=f"(v[3]), "=f"(v[4]), "=f"(v[5]), "=f"(v[6]), "=f"(v[7]), "=f"(v[8]), "=f"(v[9]), "=f"(v[10]),
                   "=f"(v[11]), "=f"(v[12]), "=f"(v[13]), "=f"(v[14]), "=f"(v[15])
                 : "r"(taddr));
}
__device__ __forceinline__ void tmem_ld16_wait(float (&v)[16]) {
    asm volatile("tcgen05.wait::ld.sync.aligned;"
                 : "+f"(v[0]), "+f"(v[1]), "+f"(v[2]), "+f"(v[3]), "+f"(v[4]), "+f"(v[5]), "+f"(v[6]), "+f"(v[7]), "+f"(v[8]), "+f"(v[9]), "+f"(v[10]),
                   "+f"(v[11]), "+f"(v[12]), "+f"(v[13]), "+f"(v[14]), "+f"(v[15])
                 :
                 : "memory");
}
__device__ __forceinline__ void tmem_ld16(uint32_t taddr, float (&v)[16]) {
    tmem_ld16_issue(taddr, v);
    tmem_ld16_wait(v);
}
__device__ __forceinline__ void tmem_st16(uint32_t taddr, const float (&v)[16]) {       // the caller issues tcgen05.wait::st
    asm volatile("tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,%16};" ::"r"(taddr),
                 "r"(__float_as_uint(v[0])), "r"(__float_as_uint(v[1])), "r"(__float_as_uint(v[2])), "r"(__float_as_uint(v[3])), "r"(__float_as_uint(v[4])),
                 "r"(__float_as_uint(v[5])), "r"(__float_as_uint(v[6])), "r"(__float_as_uint(v[7])), "r"(__float_as_uint(v[8])), "r"(__float_as_uint(v[9])),
                 "r"(__float_as_uint(v[10])), "r"(__float_as_uint(v[11])), "r"(__float_as_uint(v[12])), "r"(__float_as_uint(v[13])),
                 "r"(__float_as_uint(v[14])), "r"(__float_as_uint(v[15]))
                 : "memory");
}
__device__ __forceinline__ void cp_async16_zfill(void *dst_smem, const void *src_gmem, bool ok) {
    const unsigned d = (unsigned)__cvta_generic_to_shared(dst_smem);
    const int n = ok ? 16 : 0;                               // src-size 0: the 16 bytes are zero-filled, the source is not read
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(d), "l"(src_gmem), "r"(n) : "memory");
}
__device__ __forceinline__ uint32_t swz32(uint32_t off) { return off ^ (((off >> 7) & 1u) << 4); }
__device__ __forceinline__ uint32_t swz64(uint32_t off) { return off ^ (((off >> 7) & 3u) << 4); }

template <int MH>
struct FwdTcGeom {
    static constexpr int M = 2 * MH + 1, HF = MH / 2;
    static constexpr int OX = (MH + 3) / 4 * 4;              // the sample window of a block starts OX samples before its first symbol (16-byte aligned)
    static constexpr int SH = OX - MH;                       // ... i.e. SH samples before the first FIR tap
    static constexpr int NKF = (6 + 2 * MH + SH) / 8 + 1;    // FIR K steps (8 samples) per rx row: last sample used = 2*3 + 2 MH + SH
    static constexpr int NKD = (MH + 3) / 2 + 1;             // channel-convolution K steps (2 positions): last position used = 3 + MH
    static constexpr int TAPF_FLOATS = 4 * NKF * 256;        // per step: N = 32 ([hi | lo] x 4 symbols x 4 outputs) x K = 8
    static constexpr int TAPD_FLOATS = NKD * 512;            // per step: N = 64 ([hi | lo] x 2 phases x 4 symbols x 4 outputs) x K = 8
    // issue order of the MMAs (see the FIR issue loop): position t -> K step.  FIR: steps FSL, FSL + 1 of every rx row hold the taps MH - 1 ... MH + 1 of
    // the four symbols of a block (samples OX - 1 ... OX + 7); convolution: the three steps from CSL on hold positions HF ... HF + 4
    static constexpr int FSL = (OX - 1) / 8, CSL = HF / 2;
    static_assert(FSL + 1 < NKF && CSL + 2 < NKD, "centre steps");
    __host__ __device__ static constexpr int fir_step(int t) {                   // returns row * NKF + step
        if (t < 4 * NKF) return t;                           // x_lo: any order
        t -= 4 * NKF;
        if (t < 4 * (NKF - 2)) {
            const int c = t / (NKF - 2 > 0 ? NKF - 2 : 1), n = t - c * (NKF - 2);
            return c * NKF + (n < FSL ? n : n + 2);
        }
        t -= 4 * (NKF - 2);
        return (t >> 1) * NKF + FSL + (t & 1);
    }
    __host__ __device__ static constexpr int conv_step(int t) {
        if (t < NKD) return t;                               // q_lo
        t -= NKD;
        if (t < NKD - 3) return t < CSL ? t : t + 3;
        return CSL + (t - (NKD - 3));
    }
    // both orders visit every K step exactly twice (once with the lo, once with the hi operand)
    __host__ __device__ static constexpr bool orders_are_permutations() {
        for (int st = 0; st < 4 * NKF; ++st) {
            int lo = 0, hi = 0;
            for (int t = 0; t < 8 * NKF; ++t) {
                if (fir_step(t) == st) (t < 4 * NKF ? lo : hi) += 1;
            }
            if (lo != 1 || hi != 1) return false;
        }
        for (int st = 0; st < NKD; ++st) {
            int lo = 0, hi = 0;
            for (int t = 0; t < 2 * NKD; ++t) {
                if (conv_step(t) == st) (t < NKD ? lo : hi) += 1;
            }
            if (lo != 1 || hi != 1) return false;
        }
        return true;
    }
    static constexpr size_t GROUP0 = 2048 + (size_t)(TAPF_FLOATS + TAPD_FLOATS) * 4;
    static constexpr size_t SMEM = GROUP0 + (size_t)FC_NG * 2 * FC_XB;
    static_assert(8 * 127 + 8 * NKF <= 4 * FC_XCH && 8 * 127 + OX + 8 <= 4 * FC_XCH, "sample window");
    static_assert(4 * 127 + 2 * NKD <= 528 && HF <= FT_HP - 2, "E_q window");
    static_assert(GROUP0 % 1024 == 0, "swizzled arrays need their pattern alignment");
};

template <int NL, int MH>
__global__ void __launch_bounds__(FC_NT, 1) k_dp_fwd_tc(DpK p) {
    using G = FwdTcGeom<MH>;
    static_assert(G::orders_are_permutations(), "MMA issue order");
    constexpr int M = G::M, HF = G::HF, OX = G::OX, SH = G::SH, NKF = G::NKF, NKD = G::NKD;
    extern __shared__ __align__(1024) unsigned char smem[];
    uint64_t *bars = reinterpret_cast<uint64_t *>(smem);                 // fir_done[4], conv_done[4]
    uint32_t *tmem_slot = reinterpret_cast<uint32_t *>(smem + 64);
    int *s_next = reinterpret_cast<int *>(smem + 80);                    // [4]
    float *red = reinterpret_cast<float *>(smem + 128);                  // [4 groups][4 warps][8]
    FastConst *cst = reinterpret_cast<FastConst *>(smem + 640);
    float4 *ctrF = reinterpret_cast<float4 *>(smem + 1024), *ctrD = ctrF + 12;   // taps k = MH - 1 + d of W, h: [d][input component] -> 4 outputs
    float *tapF = reinterpret_cast<float *>(smem + 2048);
    float *tapD = tapF + G::TAPF_FLOATS;
    const int tid = threadIdx.x, gt = tid & 127, lane = tid & 31;
    const int warp_u = __shfl_sync(0xffffffffu, tid >> 5, 0);           // warp-uniform for the compiler: descriptors and barrier ids live in uniform registers
    const int g = warp_u >> 2, wq = warp_u & 3;
    unsigned char *xhi = smem + G::GROUP0 + (size_t)g * 2 * FC_XB, *xlo = xhi + FC_XB;
    unsigned char *qhi = xlo, *qlo = xlo + FC_QB;                        // E_q arrays: written after the FIR MMAs have read x_lo

    // ---- tap tables (K-major, no swizzle: core matrices of 8 n-rows x 16 bytes; n-groups 256 B apart, the two k halves 128 B apart) ----
    for (int idx = tid; idx < G::TAPF_FLOATS; idx += FC_NT) {
        const int step = idx >> 8, rem = idx & 255, n = (rem >> 6) * 8 + ((rem & 31) >> 2), k8 = ((rem >> 5) & 1) * 4 + (rem & 3);
        const int c = step / NKF, s = step - c * NKF, j = 8 * s + k8;
        const int half = n >> 4, i = (n >> 2) & 3, o = n & 3, k = j - 2 * i - SH;
        float v = 0.f;
        if (k >= 0 && k < M && (k < MH || k > MH)) {         // the centre tap stays on the CUDA cores (see below)
            const int op = o >> 1, oc = o & 1, ip = c >> 1, ic = c & 1;
            const float tr = p.W[(op * 4 + ip) * M + k], ti = p.W[(op * 4 + 2 + ip) * M + k];
            v = oc == ic ? tr : (oc ? ti : -ti);             // Re = tr xr - ti xi, Im = ti xr + tr xi
        }
        tapF[idx] = half ? tf32_lo_part(v) : v;
    }
    for (int idx = tid; idx < G::TAPD_FLOATS; idx += FC_NT) {
        const int step = idx >> 9, rem = idx & 511, n = (rem >> 6) * 8 + ((rem & 31) >> 2), k8 = ((rem >> 5) & 1) * 4 + (rem & 3);
        const int j = 2 * step + (k8 >> 2), c = k8 & 3;
        const int half = n >> 5, ph = (n >> 4) & 1, i = (n >> 2) & 3, o = n & 3, a = j - i - ph;
        float v = 0.f;
        const int jj = ph ? 2 * MH - 1 - 2 * a : 2 * MH - 2 * a;
        if (a >= 0 && a < (ph ? MH : MH + 1) && (jj < MH || jj > MH)) {  // even samples: h[2MH - 2a] E_q[u + a - HF];  odd: h[2MH - 1 - 2b] E_q[u + b - HF + 1]
            const int chi = o >> 1, oc = o & 1, nu = c >> 1, ic = c & 1;
            const float hr = p.h[((chi * 2 + nu) * 2 + 0) * M + jj], hi_ = p.h[((chi * 2 + nu) * 2 + 1) * M + jj];
            v = oc == ic ? hr : (oc ? hi_ : -hi_);
        }
        tapD[idx] = half ? tf32_lo_part(v) : v;
    }
    // real-expanded taps k = MH - 1 + d of W and h, [d][input component].{4 outputs}; only the centre tap (d = 1) is read.  The table keeps
    // its three entries: with one, ptxas allocates k_dp_fwd_tc<8, 12> differently and spills 4 bytes
    if (tid < 96) {
        const int fam = tid / 48, e = tid % 48, d = e / 16, ci = (e >> 2) & 3, o = e & 3, k = MH - 1 + d;
        const int op = o >> 1, oc = o & 1, ip = ci >> 1, ic = ci & 1;
        const float tr = fam ? p.h[((op * 2 + ip) * 2 + 0) * M + k] : p.W[(op * 4 + ip) * M + k];
        const float ti = fam ? p.h[((op * 2 + ip) * 2 + 1) * M + k] : p.W[(op * 4 + 2 + ip) * M + k];
        reinterpret_cast<float *>(fam ? ctrD : ctrF)[(d * 4 + ci) * 4 + o] = oc == ic ? tr : (oc ? ti : -ti);
    }
    load_fast_const(cst, p.amp, p.P, p.var, p.nu_sc, NL);
    if (tid == 0) {
        for (int b = 0; b < 2 * FC_NG; ++b) mbar_init(bars + b, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (tid < 32) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], 512;" ::"r"(smem_u32(tmem_slot)) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");        // the tap tables are read by the tensor core
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    const uint32_t tmem = *tmem_slot;
    const FastConst &c = *cst;

    uint64_t *bar_f = bars + g, *bar_d = bars + FC_NG + g;
    const uint32_t tm_y = tmem + 128 * g + ((uint32_t)(32 * wq) << 16), tm_d = tm_y + 32, tm_x = tm_y + 96;       // this warp's TMEM lanes, this group's columns: y 32, D 64, parked rx 32
    const int nv = (int)gridDim.x * FC_NG, vcta = (int)blockIdx.x * FC_NG + g;                  // a group is a virtual CTA of the tile loop
    const int i0 = FT_R * gt;
    float accC[2] = {0.f, 0.f}, accEnt = 0.f, accV0 = 0.f, accV1 = 0.f;
    uint32_t par = 0;
    // cp.async of a tile's rx window into x_hi; a chunk lies entirely inside or outside [0, L) (zero-filled outside)
    auto stage_rx = [&](int tile_s) {
        const int64_t o_smp = 2 * (int64_t)(p.clo + tile_s * FT_T - FT_HP) - OX;            // global sample index of window sample 0
#pragma unroll 1
        for (int ch = gt; ch < FC_XCH; ch += FC_GT) {
            const int64_t s0 = o_smp + 4 * ch;
            const bool ok = s0 >= 0 && s0 + 3 < p.L;
            const uint32_t off = swz32(16u * ch);
            const float *src = p.rx + (ok ? s0 : 0);
#pragma unroll
            for (int r = 0; r < 4; ++r) cp_async16_zfill(xhi + r * FC_XCB + off, src + (int64_t)r * p.ld_rx, ok);
        }
        asm volatile("cp.async.commit_group;" ::: "memory");
    };
    // ---- residual e = D - rx of the tile whose D MMAs were waited for last (t0_res): deferred, so that it runs while the FIR MMAs of the NEXT tile
    // execute (every thread used to wait ~0.7 us per tile for them with nothing to do).  D accumulator and parked rx come from TMEM, the centre-tap part
    // dc from registers; nothing here touches shared memory.
    float2 dc[2][FT_R][2];
    int t0_res = 0;
    bool have_res = false;
    auto residual = [&]() {
        const int u0 = t0_res - FT_HP + i0;
        const bool in_seq = (u0 >= 0) && (u0 < p.B);
        const bool owned = in_seq && (i0 >= FT_HP) && (i0 < FT_HP + FT_T) && (u0 < p.chi);
        const bool counted = owned && (u0 >= p.sym_lo) && (u0 < p.sym_hi);
#pragma unroll
        for (int ph = 0; ph < 2; ++ph) {
            float dh[16], dl[16];
            float xs[16];
            tmem_ld16_issue(tm_d + 16 * ph, dh);
            tmem_ld16_issue(tm_d + 32 + 16 * ph, dl);
            tmem_ld16_issue(tm_x + 16 * ph, xs);
            tmem_ld16_wait(dh);
            tmem_ld16_wait(dl);
            tmem_ld16_wait(xs);
            if (owned) {
                float ev[4][FT_R];
#pragma unroll
                for (int k = 0; k < 4; ++k) {
#pragma unroll
                    for (int r = 0; r < FT_R; ++r) {
                        const int s = 2 * (u0 + r) + ph;
                        const bool valid = (s >= MH) && (s < p.L - MH);                     // sf:120 "valid" region
                        const float2 dcv = dc[ph][r][k >> 1];
                        ev[k][r] = valid ? ((dh[4 * r + k] + dl[4 * r + k]) + ((k & 1) ? dcv.y : dcv.x)) - xs[4 * k + r] : 0.f;
                    }
                }
                if (counted) {
#pragma unroll
                    for (int r = 0; r < FT_R; ++r) {
                        accC[0] += ev[0][r] * ev[0][r] + ev[1][r] * ev[1][r];
                        accC[1] += ev[2][r] * ev[2][r] + ev[3][r] * ev[3][r];
                    }
                }
#pragma unroll
                for (int k = 0; k < 4; ++k) st_row4(p.erows, p.B, 4 * ph + k, u0, make_float4(ev[k][0], ev[k][1], ev[k][2], ev[k][3]));
            }
        }
    };
    if (vcta < p.ntiles) stage_rx(vcta);

#pragma unroll 1
    for (int tile = vcta; tile < p.ntiles; par ^= 1) {
        const int t0 = p.clo + tile * FT_T;
        if (gt == 0) s_next[g] = p.dyn ? atomicAdd(p.tile_ctr, 1) + nv : tile + nv;
        // ---- the tile's rx window (every rx row as it lies in HBM, 16-byte chunks, SWIZZLE_32B by absolute address) was requested by cp.async
        // during the previous tile (see stage_rx below); the thread derives the lo parts of ITS OWN chunks (no barrier in between).
        asm volatile("cp.async.wait_group 0;" ::: "memory");
#pragma unroll 1
        for (int ch = gt; ch < FC_XCH; ch += FC_GT) {
            const uint32_t off = swz32(16u * ch);
#pragma unroll
            for (int r = 0; r < 4; ++r) {
                const float4 v = *reinterpret_cast<const float4 *>(xhi + r * FC_XCB + off);
                *reinterpret_cast<float4 *>(xlo + r * FC_XCB + off) = make_float4(tf32_lo_part(v.x), tf32_lo_part(v.y), tf32_lo_part(v.z), tf32_lo_part(v.w));
            }
        }
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
        named_bar_sync(1 + g, FC_GT);
        const int tile_next = s_next[g];
        if (gt == 0) {
            // ---- FIR: Y (128 x 32) = sum over the 4 rx rows and NKF K steps of (x_hi + x_lo) [w_hi | w_lo] ----
            asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
            // fully unrolled: every descriptor is a base descriptor + a compile-time constant, so the single issuing thread spends two
            // 64-bit adds per MMA (a rolled loop with the descriptor arithmetic inside kept the other 127 threads waiting ~3000 cycles)
            const uint64_t dah = umma_desc(smem_u32(xhi), 16, 256, UMMA_SW32), dal = umma_desc(smem_u32(xlo), 16, 256, UMMA_SW32);
            const uint64_t db0 = umma_desc(smem_u32(tapF), 128, 256, UMMA_SW_NONE);
            // order: the tensor core truncates every group of four products at the ulp of the accumulator (tools/tc_accum_bench.cu), so the
            // terms go in by growing magnitude -- all x_lo steps, then the x_hi steps without a centre tap, and the K steps that hold the
            // centre taps (|w| ~ 1) LAST: only those few accumulate at the ulp of the final value
#pragma unroll
            for (int t = 0; t < 8 * NKF; ++t) {
                const int st = G::fir_step(t);
                const uint64_t ao = (uint64_t)(((st / NKF) * FC_XCB + 32 * (st % NKF)) >> 4), bo = (uint64_t)((st * 1024) >> 4);
                umma_tf32_k(tmem + 128 * g, (t < 4 * NKF ? dal : dah) + ao, db0 + bo, umma_idesc_k(32), t != 0);
            }
            umma_commit_to(bar_f);
        }
        __syncwarp();
        if (have_res) residual();                            // previous tile: behind this tile's FIR MMAs
        const int u0 = t0 - FT_HP + i0;
        const bool in_seq = (u0 >= 0) && (u0 < p.B);         // B % 4 == 0: all four symbols in or out together
        const bool owned = in_seq && (i0 >= FT_HP) && (i0 < FT_HP + FT_T) && (u0 < p.chi);
        const bool counted = owned && (u0 >= p.sym_lo) && (u0 < p.sym_hi);   // sums only over this rank's symbols
        // the centre tap (k = MH: sample 2u) on the CUDA cores, in fp32, while the MMAs run: the
        // tensor core TRUNCATES every group of four products at the accumulator's ulp (tools/tc_accum_bench.cu), so the terms of
        // magnitude ~1 must not pass through it; what remains there is ~0.1 and its truncation error below the fp32 rounding noise
        float y[FT_R][4];
        {
            float2 yc[FT_R][2];
#pragma unroll
            for (int r = 0; r < FT_R; ++r) yc[r][0] = yc[r][1] = make_float2(0.f, 0.f);
            const uint32_t ch = 2u * gt + OX / 4;
            float rxs[2][16];                                // this thread's own samples [phase][4 component + symbol]: parked in TMEM for the residual
#pragma unroll
            for (int ci = 0; ci < 4; ++ci) {
                const unsigned char *row = xhi + ci * FC_XCB;
                const float4 xa = *reinterpret_cast<const float4 *>(row + swz32(16u * ch)), xb = *reinterpret_cast<const float4 *>(row + swz32(16u * (ch + 1)));
                rxs[0][4 * ci + 0] = xa.x; rxs[0][4 * ci + 1] = xa.z; rxs[0][4 * ci + 2] = xb.x; rxs[0][4 * ci + 3] = xb.z;
                rxs[1][4 * ci + 0] = xa.y; rxs[1][4 * ci + 1] = xa.w; rxs[1][4 * ci + 2] = xb.y; rxs[1][4 * ci + 3] = xb.w;
                const float4 w = ctrF[4 + ci];
#pragma unroll
                for (int r = 0; r < FT_R; ++r) {
                    const float2 xx = make_float2(rxs[0][4 * ci + r], rxs[0][4 * ci + r]);
                    yc[r][0] = __ffma2_rn(make_float2(w.x, w.y), xx, yc[r][0]);
                    yc[r][1] = __ffma2_rn(make_float2(w.z, w.w), xx, yc[r][1]);
                }
            }
            // x_hi is not read again after this point (the FIR MMAs are waited for just below): the samples the residual e = D - rx needs go to
            // the group's 32 spare TMEM columns (lane = thread), so that the NEXT tile's rows can land in x_hi during the rest of this tile
            tmem_st16(tm_x, rxs[0]);
            tmem_st16(tm_x + 16, rxs[1]);
            asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory");
            mbar_wait(bar_f, par);
            asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
            float vh[16], vl[16];
            tmem_ld16_issue(tm_y, vh);
            tmem_ld16_issue(tm_y + 16, vl);
            tmem_ld16_wait(vh);
            tmem_ld16_wait(vl);
#pragma unroll
            for (int r = 0; r < FT_R; ++r) {
                y[r][0] = (vh[4 * r] + vl[4 * r]) + yc[r][0].x;
                y[r][1] = (vh[4 * r + 1] + vl[4 * r + 1]) + yc[r][0].y;
                y[r][2] = (vh[4 * r + 2] + vl[4 * r + 2]) + yc[r][1].x;
                y[r][3] = (vh[4 * r + 3] + vl[4 * r + 3]) + yc[r][1].y;
            }
        }
        // E_q position of local symbol i0 + r is i0 + r + HF (the window of a block then starts at its own row)
        const uint32_t qoff0 = 16u * (i0 + HF);
        if (!in_seq) {
#pragma unroll
            for (int r = 0; r < FT_R; ++r) {
                const uint32_t off = swz64(qoff0 + 16u * r);
                *reinterpret_cast<float4 *>(qhi + off) = make_float4(0.f, 0.f, 0.f, 0.f);
                *reinterpret_cast<float4 *>(qlo + off) = make_float4(0.f, 0.f, 0.f, 0.f);
            }
        } else {
            // point-wise stage, rolled over the polarisation (code size); y rotates by two components per pass.  Moment form when the prior is of the
            // Maxwell-Boltzmann family (CTA-uniform: one of the two instantiations runs for the whole launch)
            auto pointwise = [&](auto mom_tag) {
            constexpr bool MOM = decltype(mom_tag)::value;
#pragma unroll 1
            for (int pol = 0; pol < 2; ++pol) {
                float vs[FT_R];
#pragma unroll
                for (int cq = 0; cq < 2; ++cq) {
                    const int cc = 2 * pol + cq;
                    float qv[FT_R][NL], m1v[FT_R], s1v[FT_R], t2v[FT_R], s3v[FT_R];
                    if (MOM) {                               // moment form, a symbol pair per packed instruction (dp_math.cuh, as in k_dp_fwd_fast)
#pragma unroll
                        for (int r = 0; r < FT_R; r += 2) {
                            float2 q2[NL], m1p, vp, entp, s1p, t2p, s3p;
                            demap_mom2<NL>(make_float2(y[r][cq], y[r + 1][cq]), c.ct[pol], c.eps[pol], c.inv_var[pol], c, q2, m1p, vp, entp, s1p, t2p, s3p);
#pragma unroll
                            for (int l = 0; l < NL; ++l) { qv[r][l] = q2[l].x; qv[r + 1][l] = q2[l].y; }
                            m1v[r] = m1p.x; m1v[r + 1] = m1p.y;
                            s1v[r] = s1p.x; s1v[r + 1] = s1p.y;
                            t2v[r] = t2p.x; t2v[r + 1] = t2p.y;
                            s3v[r] = s3p.x; s3v[r + 1] = s3p.y;
                            const int u = u0 + r;
                            if (counted && u >= MH && u < p.B - MH) accEnt += entp.x;         // sf:132
                            if (counted && u + 1 >= MH && u + 1 < p.B - MH) accEnt += entp.y;
                            vs[r] = cq ? vs[r] + vp.x : vp.x;
                            vs[r + 1] = cq ? vs[r + 1] + vp.y : vp.y;
                        }
                    } else {
#pragma unroll
                        for (int r = 0; r < FT_R; ++r) {
                            float m2, ent, S2;
                            demap_fast<NL, true>(y[r][cq], c.c2[pol], c.inv_var[pol], c, qv[r], m1v[r], m2, ent, s1v[r], S2, s3v[r]);
                            t2v[r] = fmaf(-2.f * m1v[r], s1v[r], S2);
                            const int u = u0 + r;
                            if (counted && u >= MH && u < p.B - MH) accEnt += ent;            // sf:132
                            const float v = m2 - m1v[r] * m1v[r];                             // sf:113
                            vs[r] = cq ? vs[r] + v : v;
                        }
                    }
#pragma unroll
                    for (int r = 0; r < FT_R; ++r) {
                        const uint32_t off = swz64(qoff0 + 16u * r) + 4u * cc;
                        *reinterpret_cast<float *>(qhi + off) = m1v[r];
                        *reinterpret_cast<float *>(qlo + off) = tf32_lo_part(m1v[r]);
                    }
                    if (owned) {
                        if (p.q != nullptr) {                // NULL in the frame loops that only keep a section of every window
#pragma unroll
                            for (int l = 0; l < NL; ++l)
                                st_row4(p.q, p.ld_q, cc * NL + l, u0, make_float4(qv[0][l], qv[1][l], qv[2][l], qv[3][l]));
                            st_row4(p.out, p.ld_out, cc, u0, make_float4(y[0][cq], y[1][cq], y[2][cq], y[3][cq]));
                        }
                        st_row4(p.m1rows, p.B, cc, u0, make_float4(m1v[0], m1v[1], m1v[2], m1v[3]));
                        if (p.need_bwd) {
                            st_row4(p.srows, p.B, cc, u0, make_float4(s1v[0], s1v[1], s1v[2], s1v[3]));
                            st_row4(p.srows, p.B, 4 + cc, u0, make_float4(t2v[0], t2v[1], t2v[2], t2v[3]));
                            st_row4(p.srows, p.B, 8 + cc, u0, make_float4(s3v[0], s3v[1], s3v[2], s3v[3]));
                        }
                        if (p.qk != nullptr && counted) {    // batch-split: the rank that counts a symbol keeps it
                            const int k0 = u0 - p.keep_lo;
                            if (p.keep_vec && k0 >= 0 && k0 + FT_R <= p.keep_n) {            // all four symbols kept, 16-byte aligned destination
                                const int64_t col = p.keep_base + k0;
#pragma unroll
                                for (int l = 0; l < NL; ++l)
                                    *reinterpret_cast<float4 *>(p.qk + (int64_t)(cc * NL + l) * p.ld_qk + col) = make_float4(qv[0][l], qv[1][l], qv[2][l], qv[3][l]);
                                *reinterpret_cast<float4 *>(p.outk + (int64_t)cc * p.ld_outk + col) = make_float4(y[0][cq], y[1][cq], y[2][cq], y[3][cq]);
                            } else if (k0 > -FT_R && k0 < p.keep_n) {
#pragma unroll 1
                                for (int r = 0; r < FT_R; ++r) {
                                    const int u = u0 + r;
                                    if (u >= p.keep_lo && u < p.keep_lo + p.keep_n) {
                                        const int64_t col = p.keep_base + (u - p.keep_lo);
                                        for (int l = 0; l < NL; ++l)
                                            p.qk[(int64_t)(cc * NL + l) * p.ld_qk + col] = f4c(make_float4(qv[0][l], qv[1][l], qv[2][l], qv[3][l]), r);
                                        p.outk[(int64_t)cc * p.ld_outk + col] = f4c(make_float4(y[0][cq], y[1][cq], y[2][cq], y[3][cq]), r);
                                    }
                                }
                            }
                        }
                    }
                }
                if (counted) {
                    const float vsum = (vs[0] + vs[1]) + (vs[2] + vs[3]);
                    accV0 += pol ? 0.f : vsum;
                    accV1 += pol ? vsum : 0.f;
#pragma unroll
                    for (int r = 0; r < FT_R; ++r) {
                        const int u = u0 + r;
                        if (u < MH || u >= p.B - MH) {
                            const int slot = (u < MH) ? u : MH + (u - (p.B - MH));
                            p.edge_vs[2 * MH * pol + slot] = vs[r];
                        }
                    }
                }
#pragma unroll
                for (int r = 0; r < FT_R; ++r) {             // rotate: the next pass finds its components in slots 0,1
                    float t;
                    t = y[r][0]; y[r][0] = y[r][2]; y[r][2] = t;
                    t = y[r][1]; y[r][1] = y[r][3]; y[r][3] = t;
                }
            }
            };
            if (c.quad) pointwise(std::true_type{});
            else pointwise(std::false_type{});
        }
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
        asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
        named_bar_sync(1 + g, FC_GT);
        if (gt == 0) {
            // ---- D (128 x 64: [hi | lo] x even / odd sample x 4 symbols x 4 components) = sum over NKD K steps of (q_hi + q_lo) [h_hi | h_lo] ----
            asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
            const uint64_t dqh = umma_desc(smem_u32(qhi), 16, 512, UMMA_SW64), dql = umma_desc(smem_u32(qlo), 16, 512, UMMA_SW64);
            const uint64_t db0 = umma_desc(smem_u32(tapD), 128, 256, UMMA_SW_NONE);
#pragma unroll
            for (int t = 0; t < 2 * NKD; ++t) {              // same order as the FIR: lo parts, outer taps, centre taps
                const int st = G::conv_step(t);
                const uint64_t ao = (uint64_t)((32 * st) >> 4), bo = (uint64_t)((st * 2048) >> 4);
                umma_tf32_k(tmem + 128 * g + 32, (t < NKD ? dql : dqh) + ao, db0 + bo, umma_idesc_k(64), t != 0);
            }
            umma_commit_to(bar_d);
        }
        __syncwarp();
        if (tile_next < p.ntiles) stage_rx(tile_next);       // every thread of the group is past its last read of x_hi (barrier above): the rows land during the D MMAs and the next tile's top
        // centre tap of h (j = MH) on the CUDA cores while the MMAs run: even sample h[MH] E_q[u]; the odd samples have no centre-tap term
        {
            float4 eq[FT_R];
#pragma unroll
            for (int r = 0; r < FT_R; ++r) eq[r] = *reinterpret_cast<const float4 *>(qhi + swz64(qoff0 + 16u * r));
#pragma unroll
            for (int r = 0; r < FT_R; ++r) {
                float2 a0 = make_float2(0.f, 0.f), a1 = a0;
#pragma unroll
                for (int ci = 0; ci < 4; ++ci) {
                    const float4 w = ctrD[4 + ci];
                    const float q0 = f4c(eq[r], ci);
                    a0 = __ffma2_rn(make_float2(w.x, w.y), make_float2(q0, q0), a0);
                    a1 = __ffma2_rn(make_float2(w.z, w.w), make_float2(q0, q0), a1);
                }
                dc[0][r][0] = a0; dc[0][r][1] = a1; dc[1][r][0] = dc[1][r][1] = make_float2(0.f, 0.f);
            }
        }
        mbar_wait(bar_d, par);
        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");

        t0_res = t0;                                         // the residual of this tile runs behind the FIR MMAs of the next one (or after the loop)
        have_res = true;
        asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
        named_bar_sync(1 + g, FC_GT);                        // x_hi, the E_q arrays and both accumulators are free for the next tile
        tile = tile_next;
    }

    if (have_res) residual();                                // last tile

    // ---- this group's partial sums (fixed order) ----
    {
        float v[5] = {accC[0], accC[1], accEnt, accV0, accV1};
#pragma unroll
        for (int i = 0; i < 5; ++i) v[i] = warp_sum(v[i]);
        if (lane == 0) {
#pragma unroll
            for (int i = 0; i < 5; ++i) red[(g * 4 + wq) * 8 + i] = v[i];
        }
        named_bar_sync(1 + g, FC_GT);
        if (gt == 0) {
            double *dst = p.part_fwd + (int64_t)vcta * 8;
#pragma unroll
            for (int i = 0; i < 5; ++i) dst[i] = (double)((red[(g * 4 + 0) * 8 + i] + red[(g * 4 + 1) * 8 + i]) + (red[(g * 4 + 2) * 8 + i] + red[(g * 4 + 3) * 8 + i]));
        }
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    if (tid < 32) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, 512;" ::"r"(tmem) : "memory");
}

template <int NL, int MH>
static int fwd_tc_launch_t(DpK p, cudaStream_t st, int *nparts) {
    static SmemAttrCache set;
    using G = FwdTcGeom<MH>;
    if (int rc = ensure_dyn_smem(k_dp_fwd_tc<NL, MH>, G::SMEM, set)) return rc;
    const int nvc = min(FC_NG * sm_count(), p.ntiles), grid = (nvc + FC_NG - 1) / FC_NG;
    ktime_begin(VAEQ_K_DP_FWD, st);
    k_dp_fwd_tc<NL, MH><<<grid, FC_NT, G::SMEM, st>>>(p);
    ktime_end(VAEQ_K_DP_FWD, st);
    VAEQ_LAUNCH_CHECK("k_dp_fwd_tc");
    *nparts = grid * FC_NG;
    return VAEQ_OK;
}

// forward kernel of the fast path with its contractions on tcgen05; p.ntiles = number of 496-symbol tiles; returns 0 if (n_lev, M_est)
// is not built
int dp_fwd_tc_launch(const DpK &p, int n_lev, cudaStream_t st, int *nparts, int *rc) {
#define TC_CASE(NL_, MH_)                                           \
    if (n_lev == NL_ && p.mh == MH_) {                              \
        *rc = fwd_tc_launch_t<NL_, MH_>(p, st, nparts);             \
        return 1;                                                   \
    }
    TC_CASE(8, 12)
    TC_CASE(8, 6)
    TC_CASE(8, 4)
    TC_CASE(8, 2)
    TC_CASE(4, 12)
    TC_CASE(2, 12)
#undef TC_CASE
    return 0;
}

}  // namespace vaeq
