// Gray-labelled bits of the ASK components (extension, not in the reference): the labelling and the bit marginals of the level
// posteriors, shared by the bit-metric rate (BMI: eval.cu k_gmi<.., BITS>, eval_runs.cu k_gmi_runs<.., BITS>) and the bit LLRs
// (eval.cu k_bit_llr), so the labelling exists once in the library.
#pragma once

namespace vaeq {

// Labels: per ASK component the binary reflected Gray code over the ascending level index, g(l) = l ^ (l >> 1), m = log2(NL) bits,
// MSB first (NL 2: 0 1; 4: 0 1 3 2; 8: 0 1 3 2 6 7 5 4).  With S = NL - 1 the labels satisfy g(S - l) = g(l) ^ 2^(m-1): mirroring a
// level, which is what the rotations by pi and pi/2 and the IQ flip do to a component, flips the MSB of its label and leaves the other
// bits.  Under any of those hypotheses the set of levels with bit i = v maps onto a set with bit i = v' for every i, so the bit-metric
// rate is invariant under the same symmetries the SER forgives.
__host__ __device__ constexpr int gray_label(int l) { return l ^ (l >> 1); }
template <int NL>
__host__ __device__ constexpr int gray_bits() { return NL == 2 ? 1 : NL == 4 ? 2 : 3; }
// bit i (0 = MSB) of the label of level l
template <int NL>
__host__ __device__ constexpr int gray_bit(int l, int i) { return (gray_label(l) >> (gray_bits<NL>() - 1 - i)) & 1; }

// Bit posteriors of one component, q(b_i = v | y) = sum over the levels l with bit i of g(l) equal to v of qv[l], i = 0 (MSB) .. m - 1,
// v = 0, 1; no renormalisation (as GMI, q is used as given).  T: the accumulation type (double for the rate, float for the LLRs).
template <int NL, typename T>
__device__ __forceinline__ void bit_marginals(const float (&qv)[NL], T (&pb)[gray_bits<NL>()][2]) {
#pragma unroll
    for (int i = 0; i < gray_bits<NL>(); ++i) {
        pb[i][0] = T(0);
        pb[i][1] = T(0);
#pragma unroll
        for (int l = 0; l < NL; ++l) pb[i][gray_bit<NL>(l, i)] += (T)qv[l];
    }
}

// One component's share of the BMI sum: sum over the m bits of log2 max(q(b_i = bit i of g(lev) | y), 1e-30), in double, taken as the
// log2 of the product of the clamped factors (at least 1e-90: no underflow), so a symbol costs one log per component as GMI does
template <int NL>
__device__ __forceinline__ double bmi_log2_component(const float (&qv)[NL], int lev) {
    constexpr int m = gray_bits<NL>();
    double pb[m][2];
    bit_marginals<NL>(qv, pb);
    const int g = gray_label(lev);
    double prod = 1.0;
#pragma unroll
    for (int i = 0; i < m; ++i) prod *= fmax((g >> (m - 1 - i)) & 1 ? pb[i][1] : pb[i][0], 1e-30);
    return log2(prod);
}

}  // namespace vaeq
