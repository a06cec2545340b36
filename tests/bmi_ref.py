"""Float64 reference of the Gray-labelled bits, the bit-metric decoding rate (BMI) and the bit LLRs (an extension, not in the reference
implementation), the definition the CUDA BMI and bit-LLR kernels are checked against.  Level indices of tx come from
oracle.vaeq_oracle._tx_levels, the same mapping oracle.gmi_from_posteriors uses."""
import torch

from oracle.vaeq_oracle import _tx_levels


def gray_labels(n):
    """Binary reflected Gray labels g(l) = l ^ (l >> 1) of the n levels of an ASK component, ascending level index, MSB first;
    g(n - 1 - l) = g(l) ^ 2^(m-1), so mirroring a level flips its MSB only."""
    return torch.tensor([l ^ (l >> 1) for l in range(n)], dtype=torch.int64)


def label_bits(n):
    """(m, n) int64: bit i (0 = MSB) of the label of level l."""
    m = n.bit_length() - 1
    g = gray_labels(n)
    return torch.stack([(g >> (m - 1 - i)) & 1 for i in range(m)])


def bit_posteriors(q):
    """q (..., 2n, N) level posteriors, I rows then Q rows -> (..., 2m, 2, N) float64: q_c(b_i = v | y) = sum of q_c[l] over the levels
    whose label has bit i = v, rows [I bits MSB..LSB | Q bits MSB..LSB], v = 0, 1.  No renormalisation."""
    n = q.shape[-2] // 2
    bits = label_bits(n).double()
    qd = q.double()
    rows = []
    for c in range(2):
        qc = qd[..., c * n:(c + 1) * n, :]
        for b in bits:
            b = b.view(n, 1)
            rows.append(torch.stack(((qc * (1 - b)).sum(-2), (qc * b).sum(-2)), dim=-2))
    return torch.stack(rows, dim=-3)


def bmi_from_posteriors(q, tx, P):
    """Bit-metric decoding rate of the Gray-labelled bits, H(X) + mean over the symbols of sum over c in {I, Q}, i < m of
    log2 max(q_c(b_i = bit i of g(lev_c) | y), 1e-30), per pol in bit/2D-symbol, float64 (the counterpart of
    oracle.gmi_from_posteriors): q (2,2n,N), tx (2,2,N) float16 whose levels are lev_c, P (n,) pmf."""
    n = q.shape[1] // 2
    m = n.bit_length() - 1
    idx = _tx_levels(tx, n)
    Pt = torch.as_tensor(P).to(torch.float64)
    H = -2 * torch.sum(Pt * torch.log2(Pt))
    bits, pb = label_bits(n), bit_posteriors(q)
    ll = torch.zeros(q.shape[0], q.shape[-1], dtype=torch.float64)
    for c in range(2):
        for i in range(m):
            v = bits[i][idx[:, c, :]]
            p = torch.gather(pb[:, c * m + i], 1, v.unsqueeze(1)).squeeze(1)
            ll += torch.log2(torch.clamp(p, min=1e-30))
    return H + ll.mean(dim=-1)


def bit_llr_from_posteriors(q):
    """Bit LLRs L = ln max(q_c(b_i = 0 | y), 1e-30) - ln max(q_c(b_i = 1 | y), 1e-30) (positive: bit 0), float64: q (..., 2n, N) ->
    (..., 2m, N), rows [I bits MSB..LSB | Q bits MSB..LSB]."""
    pb = torch.clamp(bit_posteriors(q), min=1e-30)
    return torch.log(pb[..., 0, :]) - torch.log(pb[..., 1, :])
