"""The error bound behind precision="exact" (DESIGN section 2.1), checked in numpy without a GPU.

|s_bf16(u, j) - s_fp32(u, j)| <= eps_u = RHO * S_u + RHO_B * b_max, S_u = sum_i |u_i| c_i, c_i = max_j |E[j, i]|.
s_bf16 is emulated as the tensor-core kernel forms it: round-to-nearest bf16 operands (encode.cu, prep.cu), exact
products, fp32 accumulation over the four K = 16 steps and the hi/mid/lo bf16 split of the bias.  s_fp32 follows the
fp32 path (score.cu): four interleaved 16-FMA chains, ((a0 + a1) + (a2 + a3)) + bias.  A bound with half of RHO fails
on a constructed case, so the operand term is not loose by a factor of two."""
import numpy as np
import torch

RHO = 2.0 ** -7 + 2.0 ** -12       # exact.cu
RHO_B = 2.0 ** -12
F32 = np.float32


def bf16(x):
    """Round-to-nearest-even fp32 -> bf16 (returned as fp32)."""
    b = np.asarray(x, dtype=F32).view(np.uint32).astype(np.uint64)
    b = (b + 0x7FFF + ((b >> 16) & 1)) & 0xFFFF0000
    return b.astype(np.uint32).view(F32)


def split3(bias):
    hi = bf16(bias)
    mid = bf16(bias - hi)
    lo = bf16((bias - hi) - mid)
    return hi, mid, lo


def fp32_path(u, E, bias):
    """[B, N] scores with the fp32 kernel's operation order (fmaf emulated in float64, then rounded)."""
    a = [np.zeros((u.shape[0], E.shape[0]), F32) for _ in range(4)]
    for k in range(64):
        p = u[:, k, None].astype(np.float64) * E[None, :, k].astype(np.float64)
        a[k % 4] = (p + a[k % 4]).astype(F32)
    return (((a[0] + a[1]) + (a[2] + a[3])) + bias[None, :]).astype(F32)


def bf16_path(u, E, bias):
    """[B, N] tensor-core scores: bf16 operands, exact products, fp32 accumulation, folded bias split."""
    ub, Eb = bf16(u), bf16(E)
    acc = np.zeros((u.shape[0], E.shape[0]), F32)
    for k in range(64):
        acc = (acc + (ub[:, k, None].astype(np.float64) * Eb[None, :, k].astype(np.float64))).astype(F32)
    for term in split3(bias):
        acc = (acc + term[None, :]).astype(F32)
    return acc


def eps(u, E, bias, rho=RHO):
    c = np.abs(E).max(0).astype(np.float64)
    return rho * (np.abs(u).astype(np.float64) * c).sum(1) + RHO_B * float(np.abs(bias).max(initial=0.0))


def worst_ratio(u, E, bias, rho=RHO):
    d = np.abs(bf16_path(u, E, bias).astype(np.float64) - fp32_path(u, E, bias).astype(np.float64))
    return float((d / eps(u, E, bias, rho)[:, None]).max())


def test_bf16_rounding_matches_torch():
    x = np.random.default_rng(0).standard_normal(100_000).astype(F32) * 10.0 ** np.arange(-5, 5).repeat(10_000)
    assert np.array_equal(bf16(x), torch.from_numpy(x).to(torch.bfloat16).float().numpy())


def test_bound_random_and_adversarial():
    rng = np.random.default_rng(1)
    N = 1500
    E = (rng.standard_normal((N, 64)) * 0.02).astype(F32)
    u = rng.standard_normal((24, 64)).astype(F32)
    u[0, 7] = 300.0                                                    # one large coordinate
    u[1] = 1.0 + 2.0 ** -8 + 2.0 ** -22                                # rounds up by almost half a bf16 ulp
    E[5] = np.abs(E).max(0)                                            # a row at +c_i, and one at -c_i
    E[6] = -np.abs(E).max(0)
    E[7] = 0.02 * (1.0 + 2.0 ** -8 + 2.0 ** -22)                       # rounds up as well
    u[2] = np.sign(u[2]) * 3.0
    for bias in (np.zeros(N, F32), (rng.standard_normal(N) * 0.01).astype(F32),
                 (rng.standard_normal(N) * 5.0).astype(F32)):          # a bias that dominates the dot product
        r = worst_ratio(u, E, bias)
        assert r <= 1.0, r
    # trained-like: the table x 10
    assert worst_ratio(u, E * F32(10), np.zeros(N, F32)) <= 1.0


def test_half_the_bound_fails():
    # every operand 1 + 2^-8 + 2^-22 rounds up to 1 + 2^-7: each product grows by ~2 * 2^-8 relative
    v = F32(1.0 + 2.0 ** -8 + 2.0 ** -22)
    u = np.full((1, 64), v, F32)
    E = np.full((3, 64), v, F32)
    bias = np.zeros(3, F32)
    assert worst_ratio(u, E, bias) <= 1.0
    assert worst_ratio(u, E, bias, rho=RHO / 2) > 1.0
