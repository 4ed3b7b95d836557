"""CPU model of the fp32-bounded rejection test of the production kernels (remote_candidate in
mcpar_b200/csrc/mh_kernels.cuh): the same arithmetic in numpy float32, with every approximation the
kernel makes pushed to the edge of its documented error (the SFU Box-Muller error bound returned by
normal_pair_f32, 2-ulp exp2), against the exact fp64 value of
    R = sum_s Q_s(x') / max_s Q_s(x')      (src/mcpar.cc:355-398: pacpt = qimax / qisum = 1 / R).
The kernel decides from R32 (1 +- eps); that is sound iff the true R lies inside that interval whenever
the kernel's guards (max a > -9.7, theta < 2e-3) let the fast path decide.  The GPU-side check of the
same claim is tests/test_gpu_audit.py (bit-identical runs with the fp64 route forced)."""
import numpy as np
import pytest

L2E = 1.4426950408889634
f32 = np.float32


def _model(rng, M, D, ncand, mu_scale, sig_lo, sig_hi, worst):
    mu = rng.uniform(-mu_scale, mu_scale, (M, D))
    mu[: M // 2] = mu[0] + rng.normal(0, 0.3, (M // 2, D))            # a cluster of near-coincident components
    sig = np.exp(rng.uniform(np.log(sig_lo), np.log(sig_hi), (M, D)))
    # staging (stage_pool): fp32 copies and the pool-wide scalars, rounded up
    g = np.sqrt(L2E / (2.0 * sig * sig))
    gmu32, g32, s32, mu32 = f32(g * mu), f32(g), f32(sig), f32(mu)
    mu_max = np.nextafter(f32(np.abs(mu).max()), f32(np.inf))
    isig_max = np.nextafter(f32((1.0 / sig).max()), f32(np.inf))
    # candidates
    c = rng.integers(0, M, ncand)
    v = 1.0 - rng.random((ncand, D // 2))                              # (0, 1]
    if worst:
        v[: ncand // 4] = 1.0 - rng.random((ncand // 4, D // 2)) * 1e-5   # tiny radii, where the radius bound bites
    ang = 2.0 * np.pi * rng.random((ncand, D // 2))
    r = np.sqrt(-2.0 * np.log(v))
    z = np.empty((ncand, D)); z[:, 0::2] = r * np.sin(ang); z[:, 1::2] = r * np.cos(ang)
    x_true = mu[c] + sig[c] * z
    a_true = -0.5 * (((x_true[:, None, :] - mu[None]) / sig[None]) ** 2).sum(-1)       # [ncand][M]
    R_true = np.exp(a_true - a_true.max(1, keepdims=True)).sum(1)
    # the kernel's fp32 path, each approximate quantity at the edge of its bound
    r32 = f32(r)
    zerr = f32(2.4e-6) * r32 + f32(1.7e-6) * np.minimum(f32(1.0) / np.maximum(r32, f32(1e-30)), f32(770.0))
    zerr_pair = zerr.max(1)
    sgn = rng.choice([-1.0, 1.0], (ncand, D))
    zt = f32(z + sgn * np.repeat(zerr, 2, axis=1).astype(np.float64) * (0.999 if worst else 0.3))
    xf = (s32[c] * zt + mu32[c]).astype(f32)
    xabs = np.abs(xf).max(1)
    sgmax = s32[c].max(1)
    theta = (f32(1.9e-7) * (mu_max + xabs) + zerr_pair * sgmax) * isig_max
    ref = f32((np.log2(v)).sum(1) + rng.uniform(-1e-6, 1e-6, ncand) * (D // 2))          # sum of lg2.approx(v)
    y = (gmu32[None] - g32[None] * xf[:, None, :]).astype(f32)                            # fmaf(-g, x, g mu), two roundings here
    acc = (-ref)[:, None].astype(f32)
    for i in range(D):
        acc = (acc - y[:, :, i] * y[:, :, i]).astype(f32)
    mr = acc.max(1)
    ex = np.exp2(acc.astype(np.float64)) * (1.0 + rng.uniform(-2.4e-7, 2.4e-7, acc.shape))  # ex2.approx: 2 ulp
    S = f32(ex).sum(1, dtype=f32)
    E = f32(np.exp2(mr.astype(np.float64)) * (1.0 + 2.4e-7))
    R32 = S.astype(np.float64) / E.astype(np.float64)
    eps = (f32(1.01e-4) + f32(1.0e-5) * f32(D)) + f32(2.0e-5) * f32(M) + theta * f32(21.3 * np.sqrt(D))
    fast = (mr + ref > f32(-14.0)) & (theta < f32(2.0e-3))
    return R_true, R32, eps.astype(np.float64), fast, a_true.max(1)


@pytest.mark.parametrize("M,D,mu_scale,sig_lo,sig_hi", [
    (16, 2, 6.0, 0.5, 2.5),          # the benchmark's regime
    (16, 2, 6.0, 0.05, 3.0),         # widths spread over a factor 60
    (256, 2, 10.0, 0.2, 2.0),        # config 5's pool size
    (8, 4, 5.0, 0.3, 2.0),           # d = 4 (two normal pairs per candidate)
    (16, 2, 300.0, 0.5, 2.0),        # far from the origin: roundings of mu and x' dominate theta
])
@pytest.mark.parametrize("worst", [False, True])
def test_fast_path_interval_contains_the_true_ratio(M, D, mu_scale, sig_lo, sig_hi, worst):
    rng = np.random.default_rng(1234 + M + D)
    R_true, R32, eps, fast, amax = _model(rng, M, D, 200000, mu_scale, sig_lo, sig_hi, worst)
    assert fast.mean() > 0.2, "the case must exercise the fast path"
    rel = np.abs(R_true[fast] / R32[fast] - 1.0)
    worst_ratio = (rel / eps[fast]).max()
    assert worst_ratio < 1.0, "true R outside R32 (1 +- eps): %.3g of the bound" % worst_ratio
    # whenever the fast path decides, max_s Q_s(x') > exp(-10): the reference's FPEPS offsets (mcpar.cc:357-358)
    # then move pacpt by < 2.3e-10 relative, which the 3e-10 term of the kernel's test covers
    assert amax[fast].min() > -10.0


def test_accept_test_interval_contains_exp_delta():
    """accept_test (mh_kernels.cuh): u < exp(delta) cfac is decided from e32 = ex2.approx(fp32(delta) log2 e)
    with a margin of 1e-4 either way.  Model: fp32 rounding of delta and of the product, ex2.approx at 2 ulp;
    the true exp(delta) must lie inside e32 (1 +- 1e-4) over the clamped range |delta| <= 80."""
    rng = np.random.default_rng(5)
    delta = np.concatenate([rng.uniform(-80, 80, 400000), rng.normal(0, 3, 400000), -np.exp(rng.uniform(-20, 4.3, 200000))])
    delta = delta[np.abs(delta) <= 80.0]
    dc = f32(delta)
    arg = (dc * f32(L2E)).astype(f32)
    for sgn in (-1.0, 1.0):
        e32 = f32(np.exp2(arg.astype(np.float64)) * (1.0 + sgn * 2.4e-7))
        rel = np.abs(np.exp(delta) / e32.astype(np.float64) - 1.0)
        assert rel.max() < 1.0e-4, rel.max()
    assert rel.max() < 2.0e-5                      # the margin is five times what the model needs


# ---------------------------------------------------------------- remote mode 1: sum-mixture proposal
def _summix_model(rng, M, D, npts, mu_scale, sig_lo, sig_hi, far, chunks=None):
    """summix_bounds (mh_kernels.cuh; wide_summix_bounds of mh_wide.cuh is the same arithmetic spread over lanes) in numpy
    float32 against the exact fp64 q(x)/q(x'); returns the true ratio, the kernel's interval and which points the fast
    path decides.  The step from the two sums to the interval is summix_cfac_bounds (mh_kernels.cuh), which every kernel
    family calls.  chunks = DC models the cooperative kernel (mh_coop.cuh): the exponent of a slot is summed in DC
    parameter chunks (from 0, or from nb when DC = 1), the chunk totals are added to nb, and the picked component's total
    is subtracted afterwards; its bound uses the larger rounding terms cu = (24 + D) u, cn = 4.8e-7 nbmax + ..."""
    mu = rng.uniform(-mu_scale, mu_scale, (M, D))
    mu[: M // 2] = mu[0] + rng.normal(0, 0.3, (M // 2, D))
    sig = np.exp(rng.uniform(np.log(sig_lo), np.log(sig_hi), (M, D)))
    g = np.sqrt(L2E / (2.0 * sig * sig))
    nb = (-0.5 * np.log(sig * sig)).sum(1) * L2E
    gmu32, g32, nb32 = f32(g * mu), f32(g), f32(nb)
    mumax = np.nextafter(f32(np.abs(mu).max()), f32(np.inf))
    isig = np.nextafter(f32((1.0 / sig).max()), f32(np.inf))
    nbmax = np.nextafter(f32(np.abs(nb).max()), f32(np.inf))
    c = rng.integers(0, M, npts)
    xn = mu[c] + sig[c] * rng.standard_normal((npts, D))                       # x' ~ component c
    co = rng.integers(0, M, npts)
    xo = mu[co] + sig[co] * rng.standard_normal((npts, D)) * (4.0 if far else 1.2)   # the chain's state (far: in the tails)

    def lse_true(x):
        a = (-0.5 * np.log(sig * sig)).sum(1)[None] - 0.5 * (((x[:, None, :] - mu[None]) / sig[None]) ** 2).sum(-1)
        m = a.max(1)
        return m + np.log(np.exp(a - m[:, None]).sum(1))
    true = np.exp(lse_true(xo) - lse_true(xn))

    xof, xnf = f32(xo), f32(xn)

    def totals(xf):                                                                    # cooperative kernel: E[slot] per point
        dpc = D // chunks
        e = nb32[None].repeat(len(xf), 0).astype(f32) if chunks == 1 else np.zeros((len(xf), M), f32)
        parts = []
        for ch in range(chunks):
            acc = e if chunks == 1 else np.zeros((len(xf), M), f32)
            for i in range(ch * dpc, (ch + 1) * dpc):
                y = (gmu32[None, :, i] - g32[None, :, i] * xf[:, None, i]).astype(f32)
                acc = (acc - y * y).astype(f32)
            parts.append(acc)
        if chunks == 1:
            return parts[0]
        tot = nb32[None].repeat(len(xf), 0).astype(f32)
        for a in parts:
            tot = (tot + a).astype(f32)
        return tot

    if chunks:
        En_tot, Eo_tot = totals(xnf), totals(xof)
        ref = En_tot[np.arange(npts), c]
    else:
        ref = nb32[c].copy()
        for i in range(D):
            y = (gmu32[c, i] - g32[c, i] * xnf[:, i]).astype(f32)
            ref = (ref - y * y).astype(f32)

    def ssum(xf, sgn):
        if chunks:
            acc = ((En_tot if xf is xnf else Eo_tot) - ref[:, None]).astype(f32)
        else:
            acc = (nb32[None] - ref[:, None]).astype(f32)
            for i in range(D):
                y = (gmu32[None, :, i] - g32[None, :, i] * xf[:, None, i]).astype(f32)
                acc = (acc - y * y).astype(f32)
        ex = f32(np.exp2(acc.astype(np.float64)) * (1.0 + sgn * 2.4e-7))             # ex2.approx at the edge of its bound
        ex[ex < f32(1.1754944e-38)] = 0                                                # ftz
        part = [ex[:, q::4].sum(1, dtype=f32) for q in range(4)]                       # 4 partial sums + tree
        return ((part[0] + part[1]).astype(f32) + (part[2] + part[3]).astype(f32)).astype(f32)
    out = []
    for sgn_o, sgn_n in ((1.0, -1.0), (-1.0, 1.0)):
        so, sn = ssum(xof, sgn_o), ssum(xnf, sgn_n)
        ok = (sn < 1e30) & (so < 1e30) & (sn > 0.5)
        th_n = f32(1.6e-7) * (mumax + np.abs(xnf).max(1)) * isig
        th_o = f32(1.6e-7) * (mumax + np.abs(xof).max(1)) * isig
        lvl = nbmax - ref + f32(np.log2(M)) + f32(30.0)
        En = np.maximum(lvl - np.log2(np.maximum(sn, f32(1e-37))), 30.0)
        Eo = np.maximum(lvl - np.log2(np.maximum(so, f32(1e-37))), 30.0)
        cu, cn = (4.0 + D) * 6.0e-8, 2.4e-7 * nbmax + 1.0e-5 + 1.0e-8 * M
        if chunks:
            cu, cn = (24.0 + D) * 6.0e-8, 4.8e-7 * nbmax + 1.0e-5 + 1.0e-8 * M
        eps_n = 0.75 * (2.0 * th_n * np.sqrt(D * En) + cu * En + D * th_n * th_n) + cn
        eps_o = 0.75 * (2.0 * th_o * np.sqrt(D * Eo) + cu * Eo + D * th_o * th_o) + cn
        ok &= (th_n < 1e-3) & (th_o < 1e-3) & (eps_n < 0.02) & (eps_o < 0.02)
        lo = so * (1.0 - eps_o) / (sn * (1.0 + eps_n)) * (1.0 - 1.0e-6)
        hi = (so * (1.0 + eps_o) + 2.0e-38 * M) / (sn * (1.0 - eps_n)) * (1.0 + 1.0e-6)
        out.append((lo.astype(np.float64), hi.astype(np.float64), ok))
    return true, out


@pytest.mark.parametrize("M,D,mu_scale,sig_lo,sig_hi", [
    (16, 2, 6.0, 0.5, 2.5),          # the benchmark's regime
    (256, 2, 6.0, 0.5, 2.5),         # the blueprint's pool size (configs 4 and 5)
    (16, 2, 6.0, 0.05, 3.0),         # widths spread over a factor 60: normalisations differ by 2^12
    (64, 4, 5.0, 0.3, 2.0),
    (16, 2, 300.0, 0.5, 2.0),        # far from the origin: roundings of mu and x dominate theta
])
@pytest.mark.parametrize("far", [False, True])
def test_summix_interval_contains_the_true_hastings_factor(M, D, mu_scale, sig_lo, sig_hi, far):
    rng = np.random.default_rng(77 + M + D)
    true, runs = _summix_model(rng, M, D, 60000, mu_scale, sig_lo, sig_hi, far)
    for lo, hi, ok in runs:
        assert ok.mean() > 0.5, "the case must exercise the fast path"
        inside = (true[ok] >= lo[ok]) & (true[ok] <= hi[ok])
        assert inside.all(), "q(x)/q(x') outside the kernel's interval for %d points" % (~inside).sum()
        width = (hi[ok] / np.maximum(lo[ok], 1e-300))
        # and the interval is tight: ~3e-4 of the uniforms fall inside it in the benchmark's regime (narrow
        # components or a far origin widen it through theta, still within 2 %)
        assert np.median(width) < (1.0004 if (mu_scale == 6.0 and sig_lo == 0.5) else 1.02)


@pytest.mark.parametrize("M,D,chunks,mu_scale,sig_lo,sig_hi", [
    (16, 16, None, 3.0, 0.4, 1.5),   # wide kernel, config 3's dimension
    (40, 64, None, 5.0, 0.6, 1.5),   # wide kernel at d = 64
    (40, 64, 4, 5.0, 0.6, 1.5),      # cooperative kernel: 64 slots side by side, 4 parameter chunks
    (256, 64, 1, 5.0, 0.6, 1.5),     # cooperative kernel at the blueprint's M = 256: one chunk, sums start at nb
    (256, 64, 1, 40.0, 0.7, 1.4),    # means far from the origin
])
@pytest.mark.parametrize("far", [False, True])
def test_summix_interval_wide_and_cooperative_kernels(M, D, chunks, mu_scale, sig_lo, sig_hi, far):
    rng = np.random.default_rng(91 + M + D + (chunks or 0))
    true, runs = _summix_model(rng, M, D, 3000 if D == 64 else 20000, mu_scale, sig_lo, sig_hi, far, chunks=chunks)
    for lo, hi, ok in runs:
        assert ok.mean() > 0.5, "the case must exercise the fast path"
        inside = (true[ok] >= lo[ok]) & (true[ok] <= hi[ok])
        assert inside.all(), "q(x)/q(x') outside the kernel's interval for %d points" % (~inside).sum()
        if not far:                                  # (far: q(x) underflows in fp32 at d >= 16 -- the lower bound is 0, the interval still holds the truth)
            assert np.median(hi[ok] / np.maximum(lo[ok], 1e-300)) < 1.02
