"""Kernel-level parity: every C-ABI entry point vs the CPU oracle / the
reference-generated goldens, through the ctypes binding (estorch_b200.backend).

Tolerances: integer outputs (offsets, order, ranks) bit-exact; materialised
rows bit-exact (same two fp32 roundings as the reference); fp32 reductions
within 1e-5 max-norm relative (SURVEY App. A.5: max|a-b| <= 1e-5 * max|b|).
"""
import numpy as np
import pytest
import torch

from oracle import es_oracle as orc
from conftest import load_golden, rel_err, seeded_theta

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def be():
    from estorch_b200.backend import CudaBackend
    return CudaBackend(torch.device("cuda", 0))


def dev(be, a, dtype=None):
    t = torch.from_numpy(np.ascontiguousarray(a))
    if dtype is not None:
        t = t.to(dtype)
    return t.to(be.device)


# ------------------------------------------------------------------ noise
def test_fill_noise_table_matches_oracle(be):
    n = 1 << 16
    t = be.alloc(n)
    be.fill_noise_table(t, 42)
    got = t.cpu().numpy()
    want = orc.philox_normal_table(n, 42)
    # every entry is fp16-representable (so that the 16-bit copy of the table is exact) ...
    np.testing.assert_array_equal(got, got.astype(np.float16).astype(np.float32))
    # ... and equals the oracle's Philox + Box-Muller value rounded to fp16; fp32 log/sincos differ
    # by ulps between libm and the device, which can move an entry across an fp16 rounding boundary:
    # at most one fp16 ulp (2^-8 for |z| < 8), and rarely
    diff = np.abs(got - want)
    assert diff.max() <= 2.0 ** -8 and np.count_nonzero(diff) < n // 50
    big = be.alloc(1 << 24)
    be.fill_noise_table(big, (7 << 32) | 9)
    assert abs(float(big.mean())) < 2e-3 and abs(float(big.std()) - 1.0) < 2e-3
    assert torch.isfinite(big).all()
    d2 = np.abs(big[:4096].cpu().numpy() - orc.philox_normal_table(4096, (7 << 32) | 9))
    assert d2.max() <= 2.0 ** -8 and np.count_nonzero(d2) < 4096 // 50


@pytest.mark.parametrize("pairs,n,table_len,pair_begin,gen", [
    (32, 4610, 1 << 15, 0, 0), (2048, 4610, 1 << 20, 0, 3), (512, 1001760, 1 << 22, 1024, 17),
    (5, 7, 64, 0, 1), (8192, 6020, 1 << 24, 8192, 2), (4096, 4610, 1 << 21, 0, 5), (3000, 31, 4096, 0, 2),
    (1, 100, 1 << 12, 0, 0), (256, 1001760, 1 << 28, 1792, 9)])
def test_make_offsets_bit_exact(be, pairs, n, table_len, pair_begin, gen):
    from estorch_b200.backend import new_state, write_state
    offs = be.alloc(pairs, dtype=torch.int64)
    order = be.alloc(pairs, dtype=torch.int32)
    be.make_offsets(0xDEADBEEF12345, None, gen, pair_begin, pairs, table_len, n, offs, order)
    want = orc.noise_offsets(0xDEADBEEF12345, gen, pair_begin, pairs, table_len, n)
    np.testing.assert_array_equal(offs.cpu().numpy(), want)
    np.testing.assert_array_equal(order.cpu().numpy(), np.argsort(want, kind="stable").astype(np.int32))
    # generation = device-resident counter + host offset (what a CUDA-graph replay uses)
    st = new_state(be.device)
    offs2 = be.alloc(pairs, dtype=torch.int64)
    for dev_gen, host_off in ((gen, 0), (max(gen - 1, 0), gen - max(gen - 1, 0))):
        write_state(st, generation=dev_gen)
        be.make_offsets(0xDEADBEEF12345, st, host_off, pair_begin, pairs, table_len, n, offs2, None)
        np.testing.assert_array_equal(offs2.cpu().numpy(), want)


def test_perturb_rows_bit_exact(be):
    g = load_golden("es_cartpole_p64.npz")
    theta, table, offs = g["theta0"], g["table"], g["offsets"][0]
    P, n = 64, theta.size
    rows = be.alloc(P, n)
    eps = be.alloc(P, n)
    be.perturb_rows(dev(be, theta), dev(be, table), dev(be, offs), P // 2, 0.1, 0, P, rows, eps)
    pop, epsilon = orc.sample_population(theta, table, offs, 0.1)
    np.testing.assert_array_equal(rows.cpu().numpy(), pop)
    np.testing.assert_array_equal(eps.cpu().numpy(), epsilon)
    part = be.alloc(5, n)
    be.perturb_rows(dev(be, theta), dev(be, table), dev(be, offs), P // 2, 0.1, 30, 5, part, None)
    np.testing.assert_array_equal(part.cpu().numpy(), pop[30:35])


# ------------------------------------------------------------------ evaluate
def _eval(be, dims, theta, table, offs, sigma, obs, tgt, order=None, bc_obs=0, bc_dim=0):
    pairs = len(offs)
    ret = be.zeros(2 * pairs)
    bcp = be.zeros(pairs, bc_dim) if bc_dim else None
    bcm = be.zeros(pairs, bc_dim) if bc_dim else None
    be.eval_mlp(dims, dev(be, theta), dev(be, table), dev(be, offs),
                None if order is None else dev(be, order), pairs, sigma, dev(be, obs), dev(be, tgt),
                ret[:pairs], ret[pairs:], bcp, bcm, bc_obs, bc_dim)
    torch.cuda.synchronize()
    bcs = None if not bc_dim else np.concatenate([bcp.cpu().numpy(), bcm.cpu().numpy()])
    return ret.cpu().numpy(), bcs


def test_eval_mlp_matches_reference_golden(be):
    g = load_golden("es_cartpole_p64.npz")
    dims = [int(d) for d in g["dims"]]
    for gen in range(3):
        ret, _ = _eval(be, dims, g["theta_before"][gen], g["table"], g["offsets"][gen], 0.1,
                       g["obs"], g["target"])
        ref = g["returns"][gen][:, 0]          # produced by the unmodified reference
        assert rel_err(ret, ref) < 2e-6
    # evaluation order must not change results
    order = np.argsort(g["offsets"][0], kind="stable").astype(np.int32)
    ret2, _ = _eval(be, dims, g["theta_before"][0], g["table"], g["offsets"][0], 0.1,
                    g["obs"], g["target"], order=order)
    ret1, _ = _eval(be, dims, g["theta_before"][0], g["table"], g["offsets"][0], 0.1,
                    g["obs"], g["target"])
    np.testing.assert_array_equal(ret1, ret2)


def test_eval_mlp_tiny_and_ragged(be):
    g = load_golden("es_tiny_p8.npz")
    dims = [int(d) for d in g["dims"]]
    ret, _ = _eval(be, dims, g["theta_before"][0], g["table"], g["offsets"][0], 0.05,
                   g["obs"], g["target"])                       # B = 5: ragged chunk
    assert rel_err(ret, g["returns"][0][:, 0]) < 2e-6


def test_eval_mlp_bc_matches_reference_golden(be):
    g = load_golden("nsra_bipedal_p32.npz")
    dims = [int(d) for d in g["dims"]]
    theta, offs = g["theta_before"][0], g["offsets"][0]
    ret, bcs = _eval(be, dims, theta, g["table"], offs, 0.02, g["obs"], g["target"],
                     bc_obs=int(g["bc_obs"]), bc_dim=int(g["bc_dim"]))
    assert rel_err(ret, g["returns"][0][:, 0]) < 2e-6
    pop, _ = orc.sample_population(theta, g["table"], offs, 0.02)
    _, want_bc = orc.evaluate_population(pop, dims, g["obs"], g["target"], 64, 256)
    assert rel_err(bcs, want_bc) < 2e-6


@pytest.mark.parametrize("dims,B,pairs", [([128, 512, 512, 288], 48, 4), ([17, 33, 5], 100, 6),
                                          ([4, 2], 1, 3), ([9, 130, 70, 70, 3], 256, 3)])
def test_eval_mlp_shapes_vs_oracle(be, dims, B, pairs):
    rng = np.random.RandomState(1)
    n = orc.mlp_param_count(dims)
    table_len = max(1 << 14, (n + 31) // 32 * 32 + 4096)
    table = rng.standard_normal(table_len).astype(np.float32)
    theta = (rng.standard_normal(n) * 0.1).astype(np.float32)
    obs = rng.standard_normal((B, dims[0])).astype(np.float32)
    tgt = rng.standard_normal((B, dims[-1])).astype(np.float32)
    offs = orc.noise_offsets(5, 0, 0, pairs, table_len, n)
    ret, _ = _eval(be, dims, theta, table, offs, 0.02, obs, tgt)
    pop, _ = orc.sample_population(theta, table, offs, 0.02)
    want, _ = orc.evaluate_population(pop, dims, obs, tgt)
    assert rel_err(ret, want) < 5e-6
    one = be.zeros(1)
    be.eval_mlp_center(dims, dev(be, theta), dev(be, obs), dev(be, tgt), one)
    assert abs(float(one) - float(orc.synthetic_return(orc.mlp_forward(theta, dims, obs), tgt))) \
        < 5e-6 * abs(float(one)) + 1e-7


# ------------------------------------------------------------------ rank + grad + Adam
def _rank_grad_adam(be, returns, table, offs, theta, m, v, step, novelty=None, w=(1.0, 0.0),
                    order=None, lr=0.01):
    from estorch_b200.backend import new_state, write_state, read_state, adam_desc
    P, n = returns.size, theta.size
    st = new_state(be.device)
    write_state(st, adam_step=step)
    th, mm, vv = dev(be, theta), dev(be, m), dev(be, v)
    ranks = be.zeros(P, dtype=torch.int32)
    ranks2 = be.zeros(P, dtype=torch.int32) if novelty is not None else None
    grad = be.zeros(n)
    be.rank_grad_adam(dev(be, returns), None if novelty is None else dev(be, novelty), w[0], w[1], P,
                      dev(be, table), dev(be, offs), None if order is None else dev(be, order),
                      th, mm, vv, st, adam_desc(lr=lr), ranks, ranks2, grad)
    torch.cuda.synchronize()
    assert read_state(st)["adam_step"] == step + 1
    return dict(ranks=ranks.cpu().numpy(), ranks2=None if ranks2 is None else ranks2.cpu().numpy(),
                grad=grad.cpu().numpy(), theta=th.cpu().numpy(), m=mm.cpu().numpy(), v=vv.cpu().numpy())


@pytest.mark.parametrize("name", ["es_tiny_p8.npz", "es_cartpole_p64.npz"])
def test_rank_grad_adam_matches_reference_golden(be, name):
    g = load_golden(name)
    n = g["theta0"].size
    theta, m, v = g["theta0"].copy(), np.zeros(n, np.float32), np.zeros(n, np.float32)
    for gen in range(len(g["grad"])):
        ret = np.ascontiguousarray(g["returns"][gen][:, 0])     # the reference's return bits
        out = _rank_grad_adam(be, ret, g["table"], g["offsets"][gen], theta, m, v, gen)
        np.testing.assert_array_equal(out["ranks"], orc.compute_ranks(ret))       # bit-exact
        assert rel_err(out["grad"], g["grad"][gen]) < 1e-5
        ok = np.abs(g["grad"][gen]) > 1e-4 * np.abs(g["grad"][gen]).max()      # see DESIGN.md (Adam at g~0)
        assert rel_err(out["theta"][ok], g["theta_after"][gen][ok]) < 1e-5
        assert np.abs(out["theta"] - g["theta_after"][gen]).max() <= 0.02
        # Adam alone (identical gradient bits through clamp_adam) is exact to 1e-6
        from estorch_b200.backend import new_state, write_state, adam_desc
        st = new_state(be.device); write_state(st, adam_step=gen)
        th, mm, vv = dev(be, theta), dev(be, m), dev(be, v)
        be.clamp_adam(dev(be, g["grad"][gen] * np.float32(len(ret))), len(ret), th, mm, vv, st,
                      adam_desc(lr=0.01))
        assert rel_err(th.cpu().numpy(), g["theta_after"][gen]) < 1e-6
        theta, m, v = th.cpu().numpy(), mm.cpu().numpy(), vv.cpu().numpy()
    assert rel_err(m, g["m_final"]) < 1e-5 and rel_err(v, g["v_final"]) < 1e-5


@pytest.mark.parametrize("algo,w", [("ns", (0.0, 1.0)), ("nsr", (0.5, 0.5)), ("nsra", None)])
def test_rank_grad_ns_blends_match_reference_golden(be, algo, w):
    g = load_golden(f"{algo}_bipedal_p32.npz")
    n = g["meta_theta0"].shape[1]
    for gen in range(len(g["grad"])):
        ret = g["returns"][gen]
        if algo == "nsra":
            wt = float(g["weight"][gen - 1]) if gen > 0 else 1.0   # weight in force during this generation
            ww = (np.float32(wt), np.float32(1.0 - wt))
        else:
            ww = w
        out = _rank_grad_adam(be, np.ascontiguousarray(ret[:, 0]), g["table"], g["offsets"][gen],
                              g["theta_before"][gen], np.zeros(n, np.float32), np.zeros(n, np.float32),
                              0, novelty=np.ascontiguousarray(ret[:, 1]), w=ww)
        np.testing.assert_array_equal(out["ranks"], orc.compute_ranks(ret[:, 0]))
        np.testing.assert_array_equal(out["ranks2"], orc.compute_ranks(ret[:, 1]))
        assert rel_err(out["grad"], g["grad"][gen]) < 1e-5


@pytest.mark.parametrize("n,P", [(7, 8), (4610, 4096), (400003, 64), (1001760, 32)])
def test_rank_grad_adam_sizes_vs_oracle(be, n, P):
    rng = np.random.RandomState(n)
    table_len = (n + 31) // 32 * 32 + (1 << 16)
    table = rng.standard_normal(table_len).astype(np.float32)
    offs = orc.noise_offsets(3, 1, 0, P // 2, table_len, n)
    ret = rng.standard_normal(P).astype(np.float32)
    assert len(np.unique(ret)) == P
    theta = (rng.standard_normal(n) * 0.1).astype(np.float32)
    m = (rng.standard_normal(n) * 0.01).astype(np.float32)
    v = (rng.random(n) * 1e-3).astype(np.float32)
    order = np.argsort(offs, kind="stable").astype(np.int32)
    out = _rank_grad_adam(be, ret, table, offs, theta, m, v, 5, order=order)
    np.testing.assert_array_equal(out["ranks"], orc.compute_ranks(ret))
    want = orc.calculate_grad_pairs(ret, table, offs, n)
    assert rel_err(out["grad"], want) < 1e-5
    th, mm, vv = orc.adam_step(theta, m, v, orc.negate_clamp(out["grad"]), 6)
    assert rel_err(out["theta"], th) < 1e-6 and rel_err(out["m"], mm) < 1e-6 and rel_err(out["v"], vv) < 1e-6
    # same result without the sorted order (summation order changes: 1e-6)
    out2 = _rank_grad_adam(be, ret, table, offs, theta, m, v, 5)
    assert rel_err(out2["grad"], out["grad"]) < 2e-6


def test_rank_ties_stable_by_index(be):
    ret = np.array([1.0, 0.0, 1.0, 0.0, 2.0, 2.0, -1.0, 0.0], dtype=np.float32)
    table = np.random.RandomState(0).standard_normal(4096).astype(np.float32)
    offs = orc.noise_offsets(1, 0, 0, 4, 4096, 16)
    out = _rank_grad_adam(be, ret, table, offs, np.zeros(16, np.float32), np.zeros(16, np.float32),
                          np.zeros(16, np.float32), 0)
    np.testing.assert_array_equal(out["ranks"], orc.compute_ranks(ret))


@pytest.mark.parametrize("n,P,W", [(1001760, 512, 4), (6020, 256, 2), (4610, 64, 1)])
def test_rank_grad_fp16_table_and_rank_major_layout(be, n, P, W):
    """estk_rank_grad[_adam]_h stream the EXACT fp16 copy of the table: same ranks, and the same gradient /
    theta as the fp32-table entry points (bit-identical when both take the column-split path, i.e. large n;
    a different pair split for small n only changes the fp32 summation order).  With world = W the returns
    arrive rank-major [W][2][pairs/W] (what the in-place all-gather produces): ranks_out stays in member order."""
    from estorch_b200.backend import new_state, adam_desc
    rng = np.random.RandomState(5)
    table_len = (n + 31) // 32 * 32 + (1 << 16)
    table = orc.round_f16(rng.standard_normal(table_len).astype(np.float32))
    offs = orc.noise_offsets(3, 1, 0, P // 2, table_len, n)
    order = np.argsort(offs, kind="stable").astype(np.int32)
    ret = rng.standard_normal(P).astype(np.float32)
    ret[5] = ret[P // 2 + 7]                                   # a tie: broken by member index in every layout
    theta = (rng.standard_normal(n) * 0.1).astype(np.float32)
    tb = dev(be, table)
    tb16 = be.alloc(table_len, dtype=torch.float16)
    assert be.shadow_f16(tb, tb16) == 0
    res = {}
    for name, t in (("fp32", tb), ("fp16", tb16)):
        th, mm, vv = dev(be, theta), be.zeros(n), be.zeros(n)
        ranks, g = be.zeros(P, dtype=torch.int32), be.zeros(n)
        be.rank_grad_adam(dev(be, ret), None, 1.0, 0.0, P, t, dev(be, offs), dev(be, order), th, mm, vv,
                          new_state(be.device), adam_desc(lr=0.01), ranks, None, g)
        res[name] = (ranks.cpu().numpy(), g.cpu().numpy(), th.cpu().numpy())
    np.testing.assert_array_equal(res["fp16"][0], res["fp32"][0])
    np.testing.assert_array_equal(res["fp16"][0], orc.compute_ranks(ret))
    if n > 500000:
        np.testing.assert_array_equal(res["fp16"][1], res["fp32"][1])
        np.testing.assert_array_equal(res["fp16"][2], res["fp32"][2])
    else:
        assert rel_err(res["fp16"][1], res["fp32"][1]) < 2e-6
    # sharded + rank-major: sum of the shards' raw partial sums / P == the fused gradient
    pairs, pl = P // 2, P // 2 // W
    rm = np.empty((W, 2, pl), np.float32)
    for r in range(W):
        rm[r, 0], rm[r, 1] = ret[r * pl:(r + 1) * pl], ret[pairs + r * pl: pairs + (r + 1) * pl]
    total = be.zeros(n)
    for r in range(W):
        part, ranks = be.zeros(n), be.zeros(P, dtype=torch.int32)
        so = offs[r * pl:(r + 1) * pl]
        be.rank_grad(dev(be, rm.reshape(-1)), None, 1.0, 0.0, P, tb16, dev(be, so),
                     dev(be, np.argsort(so, kind="stable").astype(np.int32)), r * pl, pl, n, part, ranks, None, world=W)
        np.testing.assert_array_equal(ranks.cpu().numpy(), res["fp32"][0])
        total += part
    assert rel_err((total / P).cpu().numpy(), res["fp32"][1]) < 2e-6


def test_rank_nan_returns_sort_last(be):
    """A non-finite return (a diverged member) ranks like numpy's argsort ranks it (estorch.py:25): NaN last,
    NaNs among themselves by member index; -inf / +inf at the ends."""
    ret = np.array([0.5, np.nan, -1.0, np.inf, np.nan, -np.inf, 0.25, 0.5], dtype=np.float32)
    table = np.random.RandomState(0).standard_normal(4096).astype(np.float32)
    offs = orc.noise_offsets(1, 0, 0, 4, 4096, 16)
    out = _rank_grad_adam(be, ret, table, offs, np.zeros(16, np.float32), np.zeros(16, np.float32),
                          np.zeros(16, np.float32), 0)
    want = np.empty(8, dtype=np.int64)
    want[np.argsort(ret, kind="stable")] = np.arange(8)
    np.testing.assert_array_equal(out["ranks"], want)
    assert want[1] == 6 and want[4] == 7 and want[5] == 0 and want[3] == 5


def test_sharded_rank_grad_equals_fused(be):
    """Multi-GPU form on one GPU: sum of per-shard raw partials -> clamp_adam
    equals the fused kernel (this is what the NCCL all-reduce computes)."""
    from estorch_b200.backend import new_state, write_state, adam_desc
    rng = np.random.RandomState(9)
    n, P, W = 6020, 256, 4
    table_len = 1 << 16
    table = rng.standard_normal(table_len).astype(np.float32)
    offs = orc.noise_offsets(3, 2, 0, P // 2, table_len, n)
    ret = rng.standard_normal(P).astype(np.float32)
    theta = (rng.standard_normal(n) * 0.1).astype(np.float32)
    zeros = np.zeros(n, np.float32)
    fused = _rank_grad_adam(be, ret, table, offs, theta, zeros, zeros, 0)
    pl = P // 2 // W
    total = be.zeros(n)
    for r in range(W):
        part = be.zeros(n)
        ranks = be.zeros(P, dtype=torch.int32)
        be.rank_grad(dev(be, ret), None, 1.0, 0.0, P, dev(be, table), dev(be, offs[r * pl:(r + 1) * pl]),
                     None, r * pl, pl, n, part, ranks)
        total += part
        np.testing.assert_array_equal(ranks.cpu().numpy(), fused["ranks"])
    st = new_state(be.device)
    th, mm, vv = dev(be, theta), dev(be, zeros), dev(be, zeros)
    gout = be.zeros(n)
    be.clamp_adam(total, P, th, mm, vv, st, adam_desc(lr=0.01), gout)
    assert rel_err(gout.cpu().numpy(), fused["grad"]) < 2e-6
    ok = np.abs(fused["grad"]) > 1e-4 * np.abs(fused["grad"]).max()
    assert rel_err(th.cpu().numpy()[ok], fused["theta"][ok]) < 1e-5
    # gradient-only epilogue (non-Adam optimizers): clamp(-g)
    gonly = be.zeros(n)
    be.clamp_adam(total, P, None, None, None, None, adam_desc(), gonly)
    np.testing.assert_allclose(gonly.cpu().numpy(), orc.negate_clamp(gout.cpu().numpy()), rtol=0, atol=0)


def test_full_size_north_star_gradient_property(be):
    """P=4096, n=1,001,760 (BASELINE north star): the kernel's gradient equals an
    independent on-device evaluation of sum_j w_j T[off_j:off_j+n] (torch fp64
    gather-matmul in chunks), and negating the returns negates the gradient."""
    from estorch_b200.backend import new_state, adam_desc
    n, P = 1001760, 4096
    pairs = P // 2
    table_len = 1 << 26
    table = be.alloc(table_len)
    be.fill_noise_table(table, 42)
    offs = be.alloc(pairs, dtype=torch.int64)
    order = be.alloc(pairs, dtype=torch.int32)
    be.make_offsets(42, None, 0, 0, pairs, table_len, n, offs, order)
    gen = torch.Generator(device="cpu").manual_seed(0)
    ret = torch.randn(P, generator=gen).to(be.device)
    assert ret.unique().numel() == P
    zeros = lambda: be.zeros(n)
    out = {}
    for sign in (1.0, -1.0):
        th, m, v, g = zeros(), zeros(), zeros(), zeros()
        ranks = be.zeros(P, dtype=torch.int32)
        be.rank_grad_adam((ret * sign).contiguous(), None, 1.0, 0.0, P, table, offs, order, th, m, v,
                          new_state(be.device), adam_desc(lr=0.01), ranks, None, g)
        out[sign] = (g, ranks, th)
    g, ranks, th = out[1.0]
    want_ranks = torch.empty(P, dtype=torch.int64, device=be.device)
    want_ranks[torch.argsort(ret, stable=True)] = torch.arange(P, device=be.device)
    assert torch.equal(ranks.long(), want_ranks)
    c = (want_ranks.double() / (P - 1) - 0.5).float()
    w = (c[:pairs] - c[pairs:]).double()
    acc = torch.zeros(n, dtype=torch.float64, device=be.device)
    idx = torch.arange(n, device=be.device)
    for j0 in range(0, pairs, 64):
        rows = table[(offs[j0:j0 + 64, None] + idx[None, :])].double()
        acc += w[j0:j0 + 64] @ rows
    want = (acc / P).float()
    assert float((g - want).abs().max() / want.abs().max()) < 1e-5
    assert float((out[-1.0][0] + g).abs().max() / g.abs().max()) < 1e-6
    # first Adam step from zero state moves every parameter by ~lr*sign(-g)
    # (|g| >> Adam eps=1e-8, so m/(sqrt(v)+eps) is +-1 to 1e-4)
    ok = g.abs() > 1e-2 * g.abs().max()
    assert float((th[ok] + 0.01 * torch.sign(-g[ok])).abs().max()) < 1e-5


# ------------------------------------------------------------------ misc
def test_knn_novelty_matches_oracle(be):
    rng = np.random.RandomState(2)
    for A, k in ((3, 10), (40, 10), (200, 5)):
        arch = rng.standard_normal((A, 256)).astype(np.float32)
        bc = rng.standard_normal((33, 256)).astype(np.float32)
        out = be.zeros(33)
        be.knn_novelty(dev(be, bc), dev(be, arch), k, out)
        want = np.array([orc.novelty(bc[i], arch, k) for i in range(33)], dtype=np.float32)
        assert rel_err(out.cpu().numpy(), want) < 1e-6


def test_track_best(be):
    from estorch_b200.backend import new_state, read_state
    st = new_state(be.device)
    theta, best = be.zeros(1000), be.zeros(1000)
    for step, (r, improves) in enumerate([(-3.0, True), (-5.0, False), (-1.0, True)]):
        theta.fill_(float(step + 1))
        be.track_best(st, torch.tensor([r], device=be.device), theta, best)
        s = read_state(st)
        assert s["generation"] == step + 1 and s["improved"] == int(improves)
        assert s["episode_reward"] == r
    assert read_state(st)["best_reward"] == -1.0
    assert float(best.min()) == 3.0 and float(best.max()) == 3.0


# ------------------------------------------------------------------ tcgen05 evaluate (bf16 operands)
@pytest.mark.parametrize("dims,B,pairs,bc", [([128, 512, 512, 288], 256, 5, 0), ([64, 64, 32], 256, 3, 0),
                                             ([128, 512, 512, 512, 512, 288], 256, 3, 0),
                                             ([64, 256, 64], 512, 4, 256), ([192, 320, 96], 256, 2, 0)])
def test_eval_mlp_bf16_tensor_core_path(be, dims, B, pairs, bc):
    """bf16-operand / fp32-accumulate tcgen05 path: within 5e-4 (max-norm relative) of the
    oracle that emulates its roundings, and within 2e-2 of the exact fp32 forward."""
    rng = np.random.RandomState(7)
    n = orc.mlp_param_count(dims)
    assert be.eval_supports_bf16(dims, B)
    table_len = (n + 31) // 32 * 32 + (1 << 14)
    table = rng.standard_normal(table_len).astype(np.float32)
    theta = np.concatenate([np.concatenate([(rng.uniform(-1, 1, dims[i] * dims[i + 1]) / np.sqrt(dims[i])),
                                            rng.uniform(-1, 1, dims[i + 1]) / np.sqrt(dims[i])])
                            for i in range(len(dims) - 1)]).astype(np.float32)
    obs = rng.standard_normal((B, dims[0])).astype(np.float32)
    tgt = rng.standard_normal((B, dims[-1])).astype(np.float32)
    offs = orc.noise_offsets(11, 0, 0, pairs, table_len, n)
    order = np.argsort(offs, kind="stable").astype(np.int32)
    ret = be.zeros(2 * pairs)
    bcp = be.zeros(pairs, bc) if bc else None
    bcm = be.zeros(pairs, bc) if bc else None
    be.eval_mlp(dims, dev(be, theta), dev(be, table), dev(be, offs), dev(be, order), pairs, 0.02, dev(be, obs),
                dev(be, tgt), ret[:pairs], ret[pairs:], bcp, bcm, 64 if bc else 0, bc, precision="bf16")
    torch.cuda.synchronize()
    got = ret.cpu().numpy()
    pop, _ = orc.sample_population(theta, table, offs, 0.02)
    outs = [orc.mlp_forward_bf16(pop[i], dims, obs) for i in range(2 * pairs)]
    emu = np.array([orc.synthetic_return(o, tgt) for o in outs], dtype=np.float32)
    exact, _ = orc.evaluate_population(pop, dims, obs, tgt)
    assert rel_err(got, emu) < 5e-4
    assert rel_err(got, exact) < 2e-2
    if bc:
        want_bc = np.stack([orc.synthetic_bc(o, 64, bc) for o in outs])
        got_bc = np.concatenate([bcp.cpu().numpy(), bcm.cpu().numpy()])
        assert np.max(np.abs(got_bc - want_bc)) < 5e-3 * np.max(np.abs(want_bc))
    one = be.zeros(1)
    be.eval_mlp_center(dims, dev(be, theta), dev(be, obs), dev(be, tgt), one, precision="bf16")
    want = float(orc.synthetic_return(orc.mlp_forward_bf16(theta, dims, obs), tgt))
    assert abs(float(one) - want) < 5e-4 * abs(want)
    # unsupported shapes are refused, not silently rerouted
    with pytest.raises(RuntimeError, match="not supported"):
        be.eval_mlp([4, 64, 2], dev(be, theta[:450]), dev(be, table), dev(be, offs), None, pairs, 0.02,
                    dev(be, obs[:, :4].copy()), dev(be, tgt[:, :2].copy()), ret[:pairs], ret[pairs:], precision="bf16")


@pytest.mark.parametrize("dims,B,pairs", [([128, 512, 512, 288], 256, 4), ([64, 256, 64], 512, 3),
                                          ([128, 512, 512, 512, 512, 288], 256, 2)])
def test_eval_mlp_bf16s_shadow_sources(be, dims, B, pairs):
    """"bf16s": producers read bf16 shadows of theta / table.  Within 5e-4 of the oracle
    that emulates exactly those roundings, within 3e-2 of the exact fp32 forward."""
    rng = np.random.RandomState(17)
    n = orc.mlp_param_count(dims)
    table_len = (n + 31) // 32 * 32 + (1 << 14)
    table = rng.standard_normal(table_len).astype(np.float32)
    theta = np.concatenate([np.concatenate([(rng.uniform(-1, 1, dims[i] * dims[i + 1]) / np.sqrt(dims[i])),
                                            rng.uniform(-1, 1, dims[i + 1]) / np.sqrt(dims[i])])
                            for i in range(len(dims) - 1)]).astype(np.float32)
    obs = rng.standard_normal((B, dims[0])).astype(np.float32)
    tgt = rng.standard_normal((B, dims[-1])).astype(np.float32)
    offs = orc.noise_offsets(11, 0, 0, pairs, table_len, n)
    th, tb = dev(be, theta), dev(be, table)
    th16 = be.alloc(n, dtype=torch.bfloat16)
    tb16 = be.alloc(table_len, dtype=torch.bfloat16)
    be.shadow_bf16(th, th16)
    be.shadow_bf16(tb, tb16)
    np.testing.assert_array_equal(th16.float().cpu().numpy(), orc.round_bf16(theta))   # cvt.rn == RNE
    ret = be.zeros(2 * pairs)
    be.eval_mlp(dims, th, tb, dev(be, offs), None, pairs, 0.02, dev(be, obs), dev(be, tgt),
                ret[:pairs], ret[pairs:], precision="bf16s", theta16=th16, table16=tb16)
    got = ret.cpu().numpy()
    exact_rows, _ = orc.sample_population(theta, table, offs, 0.02)
    rows = orc.sample_population_bf16s(theta, table, offs, 0.02)
    idx = 0
    for i in range(len(dims) - 1):                      # biases are formed from the fp32 sources
        idx += dims[i] * dims[i + 1]
        rows[:, idx: idx + dims[i + 1]] = exact_rows[:, idx: idx + dims[i + 1]]
        idx += dims[i + 1]
    emu = np.array([orc.synthetic_return(orc.mlp_forward_bf16(r, dims, obs), tgt) for r in rows], dtype=np.float32)
    exact, _ = orc.evaluate_population(exact_rows, dims, obs, tgt)
    assert rel_err(got, emu) < 5e-4
    assert rel_err(got, exact) < 3e-2
    one = be.zeros(1)
    be.eval_mlp_center(dims, th, dev(be, obs), dev(be, tgt), one, precision="bf16s", theta16=th16)
    crow = orc.round_bf16(theta).copy()
    idx = 0
    for i in range(len(dims) - 1):
        idx += dims[i] * dims[i + 1]
        crow[idx: idx + dims[i + 1]] = theta[idx: idx + dims[i + 1]]
        idx += dims[i + 1]
    want = float(orc.synthetic_return(orc.mlp_forward_bf16(crow, dims, obs), tgt))
    assert abs(float(one) - want) < 5e-4 * abs(want)


# ------------------------------------------------------------------ tcgen05 evaluate, fp16 operands (default mode)
def _f16_problem(dims, B, pairs, seed=23):
    rng = np.random.RandomState(seed)
    n = orc.mlp_param_count(dims)
    table_len = (n + 31) // 32 * 32 + (1 << 14)
    table = orc.round_f16(rng.standard_normal(table_len).astype(np.float32))   # fp16-exact, like the engine's
    theta = np.concatenate([np.concatenate([(rng.uniform(-1, 1, dims[i] * dims[i + 1]) / np.sqrt(dims[i])),
                                            rng.uniform(-1, 1, dims[i + 1]) / np.sqrt(dims[i])])
                            for i in range(len(dims) - 1)]).astype(np.float32)
    obs = rng.standard_normal((B, dims[0])).astype(np.float32)
    tgt = rng.standard_normal((B, dims[-1])).astype(np.float32)
    offs = orc.noise_offsets(11, 0, 0, pairs, table_len, n)
    return n, table, theta, obs, tgt, offs


@pytest.mark.parametrize("dims,B,pairs,bc", [([128, 512, 512, 288], 256, 5, 0), ([64, 64, 32], 256, 3, 0),
                                             ([128, 512, 512, 512, 512, 288], 256, 3, 0),
                                             ([64, 256, 64], 512, 4, 256), ([192, 320, 96], 256, 2, 0),
                                             ([256, 512, 32], 256, 2, 0)])
def test_eval_mlp_f16_tensor_core_path(be, dims, B, pairs, bc):
    """fp16-operand / fp32-accumulate tcgen05 path formed from fp32 theta + the exact fp16
    noise table: within 1e-5 (max-norm relative) of the oracle that emulates its roundings and
    within 3e-5 of the EXACT fp32 forward (estorch.py:195-202 + cartpole_es.py:14-20)."""
    n, table, theta, obs, tgt, offs = _f16_problem(dims, B, pairs)
    assert be.eval_supports_f16(dims, B)
    order = np.argsort(offs, kind="stable").astype(np.int32)
    tb = dev(be, table)
    tb16 = be.alloc(table.size, dtype=torch.float16)
    assert be.shadow_f16(tb, tb16) == 0
    np.testing.assert_array_equal(tb16.float().cpu().numpy(), table)
    ret = be.zeros(2 * pairs)
    bcp = be.zeros(pairs, bc) if bc else None
    bcm = be.zeros(pairs, bc) if bc else None
    be.eval_mlp(dims, dev(be, theta), tb, dev(be, offs), dev(be, order), pairs, 0.02, dev(be, obs),
                dev(be, tgt), ret[:pairs], ret[pairs:], bcp, bcm, 64 if bc else 0, bc, precision="f16", table16=tb16)
    torch.cuda.synchronize()
    got = ret.cpu().numpy()
    pop, _ = orc.sample_population(theta, table, offs, 0.02)
    outs = [orc.mlp_forward_f16(pop[i], dims, obs) for i in range(2 * pairs)]
    emu = np.array([orc.synthetic_return(o, tgt) for o in outs], dtype=np.float32)
    exact, _ = orc.evaluate_population(pop, dims, obs, tgt)
    print(f"f16 eval {dims} B={B}: vs emulation {rel_err(got, emu):.2e}, vs exact fp32 {rel_err(got, exact):.2e}")
    assert rel_err(got, emu) < 1e-5
    assert rel_err(got, exact) < 3e-5
    if bc:
        want_bc = np.stack([orc.synthetic_bc(orc.mlp_forward(pop[i], dims, obs), 64, bc) for i in range(2 * pairs)])
        got_bc = np.concatenate([bcp.cpu().numpy(), bcm.cpu().numpy()])
        assert np.max(np.abs(got_bc - want_bc)) < 2e-3 * np.max(np.abs(want_bc))
    one = be.zeros(1)
    be.eval_mlp_center(dims, dev(be, theta), dev(be, obs), dev(be, tgt), one, precision="f16")
    want = float(orc.synthetic_return(orc.mlp_forward(theta, dims, obs), tgt))
    assert abs(float(one) - want) < 3e-5 * abs(want)
    # a table that is not fp16-representable is reported, shapes outside the path are refused
    bad = dev(be, (table + np.float32(1e-4)).astype(np.float32))
    assert be.shadow_f16(bad, tb16) > 0
    with pytest.raises(RuntimeError, match="not supported"):
        be.eval_mlp([320, 64, 32], dev(be, theta[:22560]), tb, dev(be, offs), None, pairs, 0.02,
                    dev(be, np.zeros((256, 320), np.float32)), dev(be, np.zeros((256, 32), np.float32)),
                    ret[:pairs], ret[pairs:], precision="f16", table16=tb16)


def test_north_star_all_returns_ranks_and_gradient_f16_vs_fp32(be):
    """The north-star bar on the BENCHED evaluate path (VERDICT r1 J1): population_size = 4096,
    n = 1,001,760, B = 256.  ALL 4096 returns of the default tensor-core mode ("f16") against
    (i) the CPU oracle's fp32 forward of every member (estorch.py:195-202) and (ii) the exact
    CUDA-core kernel; then what the difference does to the rank indices, to the gradient
    estimate and to theta' (estorch.py:174-179, :236-245) -- next to the same figures for the
    fp32 kernel itself (two fp32 implementations also disagree in the last bits, and at this
    size neighbouring returns are ~1e-7 apart) and for the opt-in bf16 modes."""
    import json, os, time
    dims = [128, 512, 512, 512, 512, 288]
    n, P, pairs, sigma = orc.mlp_param_count(dims), 4096, 2048, 0.02
    torch.manual_seed(0)
    mods = []
    for i in range(len(dims) - 1):
        l = torch.nn.Linear(dims[i], dims[i + 1])
        mods += [l.weight.detach().reshape(-1), l.bias.detach()]
    theta = torch.cat(mods).contiguous()
    g = torch.Generator().manual_seed(1234)
    obs, tgt = torch.randn(256, 128, generator=g), torch.randn(256, 288, generator=g)
    table = be.alloc(1 << 26)
    be.fill_noise_table(table, 42)
    offs, order = be.alloc(pairs, dtype=torch.int64), be.alloc(pairs, dtype=torch.int32)
    be.make_offsets(42, None, 0, 0, pairs, table.numel(), n, offs, order)
    tb16 = be.alloc(table.numel(), dtype=torch.float16)
    assert be.shadow_f16(table, tb16) == 0                      # the engine's table is fp16-exact
    tbb, thb = be.alloc(table.numel(), dtype=torch.bfloat16), be.alloc(n, dtype=torch.bfloat16)
    th_d, obs_d, tgt_d = theta.to(be.device), obs.to(be.device), tgt.to(be.device)
    be.shadow_bf16(table, tbb); be.shadow_bf16(th_d, thb)
    res = {}
    for mode in ("fp32", "f16", "bf16", "bf16s"):
        r = be.zeros(P)
        be.eval_mlp(dims, th_d, table, offs, order, pairs, sigma, obs_d, tgt_d, r[:pairs], r[pairs:], precision=mode,
                    **({"table16": tb16} if mode == "f16" else {"theta16": thb, "table16": tbb} if mode == "bf16s" else {}))
        res[mode] = r
    torch.cuda.synchronize()
    # ---- CPU oracle: fp32 forward of every member on rows materialised like estorch.py:189-192
    t0 = time.time()
    tab_h, offs_h, th_h = table.cpu().numpy(), offs.cpu().numpy(), theta.numpy()
    obs_h, tgt_h = obs.numpy(), tgt.numpy()
    want = np.empty(P, np.float32)
    for j0 in range(0, pairs, 64):
        sl = offs_h[j0: j0 + 64]
        pop, _ = orc.sample_population(th_h, tab_h, sl, sigma)
        rr, _ = orc.evaluate_population(pop, dims, obs_h, tgt_h)
        want[j0: j0 + len(sl)] = rr[:len(sl)]
        want[pairs + j0: pairs + j0 + len(sl)] = rr[len(sl):]
    cpu_s = time.time() - t0
    assert len(np.unique(want)) > 2048

    from estorch_b200.backend import adam_desc, new_state

    def update(returns):
        th, m, v = th_d.clone(), be.zeros(n), be.zeros(n)
        ranks, grad = be.zeros(P, dtype=torch.int32), be.zeros(n)
        be.rank_grad_adam(returns, None, 1.0, 0.0, P, table, offs, order, th, m, v, new_state(be.device),
                          adam_desc(lr=0.01), ranks, None, grad)
        return ranks.cpu().numpy().astype(np.int64), grad.cpu().numpy(), th.cpu().numpy()

    base_ranks, base_g, base_th = update(torch.from_numpy(want).to(be.device))
    np.testing.assert_array_equal(base_ranks, orc.compute_ranks(want))      # rank indices: bit-exact on identical returns
    spread = float(want.std())
    gaps = np.diff(np.sort(want.astype(np.float64)))
    report = {"population_size": P, "n_parameters": n, "cpu_oracle_seconds": round(cpu_s, 1),
              "returns_mean": float(want.mean()), "returns_std": spread,
              "median_gap_between_neighbouring_returns_rel": float(np.median(gaps) / abs(want.mean())), "modes": {}}
    for mode, r in res.items():
        got = r.cpu().numpy()
        ranks, gg, th2 = update(r)
        d = np.abs(ranks - base_ranks)
        report["modes"][mode] = {
            "returns_max_rel_err_vs_cpu_fp32": rel_err(got, want),
            "returns_max_err_over_std": float(np.max(np.abs(got.astype(np.float64) - want)) / spread),
            "rank_indices_differing": int(np.count_nonzero(d)), "rank_max_displacement": int(d.max()),
            "rank_mean_displacement": float(d.mean()),
            "grad_rel_inf_vs_cpu_returns": rel_err(gg, base_g),
            "grad_rel_l2_vs_cpu_returns": float(np.linalg.norm(gg - base_g) / np.linalg.norm(base_g)),
            "theta_moved_entries_differing": int(np.count_nonzero(np.abs(th2 - base_th) > 1e-6))}
    print("NORTH_STAR_PRECISION " + json.dumps(report))
    out_dir = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "gpurun_out")
    if os.path.isdir(out_dir):
        json.dump(report, open(os.path.join(out_dir, "north_star_precision.json"), "w"), indent=1)
    m = report["modes"]
    assert m["fp32"]["returns_max_rel_err_vs_cpu_fp32"] < 2e-6
    # the parity bar of the default mode: every one of the 4096 returns within 1e-5 (max-norm relative)
    # of the reference's fp32 CPU arithmetic
    assert m["f16"]["returns_max_rel_err_vs_cpu_fp32"] < 1e-5
    # rank agreement and its effect on the update, as measured bounds (fp32-vs-fp32 is the floor)
    assert m["f16"]["rank_mean_displacement"] < 8 * max(1.0, m["fp32"]["rank_mean_displacement"])
    assert m["f16"]["grad_rel_l2_vs_cpu_returns"] < 3e-2
    assert m["f16"]["grad_rel_l2_vs_cpu_returns"] < 0.5 * m["bf16"]["grad_rel_l2_vs_cpu_returns"]


# ------------------------------------------------------------------ conv + VirtualBatchNorm evaluate
def test_eval_conv_vbn_matches_oracle_and_reference_golden(be):
    """examples/atari.py policy: (1) the centre evaluation reproduces the logits-based
    return of the reference's own forward (golden), (2) perturbed members match the oracle."""
    g = load_golden("atari_forward.npz")
    theta = seeded_theta(g)
    xref = g["xref8"].astype(np.float32) / np.float32(255)
    x = g["x8"].astype(np.float32) / np.float32(255)
    A, R, B = 4, xref.shape[0], x.shape[0]
    rng = np.random.RandomState(3)
    tgt = rng.standard_normal((B, A)).astype(np.float32)
    scratch = torch.empty(be.conv_scratch_bytes(R, B), dtype=torch.uint8, device=be.device)
    one = be.zeros(1)
    be.eval_conv_vbn(A, dev(be, theta), None, None, None, 1, 0.0, dev(be, xref), dev(be, x), dev(be, tgt),
                     one, None, scratch)
    want = float(orc.synthetic_return(g["logits"], tgt))          # logits from the unmodified reference
    assert abs(float(one) - want) < 2e-5 * abs(want)
    n = theta.size
    pairs = 3
    table_len = (n + 31) // 32 * 32 + (1 << 12)
    table = rng.standard_normal(table_len).astype(np.float32)
    offs = orc.noise_offsets(5, 0, 0, pairs, table_len, n)
    ret = be.zeros(2 * pairs)
    be.eval_conv_vbn(A, dev(be, theta), dev(be, table), dev(be, offs), None, pairs, 0.02, dev(be, xref),
                     dev(be, x), dev(be, tgt), ret[:pairs], ret[pairs:], scratch)
    pop, _ = orc.sample_population(theta, table, offs, 0.02)
    want = np.array([orc.synthetic_return(orc.atari_forward(pop[i], A, xref, x), tgt) for i in range(2 * pairs)])
    assert rel_err(ret.cpu().numpy(), want) < 5e-5
