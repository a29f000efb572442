"""Pin the CPU oracle against the reference's own outputs (tests/golden/*.npz,
written by tests/golden/make_golden.py from the unmodified reference)."""
import numpy as np
import pytest

from oracle import es_oracle as orc
from conftest import load_golden, rel_err, seeded_theta


def test_rank_docstring_vector():
    # the only known-answer vector in the reference tree: estorch/estorch.py:31-35
    expected = np.array([-0.5, -0.33333333, 0., -0.16666667, 0.33333333, 0.16666667, 0.5])
    got = orc.rank_transformation([-123, -50, 3, -5, 20, 10, 100])
    np.testing.assert_allclose(got, expected, atol=5e-9)
    g = load_golden("rank_docstring.npz")
    np.testing.assert_array_equal(got, g["expected"])          # bit-exact float64
    np.testing.assert_array_equal(orc.compute_ranks(g["rewards"]), g["ranks"])


def test_rank_p4096_bit_exact():
    g = load_golden("rank_p4096.npz")
    np.testing.assert_array_equal(orc.compute_ranks(g["rewards"]), g["ranks"])
    np.testing.assert_array_equal(orc.rank_transformation(g["rewards"]), g["centred"])


def test_rank_ties_stable_by_index():
    r = np.array([1.0, 0.0, 1.0, 0.0], dtype=np.float32)
    np.testing.assert_array_equal(orc.compute_ranks(r), [2, 0, 3, 1])


@pytest.mark.parametrize("name", ["es_tiny_p8.npz", "es_cartpole_p64.npz"])
def test_es_generations_match_reference(name):
    g = load_golden(name)
    dims = [int(d) for d in g["dims"]]
    P, sigma = int(g["P"]), float(g["sigma"])
    n = orc.mlp_param_count(dims)
    theta = g["theta0"].copy()
    m = np.zeros(n, np.float32)
    v = np.zeros(n, np.float32)
    best = -np.inf
    for gen in range(len(g["grad"])):
        offs = orc.noise_offsets(int(g["noise_seed"]), gen, 0, P // 2, len(g["table"]), n)
        np.testing.assert_array_equal(offs, g["offsets"][gen])
        np.testing.assert_array_equal(theta, g["theta_before"][gen]) if gen == 0 else None
        res = orc.es_generation(theta, m, v, gen, g["table"], offs, sigma, dims,
                                g["obs"], g["target"])
        ref_ret = g["returns"][gen][:, 0]
        assert rel_err(res["returns"], ref_ret) < 2e-6
        # stage B: identical return bits -> identical ranks, grad within 1e-5
        resB = orc.es_generation(theta, m, v, gen, g["table"], offs, sigma, dims,
                                 g["obs"], g["target"], returns=ref_ret)
        assert rel_err(resB["grad"], g["grad"][gen]) < 1e-5
        # Adam on identical gradient bits reproduces torch.optim.Adam ...
        th, m1, v1 = orc.adam_step(theta, m, v, orc.negate_clamp(g["grad"][gen]), gen + 1)
        assert rel_err(th, g["theta_after"][gen]) < 1e-6
        # ... and end-to-end theta is within 1e-5 wherever Adam's m/(sqrt(v)+eps) is
        # well conditioned (|g| not within ~1e-4 of zero: there the step flips sign
        # on a 1e-7 gradient difference -- a property of Adam, see DESIGN.md)
        ok = np.abs(g["grad"][gen]) > 1e-4 * np.abs(g["grad"][gen]).max()
        assert rel_err(resB["theta"][ok], g["theta_after"][gen][ok]) < 1e-5
        assert np.abs(resB["theta"] - g["theta_after"][gen]).max() <= 2.0 * 0.01
        resB["theta"], resB["m"], resB["v"] = th, m1, v1
        # the pair-difference form (what the CUDA kernel evaluates) agrees too
        gp = orc.calculate_grad_pairs(ref_ret, g["table"], offs, n)
        assert rel_err(gp, g["grad"][gen]) < 1e-5
        assert abs(float(resB["episode_reward"]) - float(g["episode_reward"][gen])) < 1e-5
        best = max(best, float(g["episode_reward"][gen]))
        assert best == pytest.approx(float(g["best_reward"][gen]))
        theta, m, v = resB["theta"], resB["m"], resB["v"]
    assert rel_err(m, g["m_final"]) < 1e-5
    assert rel_err(v, g["v_final"]) < 1e-5


@pytest.mark.parametrize("algo", ["ns", "nsr", "nsra"])
def test_ns_family_match_reference(algo):
    g = load_golden(f"{algo}_bipedal_p32.npz")
    dims = [int(d) for d in g["dims"]]
    P, sigma, k = int(g["P"]), float(g["sigma"]), int(g["k"])
    n = orc.mlp_param_count(dims)
    bc_obs, bc_dim = int(g["bc_obs"]), int(g["bc_dim"])
    thetas = g["meta_theta0"].copy()
    M = thetas.shape[0]
    ms = np.zeros((M, n), np.float32)
    vs = np.zeros((M, n), np.float32)
    steps = [0] * M
    archive = [orc.synthetic_bc(orc.mlp_forward(thetas[i], dims, g["obs"]), bc_obs, bc_dim)
               for i in range(M)]
    np.testing.assert_allclose(np.stack(archive), g["archive0"], rtol=1e-5, atol=1e-6)
    weight, t, best = 1.0, 0, -np.inf
    for gen in range(len(g["grad"])):
        idx = int(g["idx"][gen])                     # np.random.choice draw, injected
        theta = thetas[idx]
        np.testing.assert_allclose(theta, g["theta_before"][gen], rtol=0, atol=1e-7)
        offs = g["offsets"][gen]
        pop, eps = orc.sample_population(theta, g["table"], offs, sigma)
        rets, bcs = orc.evaluate_population(pop, dims, g["obs"], g["target"], bc_obs, bc_dim)
        arch = np.stack(archive)
        nov = np.array([orc.novelty(bcs[i], arch, k) for i in range(P)], dtype=np.float32)
        ref = g["returns"][gen]
        assert rel_err(rets, ref[:, 0]) < 2e-6
        assert rel_err(nov, ref[:, 1]) < 2e-5
        wref = float(g["weight"][gen])
        grad = orc.calculate_grad(ref, eps, sigma, algo=algo, weight=weight)
        assert rel_err(grad, g["grad"][gen]) < 1e-5
        steps[idx] += 1
        th, m_, v_ = orc.adam_step(theta, ms[idx], vs[idx], orc.negate_clamp(g["grad"][gen]),
                                   steps[idx])
        assert rel_err(th, g["theta_after"][gen]) < 1e-5
        thetas[idx], ms[idx], vs[idx] = th, m_, v_
        out = orc.mlp_forward(th, dims, g["obs"])
        ep = float(orc.synthetic_return(out, g["target"]))
        assert abs(ep - float(g["episode_reward"][gen])) < 1e-5
        archive.append(orc.synthetic_bc(out, bc_obs, bc_dim))
        assert len(archive) == int(g["archive_len"][gen])
        if algo == "nsra":
            weight, t, best = orc.nsra_weight_update(weight, t, float(g["episode_reward"][gen]),
                                                     best, weight_t=2)
            assert weight == pytest.approx(wref)
            assert t == int(g["t"][gen])
    np.testing.assert_allclose(np.stack(archive), g["archive_final"], rtol=1e-4, atol=1e-5)
    assert rel_err(ms, g["meta_m"]) < 1e-5
    assert rel_err(vs, g["meta_v"]) < 1e-5


def test_vbn_matches_reference():
    g = load_golden("vbn.npz")
    mean, var = orc.vbn_stats(g["xref"])
    y_ref = orc.vbn_normalize(g["xref"], mean, var, g["gamma"], g["beta"])
    y = orc.vbn_normalize(g["x"], mean, var, g["gamma"], g["beta"])
    np.testing.assert_allclose(y_ref, g["y_ref"], rtol=1e-5, atol=1e-5)
    np.testing.assert_allclose(y, g["y"], rtol=1e-5, atol=1e-5)


def test_atari_forward_matches_reference():
    g = load_golden("atari_forward.npz")
    theta = seeded_theta(g)
    xref = g["xref8"].astype(np.float32) / np.float32(255)
    x = g["x8"].astype(np.float32) / np.float32(255)
    logits = orc.atari_forward(theta, 4, xref, x)
    assert rel_err(logits, g["logits"]) < 1e-4


def test_philox_known_answer():
    # Random123 known-answer test: philox4x32-10, counter = key = 0
    x = orc.philox4x32_10(np.array([0], dtype=np.uint64), 0)
    assert [int(v[0]) for v in x] == [0x6627e8d5, 0xe169c58d, 0xbc57ac4c, 0x9b00dbd8]


def test_philox_table_is_unit_normal():
    t = orc.philox_normal_table(1 << 18, 42)
    assert abs(float(t.mean())) < 0.01 and abs(float(t.std()) - 1.0) < 0.01
    assert np.isfinite(t).all() and float(np.abs(t).max()) < 6.0
    np.testing.assert_array_equal(t[:64], orc.philox_normal_table(64, 42))


def test_offsets_aligned_and_in_range():
    offs = orc.noise_offsets(42, 3, 0, 2048, 1 << 20, 4610)
    assert (offs % 32 == 0).all() and offs.min() >= 0
    assert offs.max() + 4640 <= (1 << 20)
    # shard consistency: rank r's slice equals the same slice of the global list
    np.testing.assert_array_equal(orc.noise_offsets(42, 3, 512, 512, 1 << 20, 4610),
                                  offs[512:1024])
