#!/usr/bin/env python
"""Generate the golden fixtures in this directory from the UNMODIFIED reference.

Runs only in the build container (needs /root/reference); the fixtures it
writes are committed and are what travels to the GPU box.  The reference is
imported as-is through two shims (SURVEY 8c): a single-rank ``mpi4py`` stand-in
(the reference imports it at estorch.py:10; with n_proc=1 no MPI call is made)
and ``np.int = int`` (estorch.py:453 uses the alias numpy removed).  The
reference classes are driven through their own documented hooks:
``_sample_policy`` is overridden to inject eps = sigma * T[off : off+n]
(examples/custom_es.py:12-18 shows this is the supported extension point);
rank_transformation, torch.mm, negate/clamp, torch.optim.Adam.step,
cKDTree novelty and the NSRA schedule all run as the reference's own code.

    python tests/golden/make_golden.py
"""
import os
import sys
import types

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.dirname(HERE))     # tests/: conftest.seeded_theta


def _install_shims():
    m = types.ModuleType("mpi4py")
    MPI = types.ModuleType("mpi4py.MPI")

    class _Comm:
        def Get_rank(self): return 0
        def Get_size(self): return 1
        def send(self, *a, **k): pass
        def bcast(self, x, root=0): return x

    class Status:
        def Get_tag(self): return 0

    MPI.COMM_WORLD, MPI.Status, m.MPI = _Comm(), Status, MPI
    sys.modules["mpi4py"], sys.modules["mpi4py.MPI"] = m, MPI
    np.int = int
    for name in ("gym", "skimage", "skimage.transform"):
        sys.modules.setdefault(name, types.ModuleType(name))
    sys.modules["skimage.transform"].resize = lambda *a, **k: None
    sys.path.insert(0, "/root/reference")
    sys.path.insert(0, "/root/reference/examples")


_install_shims()
import estorch as ref  # noqa: E402  (the reference)
from oracle import es_oracle as orc  # noqa: E402


class MLP(torch.nn.Module):
    def __init__(self, dims):
        super().__init__()
        layers = []
        for i in range(len(dims) - 1):
            layers.append(torch.nn.Linear(dims[i], dims[i + 1]))
            if i + 2 < len(dims):
                layers.append(torch.nn.ReLU())
        self.net = torch.nn.Sequential(*layers)

    def forward(self, x):
        return self.net(x)


class SynthAgent:
    """rollout = -mean((policy(obs)-y)^2); NS: + bc = policy(obs[:bc_obs]).flatten()[:bc_dim]."""
    def __init__(self, obs, target, bc_obs=0, bc_dim=0):
        self.obs, self.target, self.bc_obs, self.bc_dim = obs, target, bc_obs, bc_dim

    def rollout(self, policy):
        with torch.no_grad():
            out = policy(self.obs)
            r = float(-((out - self.target) ** 2).mean())
            if self.bc_dim:
                return r, out[:self.bc_obs].flatten()[:self.bc_dim].numpy().copy()
        return r


def _flat(params):
    return torch.nn.utils.parameters_to_vector(params).detach().cpu().numpy().copy()


def _adam_state(opt, policy):
    m = np.concatenate([opt.state[p]["exp_avg"].reshape(-1).numpy() for p in policy.parameters()])
    v = np.concatenate([opt.state[p]["exp_avg_sq"].reshape(-1).numpy() for p in policy.parameters()])
    return m.copy(), v.copy()


def make_table(length, seed):
    g = torch.Generator().manual_seed(seed)
    return torch.randn(length, generator=g, dtype=torch.float32).numpy().copy()


def run_reference(cls, dims, P, sigma, n_gen, table, noise_seed, obs, target,
                  bc_obs=0, bc_dim=0, extra_kwargs=None, torch_seed=0, np_seed=123):
    rec = dict(theta_before=[], offsets=[], grad=[], returns=[], theta_after=[],
               episode_reward=[], best_reward=[], idx=[], weight=[], t=[], archive_len=[])
    tab_t = torch.from_numpy(table)
    n = orc.mlp_param_count(dims)

    class Rec(cls):
        def _sample_policy(self, policy):
            theta = torch.nn.utils.parameters_to_vector(policy.parameters()).detach().cpu()
            offs = orc.noise_offsets(noise_seed, self.step, 0, P // 2, len(table), n)
            t = torch.stack([tab_t[o:o + n] for o in offs])
            eps = t * self.sigma
            rec["theta_before"].append(theta.numpy().copy())
            rec["offsets"].append(offs)
            return torch.cat((theta + eps, theta - eps)), torch.cat((eps, -eps))

        def _calculate_grad(self, epsilon):
            g = super()._calculate_grad(epsilon)
            rec["grad"].append(g.numpy().copy())
            return g

        def log(self):
            rec["returns"].append(self.population_returns.copy())
            rec["episode_reward"].append(self.episode_reward)
            rec["best_reward"].append(self.best_reward)
            if hasattr(self, "meta_population"):
                pol = self.meta_population[self.idx][0]
                rec["idx"].append(self.idx)
                rec["archive_len"].append(len(self._archive))
            else:
                pol = self.policy
            rec["theta_after"].append(_flat(pol.parameters()))
            rec["weight"].append(getattr(self, "weight", np.nan))
            rec["t"].append(getattr(self, "t", -1))

    torch.manual_seed(torch_seed)
    np.random.seed(np_seed)
    kw = dict(extra_kwargs or {})
    es = Rec(MLP, SynthAgent, torch.optim.Adam, population_size=P, sigma=sigma,
             policy_kwargs={"dims": dims},
             agent_kwargs=dict(obs=obs, target=target, bc_obs=bc_obs, bc_dim=bc_dim),
             optimizer_kwargs={"lr": 0.01}, **kw)
    out = dict(dims=np.array(dims), P=P, sigma=sigma, noise_seed=noise_seed, table=table,
               obs=obs.numpy(), target=target.numpy(), bc_obs=bc_obs, bc_dim=bc_dim)
    if hasattr(es, "meta_population"):
        out["meta_theta0"] = np.stack([_flat(p.parameters()) for p, _ in es.meta_population])
        out["archive0"] = np.stack(es._archive)
        out["k"] = es.k
    else:
        out["theta0"] = _flat(es.policy.parameters())
    es.train(n_steps=n_gen, n_proc=1)
    for k_, v_ in rec.items():
        out[k_] = np.array(v_)
    if hasattr(es, "meta_population"):
        out["archive_final"] = np.stack(es._archive)
        ms, vs = [], []
        for pol, opt in es.meta_population:
            if len(opt.state):
                m_, v_ = _adam_state(opt, pol)
            else:
                m_ = v_ = np.zeros(n, np.float32)
            ms.append(m_); vs.append(v_)
        out["meta_m"], out["meta_v"] = np.stack(ms), np.stack(vs)
        out["meta_theta_final"] = np.stack([_flat(p.parameters()) for p, _ in es.meta_population])
    else:
        out["m_final"], out["v_final"] = _adam_state(es.optimizer, es.policy)
        bp = es.best_policy_dict
        out["best_theta"] = np.concatenate([bp[k].reshape(-1).numpy() for k in bp])
    return out


def write_atari_fixture():
    """Atari conv + VBN policy forward (examples/atari.py:14-37).  The 677k parameters are stored as the
    recipe of conftest.seeded_theta (default-init ranges, gamma/beta spread around 1/0), not as values,
    to keep the fixture small; frames are stored as uint8."""
    import atari as ref_atari  # the reference example module (gym/skimage shimmed)
    from conftest import seeded_theta
    recipe = dict(theta_seed=2024, theta_sizes=[], theta_lo=[], theta_hi=[])
    fan_in = 1
    for name, shape in orc.atari_param_layout(4):
        if name.endswith(".w") and len(shape) > 1:
            fan_in = int(np.prod(shape[1:]))
        lo, hi = (0.8, 1.2) if name.startswith("bn") and name.endswith(".w") else \
            (-0.2, 0.2) if name.startswith("bn") else (-fan_in ** -0.5, fan_in ** -0.5)
        recipe["theta_sizes"].append(int(np.prod(shape)))
        recipe["theta_lo"].append(lo)
        recipe["theta_hi"].append(hi)
    recipe = {k: np.array(v) for k, v in recipe.items()}
    g = torch.Generator().manual_seed(4321)
    xref8 = (torch.rand(8, 4, 84, 84, generator=g) * 255).round().to(torch.uint8)
    x8 = (torch.rand(3, 4, 84, 84, generator=g) * 255).round().to(torch.uint8)
    pol = ref_atari.Policy(4, xref8.float() / 255)
    torch.nn.utils.vector_to_parameters(torch.from_numpy(seeded_theta(recipe)), pol.parameters())
    with torch.no_grad():
        logits = pol(x8.float() / 255)
    np.savez_compressed(os.path.join(HERE, "atari_forward.npz"), xref8=xref8.numpy(), x8=x8.numpy(),
                        logits=logits.numpy(), **recipe)


def main():
    # --- the one known-answer vector the reference ships (estorch.py:31-35) ---
    doc_in = np.array([-123, -50, 3, -5, 20, 10, 100], dtype=np.float64)
    np.savez(os.path.join(HERE, "rank_docstring.npz"), rewards=doc_in,
             expected=ref.rank_transformation(list(doc_in)),
             ranks=ref.estorch._compute_ranks(list(doc_in)))

    # --- rank transform on larger tie-free inputs ---
    rng = np.random.RandomState(5)
    r4096 = rng.standard_normal(4096).astype(np.float32)
    assert len(np.unique(r4096)) == 4096
    np.savez_compressed(os.path.join(HERE, "rank_p4096.npz"), rewards=r4096,
                        ranks=ref.estorch._compute_ranks(r4096),
                        centred=ref.rank_transformation(r4096))

    g = torch.Generator().manual_seed(1234)
    # --- classic ES, CartPole-shape MLP (BASELINE config 1/2 shape), P=64 ---
    dims = [4, 64, 64, 2]
    obs = torch.randn(256, 4, generator=g)
    tgt = torch.randn(256, 2, generator=g)
    table = make_table(1 << 15, 42)
    out = run_reference(ref.ES, dims, 64, 0.1, 3, table, 7, obs, tgt)
    np.savez_compressed(os.path.join(HERE, "es_cartpole_p64.npz"), **out)

    # --- tiny case for pure-python loops: Linear(3,2), P=8 ---
    dims = [3, 2]
    obs = torch.randn(5, 3, generator=g)
    tgt = torch.randn(5, 2, generator=g)
    out = run_reference(ref.ES, dims, 8, 0.05, 2, make_table(1 << 10, 43), 11, obs, tgt)
    np.savez_compressed(os.path.join(HERE, "es_tiny_p8.npz"), **out)

    # --- NS family, BipedalWalker-shape MLP (BASELINE config 4 shape), P=32 ---
    dims = [24, 64, 64, 4]
    obs = torch.randn(256, 24, generator=g)
    tgt = torch.randn(256, 4, generator=g)
    table = make_table(1 << 15, 44)
    for name, cls, kw in (("ns", ref.NS_ES, {}), ("nsr", ref.NSR_ES, {}),
                          ("nsra", ref.NSRA_ES, {"weight_t": 2})):
        out = run_reference(cls, dims, 32, 0.02, 5, table, 13, obs, tgt,
                            bc_obs=64, bc_dim=256, extra_kwargs=kw)
        np.savez_compressed(os.path.join(HERE, f"{name}_bipedal_p32.npz"), **out)

    # --- VirtualBatchNorm two-call protocol (modules.py:48-58) ---
    vbn = ref.VirtualBatchNorm(3)
    with torch.no_grad():
        vbn.weight.copy_(torch.tensor([0.5, 1.5, -2.0]))
        vbn.bias.copy_(torch.tensor([0.1, -0.2, 0.3]))
        xref = torch.randn(6, 3, 5, 4, generator=g)
        x = torch.randn(2, 3, 5, 4, generator=g)
        y_ref = vbn(xref)
        assert vbn.mean is not None
        y = vbn(x)
        assert vbn.mean is None
    np.savez_compressed(os.path.join(HERE, "vbn.npz"), xref=xref.numpy(), x=x.numpy(),
                        gamma=vbn.weight.detach().numpy(), beta=vbn.bias.detach().numpy(),
                        y_ref=y_ref.numpy(), y=y.numpy())

    write_atari_fixture()
    print("fixtures written to", HERE)
    for f in sorted(os.listdir(HERE)):
        if f.endswith(".npz"):
            print(f"  {f}: {os.path.getsize(os.path.join(HERE, f)) / 1024:.1f} KB")


if __name__ == "__main__":
    main()
