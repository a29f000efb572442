"""Drop-in check: user programs written against the original estorch API run unchanged on this package.

The programs below are the four usage patterns of the original project's example scripts
(examples/cartpole_es.py, early_stopping.py, custom_es.py, nsra_es.py): the same classes, constructor
arguments, overridden hooks and attribute accesses, at test size (``n_proc=1``, a few generations,
population 8).  They ``import estorch``, which resolves to ``estorch_b200``, see a stand-in ``gym``
(gym is not a dependency) and run on the CPU stand-in backend of tests/_oracle_backend.py.
"""
import collections
import math
import sys
import types

import numpy as np
import pytest
import torch

import estorch_b200
from _oracle_backend import OracleBackend


class _Space:
    def __init__(self, shape=None, n=None):
        self.shape, self.n = shape, n


class CartPoleStandIn:
    """Textbook cart-pole (Barto, Sutton & Anderson 1983 equations, Euler steps of 20 ms) with
    the pre-0.26 gym protocol the reference examples use: reset() -> obs,
    step(a) -> (obs, reward, done, info); episodes end at |x| > 2.4, |angle| > 12 deg or 500 steps."""
    gravity, m_cart, m_pole, half_len, force, tau = 9.8, 1.0, 0.1, 0.5, 10.0, 0.02

    def __init__(self, seed=0):
        self.observation_space, self.action_space = _Space(shape=(4,)), _Space(n=2)
        self.rng = np.random.RandomState(seed)
        self.state, self.t = None, 0

    def reset(self):
        self.state, self.t = self.rng.uniform(-0.05, 0.05, size=4), 0
        return self.state.astype(np.float32)

    def step(self, action):
        x, x_dot, th, th_dot = self.state
        f = self.force if int(action) == 1 else -self.force
        total_m, pm_l = self.m_cart + self.m_pole, self.m_pole * self.half_len
        tmp = (f + pm_l * th_dot ** 2 * math.sin(th)) / total_m
        th_acc = (self.gravity * math.sin(th) - math.cos(th) * tmp) / \
                 (self.half_len * (4.0 / 3.0 - self.m_pole * math.cos(th) ** 2 / total_m))
        x_acc = tmp - pm_l * th_acc * math.cos(th) / total_m
        self.state = np.array([x + self.tau * x_dot, x_dot + self.tau * x_acc,
                               th + self.tau * th_dot, th_dot + self.tau * th_acc])
        self.t += 1
        done = bool(abs(self.state[0]) > 2.4 or abs(self.state[2]) > 12 * math.pi / 180 or self.t >= 500)
        return self.state.astype(np.float32), 1.0, done, {}

    def render(self):
        pass


class WalkerStandIn:
    """A 24-observation / 4-action continuous-control stand-in with the shape of BipedalWalker-v3
    (examples/nsra_es.py): a damped linear system pushed by the actions; 40-70 steps per episode,
    reward = forward velocity minus an action cost."""

    def __init__(self, seed=0):
        self.observation_space, self.action_space = _Space(shape=(24,)), _Space(shape=(4,))
        self.rng = np.random.RandomState(seed)
        self.mix = self.rng.standard_normal((4, 24)).astype(np.float32) * 0.3

    def reset(self):
        self.state = self.rng.uniform(-0.1, 0.1, size=24).astype(np.float32)
        self.t, self.horizon = 0, int(self.rng.randint(40, 71))
        return self.state.copy()

    def step(self, action):
        a = np.clip(np.asarray(action, dtype=np.float32).reshape(4), -1.0, 1.0)
        self.state = (0.9 * self.state + a @ self.mix).astype(np.float32)
        self.t += 1
        return self.state.copy(), float(self.state[0] - 0.01 * np.sum(a * a)), self.t >= self.horizon, {}

    def render(self):
        pass




class Policy(torch.nn.Module):
    """The examples' policy: two hidden layers of 64 with ReLU."""

    def __init__(self, n_input, n_output):
        super().__init__()
        self.linear_1 = torch.nn.Linear(n_input, 64)
        self.linear_2 = torch.nn.Linear(64, 64)
        self.linear_3 = torch.nn.Linear(64, n_output)

    def forward(self, x):
        return self.linear_3(torch.relu(self.linear_2(torch.relu(self.linear_1(x)))))


class CartPoleAgent:
    """A gym-style host agent: greedy discrete actions, return = summed reward."""

    def __init__(self, device=torch.device("cpu")):
        import gym
        self.env, self.device = gym.make("CartPole-v1"), device

    def rollout(self, policy, render=False):
        observation, done, total = self.env.reset(), False, 0.0
        with torch.no_grad():
            while not done:
                action = int(torch.argmax(policy(torch.from_numpy(observation).float().to(self.device))))
                observation, reward, done, _ = self.env.step(action)
                if render:
                    self.env.render()
                total += reward
        return total


class WalkerAgent:
    """The novelty-search agent protocol: rollout -> (reward, behaviour characterisation), the
    characterisation being the first and the last ``n`` actions of the episode."""

    def __init__(self, device=torch.device("cpu"), n=32):
        import gym
        self.env, self.device, self.n = gym.make("BipedalWalker-v3"), device, n

    def rollout(self, policy, render=False):
        observation, done, total = self.env.reset(), False, 0.0
        first, last = [], collections.deque(maxlen=self.n)
        with torch.no_grad():
            while not done:
                action = policy(torch.from_numpy(observation).float().to(self.device)).cpu().numpy()
                observation, reward, done, _ = self.env.step(action)
                total += reward
                last.append(action)
                if len(first) < self.n:
                    first.append(action)
        return total, np.concatenate([first, last]).flatten()


def cartpole_program(n_steps, population=8):
    """examples/cartpole_es.py: train, then roll out es.policy and a Policy loaded from es.best_policy_dict."""
    import estorch
    device = torch.device("cpu")
    agent = CartPoleAgent()
    n_input, n_output = agent.env.observation_space.shape[0], agent.env.action_space.n
    es = estorch.ES(Policy, CartPoleAgent, torch.optim.Adam, population_size=population, sigma=0.02, device=device,
                    policy_kwargs={"n_input": n_input, "n_output": n_output}, agent_kwargs={"device": device},
                    optimizer_kwargs={"lr": 0.01})
    es.train(n_steps=n_steps, n_proc=1)
    print(f"Latest Policy Reward: {agent.rollout(es.policy)}")
    policy = Policy(n_input, n_output).to(device)
    policy.load_state_dict(es.best_policy_dict)
    print(f"Best Policy Reward: {agent.rollout(policy)}")
    return es


def early_stopping_program(n_steps, population=8):
    """examples/early_stopping.py: log() reads population_returns / population_parameters and calls
    terminate() once a member reaches CartPole's maximum of 500."""
    import estorch

    class ES(estorch.ES):
        def log(self):
            idx = int(np.argmax(self.population_returns[:, 0]))
            reward = self.population_returns[idx, 0]
            print(f"Reward: {reward}")
            if reward == 500:
                self.best = self.population_parameters[idx]
                self.terminate()

    device = torch.device("cpu")
    agent = CartPoleAgent()
    n_input, n_output = agent.env.observation_space.shape[0], agent.env.action_space.n
    es = ES(Policy, CartPoleAgent, torch.optim.Adam, population_size=population, sigma=0.02, device=device,
            policy_kwargs={"n_input": n_input, "n_output": n_output}, agent_kwargs={"device": device},
            optimizer_kwargs={"lr": 0.01})
    es.train(n_steps=n_steps, n_proc=1)
    policy = Policy(n_input, n_output).to(device)
    torch.nn.utils.vector_to_parameters(es.best.to(device), policy.parameters())
    print(f"Reward: {agent.rollout(policy)}")
    return es


def custom_es_program(n_steps, population=8):
    """examples/custom_es.py: a subclass overrides _sample_policy / _calculate_grad (mirrored sampling,
    PGPE-style update) and uses the package's rank_transformation."""
    import estorch

    class SymmetricES(estorch.ES):
        def _sample_policy(self, policy):
            theta = torch.nn.utils.parameters_to_vector(policy.parameters()).detach().cpu()
            epsilon = self.sigma * torch.randn(self.population_size // 2, theta.numel())
            return torch.cat((theta + epsilon, theta - epsilon)), epsilon

        def _calculate_grad(self, epsilon):
            ranked = torch.from_numpy(estorch.rank_transformation(self.population_returns.squeeze())).float()
            half = self.population_size // 2
            return (ranked[:half] - ranked[half:]) @ epsilon / (half * self.sigma)

    device = torch.device("cpu")
    agent = CartPoleAgent()
    n_input, n_output = agent.env.observation_space.shape[0], agent.env.action_space.n
    es = SymmetricES(Policy, CartPoleAgent, torch.optim.Adam, population_size=population, sigma=0.02, device=device,
                     policy_kwargs={"n_input": n_input, "n_output": n_output}, agent_kwargs={"device": device},
                     optimizer_kwargs={"lr": 0.01})
    es.train(n_steps=n_steps, n_proc=1)
    policy = Policy(n_input, n_output).to(device)
    policy.load_state_dict(es.best_policy_dict)
    print(f"Best Policy Reward: {agent.rollout(policy)}")
    return es


def nsra_program(n_steps, population=8):
    """examples/nsra_es.py: NSRA_ES with an adaptive weight, then roll out every meta-population member
    and the best policy."""
    import estorch
    device = torch.device("cpu")
    agent = WalkerAgent()
    n_input, n_output = agent.env.observation_space.shape[0], agent.env.action_space.shape[0]
    es = estorch.NSRA_ES(Policy, WalkerAgent, torch.optim.Adam, population_size=population, sigma=0.02, weight_t=10,
                         device=device, policy_kwargs={"n_input": n_input, "n_output": n_output},
                         agent_kwargs={"device": device}, optimizer_kwargs={"lr": 0.01})
    es.train(n_steps=n_steps, n_proc=1)
    for idx, (policy, _) in enumerate(es.meta_population):
        reward, _ = agent.rollout(policy)
        print(f"Reward of {idx}. policy from the meta population: {reward}")
    policy = Policy(n_input, n_output).to(device)
    policy.load_state_dict(es.best_policy_dict)
    print(f"Best Policy Reward: {agent.rollout(policy)[0]}")
    return es


@pytest.fixture
def reference_world(monkeypatch):
    """``import estorch`` -> this package (CPU stand-in backend), ``import gym`` -> the stand-in."""
    gym = types.ModuleType("gym")
    gym.make = lambda name: CartPoleStandIn() if name.startswith("CartPole") else WalkerStandIn()
    monkeypatch.setitem(sys.modules, "gym", gym)
    monkeypatch.setitem(sys.modules, "estorch", estorch_b200)
    real_init = estorch_b200.ES.__init__

    def init_with_cpu_backend(self, *a, **kw):
        kw.setdefault("_backend", OracleBackend())
        kw.setdefault("noise_table_size", 1 << 16)
        real_init(self, *a, **kw)
    monkeypatch.setattr(estorch_b200.ES, "__init__", init_with_cpu_backend)


def test_cartpole_example_runs_unmodified(reference_world, capsys):
    """cartpole_es.py: ES(Policy, Agent, Adam, ...).train(), then es.policy and
    es.best_policy_dict feed the user's own rollout (estorch.py:108-117 attributes)."""
    es = cartpole_program(n_steps=2)
    assert type(es).__name__ == "ES" and not es._fused        # a gym-style host agent: hooks path
    assert es.step == 2 and es.population_returns.shape == (8, 1) and es.population_returns.dtype == np.float32
    assert set(es.best_policy_dict) == set(Policy(4, 2).state_dict())
    out = capsys.readouterr().out
    assert "Latest Policy Reward" in out and "Best Policy Reward" in out and "Episode Reward" in out


def test_early_stopping_example_runs_unmodified(reference_world, capsys, monkeypatch):
    """early_stopping.py overrides log(), indexes population_parameters by member and
    calls terminate() (estorch.py:150-152): make every episode 'perfect' so that it triggers."""
    monkeypatch.setattr(CartPoleAgent, "rollout", lambda self, policy, render=False: 500.0)
    es = early_stopping_program(n_steps=5)
    assert es.step == 1                                            # stopped after the first generation
    assert tuple(es.best.shape) == (es.n_parameters,)
    assert "Reward: 500" in capsys.readouterr().out


def test_custom_es_example_runs_unmodified(reference_world, capsys):
    """custom_es.py overrides _sample_policy / _calculate_grad and imports
    rank_transformation from the package: the engine must honour the overrides."""
    es = custom_es_program(n_steps=2)
    assert type(es).__name__ == "SymmetricES" and not es._fused
    assert es.step == 2 and torch.isfinite(torch.nn.utils.parameters_to_vector(es.policy.parameters())).all()
    assert "Best Policy Reward" in capsys.readouterr().out


def test_nsra_example_runs_unmodified(reference_world, capsys):
    """nsra_es.py: rollout -> (reward, behaviour characterisation), the archive /
    meta-population / adaptive weight of estorch.py:388-472,623-662, es.meta_population and
    es.best_policy_dict afterwards."""
    np.random.seed(0)
    es = nsra_program(n_steps=2, population=8)
    assert type(es).__name__ == "NSRA_ES" and len(es.meta_population) == 3
    assert es.population_returns.shape == (8, 2) and len(es._archive) == 3 + 2    # +1 behaviour per generation
    assert not hasattr(es, "policy")                                              # as in the reference (estorch.py:135-137)
    assert 0.0 <= es.weight <= 1.0
    out = capsys.readouterr().out
    assert "Reward of 2. policy from the meta population" in out and "Best Policy Reward" in out
