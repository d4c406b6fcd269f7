"""GPU: several Dreamer agents in one env batch (DreamerAgents, rd_policy_dreamer_init_agents).

Every check is bitwise.  Each env's arithmetic reads only its own row of every activation and its agent's slice of the
stacked weights; a tensor-core product of one row does not depend on the other rows of its tile, the accumulation
groups and the epilogues are the single-agent launches', and the draws are keyed by the env id.  So env e under
DreamerAgents must give exactly what DreamerPolicy with agent agent_of_env[e]'s weights gives it."""
import numpy as np
import pytest

from oracle import dreamer_policy as dp

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def torch_cuda():
    import torch
    assert torch.cuda.is_available(), "these tests need a CUDA device"
    torch.cuda.set_device(0)
    return torch


@pytest.fixture(scope="module")
def austria():
    from racing_dreamer_b200.policy import load_dreamer_checkpoint
    return load_dreamer_checkpoint("austria_dreamer")


def make_env(**kw):
    from racing_dreamer_b200 import BatchedRaceEnv, EnvConfig
    base = dict(tracks=("austria",), action_repeat=4, reset_mode="random", seed=3)
    base.update(kw)
    return BatchedRaceEnv(EnvConfig(**base), device="cuda:0")


def assignment(kind, n, G, seed=0):
    if kind == "random":   # non-contiguous, every agent present
        a = np.random.RandomState(seed).randint(0, G, n)
        a[:G] = np.arange(G)
        return a.astype(np.int32)
    if kind == "slot":     # one agent per car slot of four-car worlds
        return (np.arange(n) % 4 % G).astype(np.int32)
    # contiguous groups whose sizes are not multiples of 128
    return np.minimum(np.arange(n) * G // n, G - 1).astype(np.int32)


def run(torch, pol, inputs, steps, training, noise, before_step=None):
    """set_state(inputs' state) then `steps` agent steps on fixed inputs; actions, diagnostics and state per step"""
    pol.set_state(*inputs["state"])
    out = []
    for k in range(steps):
        if before_step:
            before_step(k)
        kw = dict(debug=True, noise=noise, training=training)
        if noise == "explicit":
            kw.update(eps_stoch=inputs["eps_stoch"][k])
            kw.update(dict(eps_sample=inputs["eps_sample"][k], eps_expl=inputs["eps_expl"][k]) if training
                      else dict(eps_actor=inputs["eps_actor"][k]))
        a = pol.act(inputs["obs"], **kw) if "obs" in inputs else pol.act(occupancy=inputs["occ"], **kw)
        d = pol.diagnostics()
        out.append([a.clone()] + [d[k].clone() for k in ("mean", "std", "actor_mean", "actor_std", "action", "logp", "index")]
                   + [t.clone() for t in pol.get_state()])
    torch.cuda.synchronize()
    return out


def make_inputs(torch, rng, n, steps, n_samples=100, deter=200, occupancy=False):
    t = lambda x: torch.from_numpy(np.ascontiguousarray(x, np.float32)).cuda()   # noqa: E731
    inp = {"state": (t(rng.standard_normal((n, 30))), t(rng.uniform(-1, 1, (n, deter))), t(rng.uniform(-1, 1, (n, 2)))),
           "eps_stoch": [t(rng.standard_normal((n, 30))) for _ in range(steps)],
           "eps_actor": [t(rng.standard_normal((n, n_samples, 2))) for _ in range(steps)],
           "eps_sample": [t(rng.standard_normal((n, 2))) for _ in range(steps)],
           "eps_expl": [t(rng.standard_normal((n, 2))) for _ in range(steps)]}
    if occupancy:
        inp["occ"] = torch.from_numpy((rng.rand(n, 64, 64, 1) < 0.3).astype(np.uint8)).cuda()
    else:
        inp["obs"] = t(rng.uniform(0, 15, (n, 1080)))
    return inp


def check_equivalent(torch, env, weights, agent_of_env, inputs, noise, precision, training, steps=2, **expl):
    from racing_dreamer_b200 import DreamerAgents, DreamerPolicy
    G, R = len(weights), env.cfg.action_repeat
    agents = DreamerAgents(env, weights, agent_of_env, noise=noise, precision=precision, **expl)
    seen = {g: [] for g in range(G)}   # each agent's env_steps before each step
    got = run(torch, agents, inputs, steps, training, noise,
              lambda k: [seen[g].append(agents.env_steps(g)) for g in range(G)])
    for g in range(G):
        n_g = int((agent_of_env == g).sum())
        assert agents.env_steps(g) == (steps * n_g * R if training else 0)
    for g in range(G):
        amount = expl.get("expl_amount", 0.3)
        pol = DreamerPolicy(env, weights[g], noise=noise, precision=precision,
                            expl_amount=amount[g] if np.ndim(amount) else amount,
                            expl_decay=expl.get("expl_decay", 0.0), expl_min=expl.get("expl_min", 0.0))
        ref = run(torch, pol, inputs, steps, training, noise,
                  lambda k: setattr(pol, "env_steps", seen[g][k]))
        rows = torch.from_numpy(np.flatnonzero(agent_of_env == g)).cuda()
        for k in range(steps):
            for i, (x, y) in enumerate(zip(got[k], ref[k])):
                assert torch.equal(x[rows], y[rows]), f"agent {g}, step {k}, output {i}"
    return agents


@pytest.mark.parametrize("training", [False, True])
@pytest.mark.parametrize("noise", ["zero", "explicit", "philox"])
@pytest.mark.parametrize("precision", ["tf32x3", "tf32"])
def test_equivalent_to_single_agent_policies(torch_cuda, austria, precision, noise, training):
    torch = torch_cuda
    n = 300
    env = make_env(n_envs=n, env_id_offset=12345)
    rng = np.random.RandomState(5)
    inputs = make_inputs(torch, rng, n, 2)
    pool = [austria, dp.random_weights(41), dp.random_weights(42, normalized=True)]
    cases = [(2, "random", [0, 2], {}),
             (3, "slot", [0, 1, 2], dict(expl_amount=[0.3, 0.5, 0.1], expl_decay=1000.0, expl_min=0.05)),
             (2, "contiguous", [2, 1], dict(expl_amount=[0.2, 0.4]))]
    for G, kind, pick, expl in cases:
        check_equivalent(torch, env, [pool[i] for i in pick], assignment(kind, n, G), inputs, noise, precision,
                         training, **expl)
    env.close()


def test_closed_loop_against_single_agent_handles(torch_cuda, austria):
    """20 rollout steps in 4-car worlds with resets == G handles each driven by one DreamerPolicy on combined actions"""
    torch = torch_cuda
    from racing_dreamer_b200 import DreamerAgents, DreamerPolicy
    n, G, steps = 64, 2, 20
    ws = [austria, dp.random_weights(42, normalized=True)]
    aoe = assignment("slot", n, G)
    cfg = dict(n_envs=n, agents_per_world=4, auto_reset=True, time_limit_steps=7, seed=21)
    env = make_env(**cfg)
    env.reset()
    agents = DreamerAgents(env, ws, aoe)
    singles = []
    for g in range(G):
        e = make_env(**cfg)
        e.reset()
        singles.append((e, DreamerPolicy(e, ws[g])))
    masks = [torch.from_numpy(aoe == g).cuda() for g in range(G)]
    dones = 0
    for _ in range(steps):
        obs, rew, done, _ = agents.rollout(1)
        act = agents.actions.clone()
        combined = torch.empty_like(act)
        for g, (e, pol) in enumerate(singles):
            a = pol.act()
            assert torch.equal(a[masks[g]], act[masks[g]])
            combined[masks[g]] = a[masks[g]]
        for e, _ in singles:
            o2, r2, d2, _ = e.step(combined)
            assert torch.equal(o2["lidar"], obs["lidar"]) and torch.equal(r2, rew) and torch.equal(d2, done)
        dones += int(done.sum())
    assert dones > 0, "the time limit must reset some envs"
    for e, _ in singles:
        e.close()
    env.close()


def test_recorded_rollout_holds_the_agents_actions(torch_cuda, austria):
    torch = torch_cuda
    from racing_dreamer_b200 import BatchedRaceEnv, DreamerAgents, EnvConfig
    from racing_dreamer_b200.episodes import DeviceEpisodeStore
    ec = EnvConfig(tracks=("austria",), n_envs=16, action_repeat=4, auto_reset=False,
                   reset_mode="random", time_limit_steps=30, seed=11)
    ws = [austria, dp.random_weights(41)]
    aoe = assignment("slot", 16, 2)
    runs = []
    for mode in ("rollout", "loop"):
        env = BatchedRaceEnv(ec, device="cuda:0")
        store = DeviceEpisodeStore(env, capacity_rows=400)
        pol = DreamerAgents(env, ws, aoe, expl_amount=[0.3, 0.1])
        store.reset()
        executed = set()
        if mode == "rollout":
            pol.rollout(70, training=True, store=store)
        else:
            for _ in range(70):
                a = pol.act(training=True)
                executed.update(map(bytes, a.cpu().numpy()))
                store.step(a)
        torch.cuda.synchronize()
        runs.append((store.episodes(), executed, [pol.env_steps(g) for g in range(2)]))
        env.close()
    (e1, _, s1), (e2, executed, s2) = runs
    assert len(e1) == len(e2) >= 16 and s1 == s2 == [70 * 8 * 4] * 2
    for x, y in zip(e1, e2):
        for k in x:
            assert np.array_equal(np.asarray(x[k]).view(np.uint8), np.asarray(y[k]).view(np.uint8)), k
        assert all(bytes(r) in executed for r in np.asarray(y["action"][1:], np.float32))


def test_refresh_changes_only_that_agent(torch_cuda, austria):
    torch = torch_cuda
    from racing_dreamer_b200 import DreamerAgents
    n = 300
    env = make_env(n_envs=n)
    aoe = assignment("random", n, 3, seed=4)
    ws = [austria, dp.random_weights(41), dp.random_weights(42, normalized=True)]
    new = dp.random_weights(77)
    inputs = make_inputs(torch, np.random.RandomState(8), n, 2)
    base = run(torch, DreamerAgents(env, ws, aoe), inputs, 2, False, "philox")
    fresh = run(torch, DreamerAgents(env, [ws[0], new, ws[2]], aoe), inputs, 2, False, "philox")
    pol = DreamerAgents(env, ws, aoe)
    pol.load_weights({k: torch.from_numpy(v).cuda() for k, v in new.items()}, agent=1)
    got = run(torch, pol, inputs, 2, False, "philox")
    one = torch.from_numpy(aoe == 1).cuda()
    for k in range(2):
        for x, b, f in zip(got[k], base[k], fresh[k]):
            assert torch.equal(x, f)
            assert torch.equal(x[~one], b[~one])
    assert not torch.equal(got[1][0][one], base[1][0][one])
    with pytest.raises(ValueError, match="BN head"):   # agent 2 was built with a BN head
        pol.load_weights(new, agent=2)
    with pytest.raises(ValueError, match=r"agent 3 is not in \[0, 3\)"):
        pol.load_weights(new, agent=3)
    env.close()


def test_single_agent_calls_refuse_a_multi_agent_policy(torch_cuda, austria):
    import ctypes as C
    from racing_dreamer_b200 import DreamerAgents, DreamerPolicy, _abi
    env = make_env(n_envs=8)
    pol = DreamerAgents(env, [austria, austria], np.arange(8) % 2)
    x = _abi.RdDreamerExploration()
    assert env.lib.rd_policy_dreamer_get_exploration(env._handle, C.byref(x)) == -1
    assert env.lib.rd_policy_dreamer_set_exploration(env._handle, C.byref(x)) == -1
    with pytest.raises(RuntimeError, match="use rd_policy_dreamer_set_agent_weights"):
        DreamerPolicy.load_weights(pol, dp.random_weights(41))
    assert env.lib.rd_policy_dreamer_get_agent_exploration(env._handle, 2, C.byref(x)) == -1
    env.close()


@pytest.mark.parametrize("precision", ["tf32x3", "tf32"])
def test_encoder_agents(torch_cuda, precision):
    torch = torch_cuda
    import occupancy_reference as occ_ref
    from racing_dreamer_b200 import DreamerAgents, DreamerPolicy
    n = 300
    env = make_env(n_envs=n, tracks=("austria", "columbia"), obs_type="lidar_occupancy")
    ws = [occ_ref.random_weights(51), occ_ref.random_weights(52, normalized=True)]
    aoe = assignment("random", n, 2, seed=9)
    inputs = make_inputs(torch, np.random.RandomState(10), n, 2, occupancy=True)
    for noise in ("explicit", "philox"):
        check_equivalent(torch, env, ws, aoe, inputs, noise, precision, False)
        # check_equivalent's single-agent policies replaced the handle's agents: build them again for encode()
        emb = DreamerAgents(env, ws, aoe, precision=precision).encode(inputs["occ"]).clone()
        for g in range(2):
            single = DreamerPolicy(env, ws[g], precision=precision)
            rows = torch.from_numpy(aoe == g).cuda()
            assert torch.equal(emb[rows], single.encode(inputs["occ"])[rows])
    check_equivalent(torch, env, ws, aoe, inputs, "philox", precision, True)
    env.close()
