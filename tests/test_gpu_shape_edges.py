"""GPU: the whole step at the shapes where kernels go wrong, against the autograd port.

The parity suite runs at batches that are multiples of 8, hidden widths that are multiples of 4, act_dim 2..4 and critics
of depth 2..3.  The step picks its kernels and launch geometry from the shape, so these cases reach code no other test
executes: the unclustered layer-chained path (critics deeper than C2_MAXL = 4), a partial last CTA in chain / chain2,
the FFMA fallback inside a precision-1 plan, tcgen05 and FFMA problems in one launch group, act_dim 1 and kMaxAct, the
widest chain input, single-layer and CH_MAXL-deep nets, batch 1 / 2048 and both sides of the split-K threshold.

Every case first proves which plan it landed on (the launch labels of a throwaway handle), then runs two steps with the
CUDA step's ReLU / tanh / min-routing decisions forced into the oracle (tests/_golden.py::kink_checked_step) and checks the
losses, d(action), d(mu|log_std), min(Q1, Q2), the whole optimizer state and the step counters at the parity tolerance."""
import re

import pytest
import torch

import sac_port as sp
from _golden import REL, check_port_state, core_config, cuda_relu_masks, kink_checked_step, rel_l2, rel_scalar

pytestmark = pytest.mark.gpu

LL = dict(state_dim=8, act_dim=2, actor_hidden=[256, 256], critic_hidden=[256, 256])
VS = dict(state_dim=39, act_dim=4, actor_hidden=[400, 400, 400], critic_hidden=[400, 400, 400])
GENERIC_ODD = dict(state_dim=13, act_dim=3, actor_hidden=[37, 255], critic_hidden=[257, 33], batch=77)

# (id, SacSpec kwargs, precision, env, plan the case must land on).  An odd batch leaves a partial last CTA at every rows-per-CTA
# choice (2, 4, 8) of the chain launches.
CASES = [
    ("ll-ragged", dict(LL, batch=253), 0, {}, "chain2"),
    ("b1", dict(state_dim=8, act_dim=2, actor_hidden=[64, 64], critic_hidden=[64, 64], batch=1), 0, {}, "chain2"),
    ("odd-small", dict(state_dim=5, act_dim=3, actor_hidden=[36, 20], critic_hidden=[28, 44], batch=37), 0, {}, "chain2"),
    ("deep-critic", dict(state_dim=11, act_dim=3, actor_hidden=[64, 64], critic_hidden=[32, 48, 64, 40, 24], batch=90), 0, {},
     "chain"),
    ("deepest", dict(state_dim=6, act_dim=2, actor_hidden=[24] * 8, critic_hidden=[28] * 8, batch=45), 0, {}, "chain"),
    ("single-layer", dict(state_dim=7, act_dim=2, actor_hidden=[4], critic_hidden=[8], batch=50), 0, {}, "chain2"),
    ("act8-wide", dict(state_dim=244, act_dim=8, actor_hidden=[256, 256], critic_hidden=[256, 256], batch=64), 0, {}, "chain2"),
    ("act1", dict(state_dim=3, act_dim=1, actor_hidden=[12, 12], critic_hidden=[12, 12], batch=33), 0, {}, "chain2"),
    ("mt-ragged", dict(state_dim=39, num_tasks=7, weighted_loss=True, act_dim=4, actor_hidden=[40, 40], critic_hidden=[40, 40],
                       batch=91), 0, {}, "chain2"),
    ("max-batch", dict(LL, batch=2048), 0, {}, "chain2"),
    ("generic-odd-p0", GENERIC_ODD, 0, {}, "ffma"),
    ("generic-odd-p1", GENERIC_ODD, 1, {}, "ffma"),
    # critic layer 1 is 21 wide (< 32 outputs: not tcgen05-eligible) while the actor's layer 1 is: the layer-1 forward group
    # is one tcgen05 launch + one FFMA launch
    ("tc-mixed", dict(state_dim=39, act_dim=4, actor_hidden=[400, 400], critic_hidden=[400, 21, 400], batch=301), 1, {}, "mixed"),
    ("splitk-511", dict(VS, batch=511), 1, {}, "tc"),
    ("splitk-513", dict(VS, batch=513), 1, {}, "tc"),
    # M = 31 < 32 keeps every batch-dimension problem on FFMA; the actor's forward (M = 2B = 62) stays on tcgen05
    ("tc-tiny-batch", dict(VS, batch=31), 1, {}, "mixed"),
]
BY_ID = {c[0]: c for c in CASES}

CHAIN2_LABELS = ("chain_fwd{actor,q1,q2}", "chain2{qt->y->bwd q}", "chain2{q(s,a~)->min->bwd->d(action)}", "chain_bwd{actor}")
CHAIN_LABELS = ("chain_fwd{actor,q1,q2}", "chain_fwd{qt1,qt2}", "chain_bwd{q1,q2}", "chain_fwd{q1,q2}(s,a~)",
                "chain_bwd{q1,q2}->d(action)", "chain_bwd{actor}")


@pytest.fixture(scope="module")
def cuda():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    from distributed_sac_b200 import _lib
    _lib.load()
    return torch.device("cuda", 0)


def plan_labels(cfg, env):
    """Launch labels of one step of a throwaway handle created with `cfg` under `env` (the plan is fixed at create time)."""
    from distributed_sac_b200.core import Replay, SacCore
    with pytest.MonkeyPatch.context() as mp:
        for k, v in env.items():
            mp.setenv(k, v)
        core = SacCore(cfg, 0, seed=0)
        ring = Replay(core, 8 * cfg.batch)
        ring.fill_synthetic(8 * cfg.batch)
        labels = [name for name, _ in core.profile_step(ring, 1)]
        ring.close()
        core.close()
    return labels


def check_plan(labels, plan, spec):
    gemm = [l for l in labels if l.startswith("gemm_")]
    if plan == "chain2":
        assert all(l in labels for l in CHAIN2_LABELS) and not gemm and "chain_bwd{q1,q2}" not in labels, labels
    elif plan == "chain":
        assert all(l in labels for l in CHAIN_LABELS) and not gemm, labels
        assert not any(l.startswith("chain2{") for l in labels), labels
    else:
        assert not any(l.startswith(("chain", "wgrad")) for l in labels) and "policy_head" in labels, labels
        tc = [l for l in gemm if "tcgen05" in l]
        assert bool(tc) == (plan != "ffma"), labels
        if plan == "mixed":
            # the forward pass over [s';s] and (s,a) is one launch group per layer; a group whose problems go to both
            # engines becomes a tcgen05 launch plus an FFMA launch, so there are more forward launches than layers
            fwd = [l for l in labels[:labels.index("policy_head")] if l.startswith("gemm_fwd")]
            assert len(fwd) > max(len(spec.actor_hidden), len(spec.critic_hidden)), labels


def actor_pass(spec, p_before, p_after, s, eps, forced):
    """d(action), d(mu|log_std) and min(Q1, Q2) of the step's actor pass by autograd, under the masks the CUDA step used: the
    policy at the pre-step actor and temperature, the critics after their update (LL/learner.py:218-225).  The head bias
    is expanded to one row per sample so that its gradient is d(head output) row by row."""
    B, A = s.shape[0], spec.act_dim
    p = {k: (p_before if k.startswith("actor.") else p_after)[k] for k in p_after}
    head = f"actor.{len(spec.actor_hidden)}.bias"
    rowb = p[head].expand(B, 2 * A).clone().requires_grad_(True)
    p[head] = rowb
    alpha = p_before["log_alpha"][sp.task_ids(spec, s)].exp().unsqueeze(1)
    div = float(B) if spec.weighted_loss else 1.0
    with sp.ReluTape(forced):
        act, logp, _ = sp.policy_sample(spec, p, s, eps, "cur")
        a = act.detach().requires_grad_(True)
        x = torch.cat([s, a], -1)
        qmin = sp.min_tagged(sp.mlp(p, "q1", x, "pi"), sp.mlp(p, "q2", x, "pi"), "route:pi")
        (d_action,) = torch.autograd.grad(torch.mean(-qmin) / div, a)
        (d_head,) = torch.autograd.grad((act * d_action).sum() + torch.mean(alpha * logp) / div, rowb)
    return d_action, d_head, qmin.detach()


def run_parity(spec, cfg, what, steps=2):
    """`steps` steps of a fresh handle, each from the port's state, against the port with the CUDA decisions forced.
    Returns (core, port, [losses of each step])."""
    from distributed_sac_b200.core import SacCore
    port = sp.PortLearner(spec, sp.init_params(spec, seed=3))
    core = SacCore(cfg, 0, seed=0)
    gen = torch.Generator().manual_seed(77)
    B, A = spec.batch, spec.act_dim
    losses = []
    for i in range(steps):
        b = sp.synthetic_batch(spec, seed=100 + i)
        e1, e2 = torch.randn(B, A, generator=gen), torch.randn(B, A, generator=gen)
        before = port.params()
        o, flips = kink_checked_step(core, port, spec, b, e1, e2)
        L = core.read_losses(1)[0, 0]
        assert rel_scalar(float(L[0]), o["critic_loss"]) <= REL, (what, i, "critic_loss", float(L[0]), o["critic_loss"])
        assert rel_scalar(float(L[1]), o["actor_loss"]) <= REL, (what, i, "actor_loss", float(L[1]), o["actor_loss"])
        assert rel_scalar(float(L[3]), o["entropy"]) <= REL, (what, i, "entropy", float(L[3]), o["entropy"])
        d_action, d_head, qmin = actor_pass(spec, before, port.params(), b[0], e2, cuda_relu_masks(core, spec))
        for name, got, ref in (("d_action", core.debug("d_action").reshape(B, A), d_action),
                               ("d_head", core.debug("d_head").reshape(B, 2 * A), d_head),
                               ("qmin", core.debug("qmin").reshape(B, 1), qmin)):
            assert rel_l2(got, ref) <= REL, (what, i, name, rel_l2(got, ref))
        check_port_state(core, port)
        assert core.get_steps() == port.adam_state()["step"], (what, i)
        print(f"[kinks] {what} step {i}: {sum(flips.values())} mask bits differed, all at numerically-zero pre-activations")
        losses.append(L.clone())
    return core, port, losses


def check_act(core, port, spec):
    """b200sac_act at 1, B and 2B rows (the policy head at this act_dim and a ragged last group of 8 rows)."""
    p = port.params()
    core.set_named(p)
    B, A = spec.batch, spec.act_dim
    g = torch.Generator().manual_seed(4)
    obs = sp.synthetic_batch(spec, seed=300, batch=2 * B)[0]
    for n in sorted({1, B, 2 * B}):
        eps = torch.randn(n, A, generator=g)
        ref, _, _ = sp.policy_sample(spec, p, obs[:n], eps)
        assert rel_l2(core.act(obs[:n], eps=eps), ref) <= REL, ("act", n)
        det, _, _ = sp.policy_sample(spec, p, obs[:n], torch.zeros(n, A))
        assert rel_l2(core.act(obs[:n], stochastic=False), det) <= REL, ("act, stochastic=False", n)


@pytest.mark.parametrize("cid,kw,precision,env,plan", CASES, ids=[c[0] for c in CASES])
def test_step_at_shape_edge_matches_port(cuda, monkeypatch, cid, kw, precision, env, plan):
    spec = sp.SacSpec(**kw)
    cfg = core_config(spec, precision=precision)
    check_plan(plan_labels(cfg, env), plan, spec)
    for k, v in env.items():
        monkeypatch.setenv(k, v)
    core, port, _ = run_parity(spec, cfg, cid)
    check_act(core, port, spec)
    core.close()


@pytest.mark.parametrize("cid", ["ll-ragged", "odd-small", "deep-critic"])
def test_chain_rows_per_cta_are_bit_identical(cuda, monkeypatch, cid):
    """Forced 2, 4 and 8 rows per CTA: each follows the port, and the three agree bit for bit -- the K split across warps,
    the warp-order reduction and every per-row head / tail are independent of the row count, and wgrad never sees it."""
    from distributed_sac_b200 import _lib
    _, kw, precision, _, plan = BY_ID[cid]
    spec = sp.SacSpec(**kw)
    cfg = core_config(spec, precision=precision)
    runs = []
    for rows in ("2", "4", "8"):
        env = {"B200SAC_CHAIN_ROWS": rows}
        check_plan(plan_labels(cfg, env), plan, spec)
        monkeypatch.setenv("B200SAC_CHAIN_ROWS", rows)
        core, _, losses = run_parity(spec, cfg, f"{cid} rows {rows}")
        runs.append((torch.stack(losses), [core.export_arena(w) for w in (_lib.PARAMS, _lib.ADAM_M, _lib.ADAM_V)]))
        core.close()
    for losses, arenas in runs[1:]:
        assert torch.equal(losses, runs[0][0])
        assert all(torch.equal(a, b) for a, b in zip(arenas, runs[0][1]))


VARIANTS = ([(cid, {"B200SAC_NO_CLUSTER": "1"}, "chain") for cid in ("ll-ragged", "odd-small")] +
            [(cid, {"B200SAC_FUSE": "0"}, "ffma") for cid in ("ll-ragged", "odd-small", "deep-critic")])


@pytest.mark.parametrize("cid,env,plan", VARIANTS, ids=[f"{c}-{next(iter(e))}" for c, e, _ in VARIANTS])
def test_forced_plan_at_shape_edge_matches_port(cuda, monkeypatch, cid, env, plan):
    """The unclustered chain path at the shallow shapes and the generic FFMA plan at the chain shapes."""
    _, kw, precision, _, _ = BY_ID[cid]
    spec = sp.SacSpec(**kw)
    cfg = core_config(spec, precision=precision)
    check_plan(plan_labels(cfg, env), plan, spec)
    for k, v in env.items():
        monkeypatch.setenv(k, v)
    core, _, _ = run_parity(spec, cfg, f"{cid} {env}")
    core.close()


@pytest.mark.parametrize("batch", [511, 513])
def test_split_k_slices_at_the_threshold(cuda, capfd, batch):
    """Below 512 rows every weight gradient reduces the whole batch in one problem; from 512 on it is cut into K slices
    of a multiple of 32 rows and a short last slice (the tcgen05 problem list the plan builder prints, B200SAC_PLAN_DBG)."""
    spec = sp.SacSpec(**dict(VS, batch=batch))
    capfd.readouterr()
    plan_labels(core_config(spec, precision=1), {"B200SAC_PLAN_DBG": "1"})
    ks = [int(k) for k in re.findall(r"\bW\d+x\d+x(\d+)", capfd.readouterr().err)]
    assert ks, "no weight-gradient problem in the tcgen05 plan dump"
    if batch < 512:
        assert set(ks) == {batch}, ks
    else:                  # (the split factor is per launch group, picked by the tcgen05 cost model; 1 is among the choices)
        assert any(k < batch and k % 32 for k in ks), ks
