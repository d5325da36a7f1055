"""CPU: the oracle ports and the host-side wire formats against the UNMODIFIED reference, live (what needs the reference's
code is skipped where no checkout of it is reachable).

* oracle/sac_port.py / care_port.py reproduce the reference learner's update() step for step (the committed fixtures under
  tests/golden/ are frozen outputs of the same comparison; this test re-derives them from the code in front of us);
* the bytes Learner.run() publishes (Learner.parameters_blob: a pickle stream built once whose float payloads the library gathers from the arena) hold
  exactly the Actor state_dict the reference itself wrote, as its load_state_dict takes it -- what Player.pull_parameters does (LL/player.py:75-85);
* a checkpoint written by the drop-in learner's save path (reference-written fixtures round-tripped on the GPU side, see
  tests/test_gpu_checkpoint.py) has the key set the reference's load_checkpoint() reads."""
import pickle

import numpy as np
import pytest
import torch

import ref_harness as rh
import sac_port as sp
from _golden import rel_l2, rel_scalar

needs_reference = pytest.mark.skipif(not rh.available(), reason="no checkout of the reference (B200SAC_REFERENCE, baseline/_ref)")


def _set(named, params):
    with torch.no_grad():
        for k, p in named.items():
            p.data.copy_(params[k].reshape(p.shape))


@needs_reference
@pytest.mark.parametrize("family,overrides", [
    ("LL", dict(batch_size=64)),
    ("MS", dict(batch_size=60, actor=dict(actor_hidden_dim=[32, 48]), critic=dict(critic_hidden_dim=[40, 24]))),
])
def test_port_follows_the_live_reference(family, overrides):
    import gen_golden as gg
    lrn, _ = rh.make_learner(family, overrides, seed=3)
    spec = gg._spec_of(lrn, family, family == "MS")
    params = sp.init_params(spec, seed=5)
    named = gg._named_params(lrn, family)
    _set(named, params)
    port = sp.PortLearner(spec, params)
    g = torch.Generator().manual_seed(1)
    for i in range(4):
        b = sp.synthetic_batch(spec, seed=300 + i)
        e1, e2 = torch.randn(spec.batch, spec.act_dim, generator=g), torch.randn(spec.batch, spec.act_dim, generator=g)
        lrn.memory.sample = (lambda bb: (lambda: tuple(t.clone() for t in bb)))(b)
        with rh.injected_eps([e1, e2]) as q:
            res = lrn.update()
            assert not q
        o = port.update_SAC(*b, e1, e2)
        assert rel_scalar(o["critic_loss"], res[0]) <= 1e-5 and rel_scalar(o["actor_loss"], res[1]) <= 1e-5, (i, o, res)
    got = port.params()
    for k, p in named.items():
        if k == "log_alpha":
            assert (got[k] - p.detach()).abs().max().item() <= 1e-6
        else:
            assert rel_l2(got[k], p.detach()) <= 1e-5, (k, rel_l2(got[k], p.detach()))


def test_published_blob_loads_into_the_reference_actor():
    """parameters_blob() is host logic: exercised here with a stand-in core whose arena holds the Actor state the reference's
    own save_checkpoint() wrote (tests/golden/ref_ckpt_ll_small.tar).  The unpickled blob must be exactly what a strict
    Actor.load_state_dict takes and what Player.pull_parameters hands it (LL/player.py:75-85): the reference's keys in its
    order, its shapes and dtypes, and the written values bit for bit."""
    import os
    import __graft_entry__ as ge
    ge.build()                                                    # layout() reads the library's parameter table
    from distributed_sac_b200 import names
    from distributed_sac_b200.learner import _BaseLearner
    from _golden import GOLDEN
    sd = torch.load(os.path.join(GOLDEN, "ref_ckpt_ll_small.tar"), map_location="cpu", weights_only=False)["actor"]
    km = names.actor_key_map("LL", 3)

    # stand-in core: the arena of a LunarLander learner filled with the reference-written Actor state; the device gather of
    # b200sac_blob_* is emulated on the CPU (tests/test_host_logic.py::BlobStubLib)
    import distributed_sac_b200.core as core_mod
    from distributed_sac_b200.core import CoreConfig, SacCore, layout
    from test_host_logic import BlobStubLib
    cfg = CoreConfig(batch=64)
    table, arena, _tr = layout(cfg)
    flat = np.zeros(arena, np.float32)
    core = object.__new__(SacCore)
    core.lib, core._h, core.cfg, core.table = BlobStubLib(flat), None, cfg, table
    for ref, canon in km.items():
        off, rows, cols, _t, _o, pitch = table[canon]
        flat[off:off + rows * pitch].reshape(rows, pitch)[:, :cols] = sd[ref].numpy().reshape(rows, cols)
    shim = _BaseLearner.__new__(_BaseLearner)
    shim.core = core
    shim._key_map = lambda net: km
    real_stream = core_mod._stream
    core_mod._stream = lambda: None
    try:
        blob = shim.parameters_blob()
    finally:
        core_mod._stream = real_stream
    params = pickle.loads(blob)                                   # Player.pull_parameters: _pickle.loads(server.get('parameters'))
    got = params["actor"]
    assert list(got) == list(sd)                                  # strict load_state_dict: every key, no extra
    for k, v in sd.items():
        assert isinstance(got[k], torch.Tensor) and got[k].dtype == v.dtype and got[k].shape == v.shape, (k, got[k].shape, v.shape)
        assert torch.equal(got[k], v), k


def test_reference_load_checkpoint_reads_the_keys_we_write():
    """Key sets of the reference-written fixtures == what each reference load_checkpoint() indexes (LL/learner.py:165-182,
    MS:176-190, C10:200-217); tests/test_gpu_checkpoint.py proves the drop-in learner writes exactly these trees."""
    import os
    from _golden import GOLDEN
    want = {
        "ref_ckpt_ll_small": {"episode_idx", "total_step", "local_critic_1", "local_critic_2", "critic_optimizer", "target_critic_1",
                              "target_critic_2", "actor", "actor_optimizer", "log_alpha", "log_alpha_optimizer", "alpha"},
        "ref_ckpt_ms_small": {"update_iteration", "total_step", "local_critic", "critic_optimizer", "target_critic", "actor",
                              "actor_optimizer", "log_alpha", "log_alpha_optimizer", "alpha"},
        "ref_ckpt_c10m_small": {"update_iteration", "total_step", "context_encoder", "context_encoder_optimizer", "local_critic",
                                "critic_optimizer", "target_critic", "actor", "actor_optimizer", "log_alpha", "log_alpha_optimizer", "alpha"},
    }
    for name, keys in want.items():
        ck = torch.load(os.path.join(GOLDEN, name + ".tar"), map_location="cpu", weights_only=False)
        assert set(ck) == keys, (name, set(ck) ^ keys)


@needs_reference
def test_reference_modules_accept_the_checkpoint_fixture():
    """The reference's own modules accept the reference-written fixture's state_dicts (the format is theirs)."""
    import os
    from _golden import GOLDEN
    lrn, _ = rh.make_learner("LL", dict(batch_size=64), seed=1)
    ck = torch.load(os.path.join(GOLDEN, "ref_ckpt_ll_small.tar"), map_location="cpu", weights_only=False)
    lrn.actor.load_state_dict(ck["actor"])
    lrn.local_critic_1.load_state_dict(ck["local_critic_1"])
    lrn.critic_optimizer.load_state_dict(ck["critic_optimizer"])
    assert int(lrn.critic_optimizer.state_dict()["state"][0]["step"]) == 2


def _shipped(rel):
    import os
    p = os.path.join(rh.REF_ROOT, "saved_models", rel)
    if not os.path.exists(p):
        pytest.skip(f"shipped checkpoint {rel} not in this checkout")
    return p


@needs_reference
def test_port_follows_the_reference_from_the_shipped_mtsac_checkpoint():
    """Full-size MTSAC (49/4, 400^3, B 1280, weighted loss) started from the reference's own trained checkpoint INCLUDING its
    Adam moments and step counts (saved_models/MT10_Distributed_MTSAC/checkpoint_3300000.tar, loaded the way the reference's
    load_checkpoint intends, MS/learner.py:176-190): two update() calls of the unmodified learner against the port."""
    import gen_golden as gg
    path = _shipped("MT10_Distributed_MTSAC/checkpoint_3300000.tar")
    lrn, _ = rh.make_learner("MS", None, seed=0)
    ck = torch.load(path, map_location="cpu", weights_only=False)
    lrn.local_critic.load_state_dict(ck["local_critic"]); lrn.critic_optimizer.load_state_dict(ck["critic_optimizer"])
    lrn.target_critic.load_state_dict(ck["target_critic"])
    lrn.actor.load_state_dict(ck["actor"]); lrn.actor_optimizer.load_state_dict(ck["actor_optimizer"])
    lrn.log_alpha.data = ck["log_alpha"].data.clone(); lrn.log_alpha_optimizer.load_state_dict(ck["log_alpha_optimizer"])
    weighted = bool(getattr(lrn, "use_weighted_loss", True))
    spec = gg._spec_of(lrn, "MS", weighted)
    named = gg._named_params(lrn, "MS")
    params = {k: p.detach().clone() for k, p in named.items()}
    m, v, step = gg._adam_snapshot(lrn, named, spec)
    assert int(step[0]) > 1000 and int(step[1]) > 1000              # a trained state: the bias corrections are ~1
    port = sp.PortLearner(spec, params, adam_state={"m": m, "v": v, "step": tuple(int(x) for x in step)})
    g = torch.Generator().manual_seed(11)
    for i in range(2):
        b = sp.synthetic_batch(spec, seed=900 + i)
        e1, e2 = torch.randn(spec.batch, spec.act_dim, generator=g), torch.randn(spec.batch, spec.act_dim, generator=g)
        lrn.memory.sample = (lambda bb: (lambda: tuple(t.clone() for t in bb)))(b)
        with rh.injected_eps([e1, e2]) as q:
            res = lrn.update()
            assert not q
        o = port.update_SAC(*b, e1, e2)
        assert rel_scalar(o["critic_loss"], res[0]) <= 1e-5 and rel_scalar(o["actor_loss"], res[1]) <= 1e-5, (i, o, res)
    got, st = port.params(), port.adam_state()
    m2, v2, step2 = gg._adam_snapshot(lrn, named, spec)
    assert tuple(st["step"]) == tuple(int(x) for x in step2)
    for k, p in named.items():
        if k == "log_alpha":
            assert (got[k] - p.detach()).abs().max().item() <= 1e-6
            continue
        assert rel_l2(got[k], p.detach()) <= 1e-5, (k, rel_l2(got[k], p.detach()))
        if k in m2 and "_target" not in k:
            assert rel_l2(st["m"][k], m2[k]) <= 1e-4 and rel_l2(st["v"][k], v2[k]) <= 1e-4, k


@needs_reference
def test_care_port_follows_the_reference_from_a_shipped_care_checkpoint():
    """The same for CARE(M) at its configured shape (B 1280, K 6, 768-d task embeddings) from
    saved_models/MT10_Distributed_CARE/CARE(M)/checkpoint_6300000.tar with its optimizer states (C10/learner.py:200-217)."""
    import care_port as cp
    import gen_golden as gg
    path = _shipped("MT10_Distributed_CARE/CARE(M)/checkpoint_6300000.tar")
    lrn, _ = rh.make_learner("C10", dict(use_modified_care=True), seed=0)
    ck = torch.load(path, map_location="cpu", weights_only=False)
    lrn.context_encoder.load_state_dict(ck["context_encoder"])
    lrn.local_critic.load_state_dict(ck["local_critic"]); lrn.critic_optimizer.load_state_dict(ck["critic_optimizer"])
    lrn.target_critic.load_state_dict(ck["target_critic"])
    lrn.actor.load_state_dict(ck["actor"]); lrn.actor_optimizer.load_state_dict(ck["actor_optimizer"])
    lrn.log_alpha.data = ck["log_alpha"].data.clone(); lrn.log_alpha_optimizer.load_state_dict(ck["log_alpha_optimizer"])
    spec = cp.CareSpec(modified=True, weighted_loss=True)
    named = gg._care_named(lrn)
    params = {k: p.detach().clone() for k, p in named.items()}
    # the actor's own state encoder: the reference ties it to the critic's at the end of every update (learner.py:402), so the
    # checkpoint holds equal copies; the port keeps one
    ase, cse = dict(lrn.actor.state_encoder.named_parameters()), dict(lrn.local_critic.state_encoder.named_parameters())
    assert all(torch.equal(ase[k], cse[k]) for k in ase)
    port = cp.CarePortLearner(spec, params)
    opts = {"critic": lrn.critic_optimizer, "actor": lrn.actor_optimizer, "alpha": lrn.log_alpha_optimizer}
    mm, vv, steps = {}, {}, [0, 0, 0]
    for k in port.trainable_names():
        tag, slot = ("alpha", 2) if k == "log_alpha" else (("actor", 1) if k.startswith("actor.") else ("critic", 0))
        stt = opts[tag].state[named[k]]
        mm[k], vv[k] = stt["exp_avg"].clone(), stt["exp_avg_sq"].clone()
        steps[slot] = int(stt["step"])
    assert steps[0] > 1000
    port.load_adam({"m": mm, "v": vv, "step": tuple(steps)})
    g = torch.Generator().manual_seed(13)
    for i in range(2):
        b = cp.synthetic_batch(spec, seed=950 + i)
        e1, e2 = torch.randn(spec.batch, spec.act_dim, generator=g), torch.randn(spec.batch, spec.act_dim, generator=g)
        lrn.memory.sample = (lambda bb: (lambda: tuple(t.clone() for t in bb)))(b)
        with rh.injected_eps([e1, e2]) as q:
            res = lrn.update()
            assert not q
        o = port.update(*b, e1, e2)
        assert rel_scalar(o["critic_loss"], res[0]) <= 1e-5 and rel_scalar(o["actor_loss"], res[1]) <= 1e-5, (i, o, res)
    got = port.params()
    for k, p in named.items():
        if k == "log_alpha":
            assert (got[k] - p.detach()).abs().max().item() <= 1e-6
        else:
            assert rel_l2(got[k], p.detach()) <= 1e-5, (k, rel_l2(got[k], p.detach()))
