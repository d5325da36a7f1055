"""CPU: host-side logic that needs no GPU -- the C-ABI library loads and exports every symbol the
header declares, the parameter layout, cfg decoding, reference key maps."""
import ctypes as C
import json
import os
import re

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def lib():
    import __graft_entry__ as ge
    ge.build()
    from distributed_sac_b200 import _lib
    return _lib.load()


def test_library_exports_every_declared_symbol(lib):
    from distributed_sac_b200 import _lib
    hdr = open(os.path.join(ROOT, "include", "b200sac.h")).read()
    declared = set(re.findall(r"\b(b200sac_[a-z0-9_]+)\s*\(", hdr))
    assert declared, "no declarations parsed"
    for name in sorted(declared):
        assert hasattr(lib, name), f"{name} declared in include/b200sac.h but not exported"
    assert declared == set(_lib.SYMBOLS), (declared ^ set(_lib.SYMBOLS))
    assert b"b200sac" in lib.b200sac_version()


def test_layout_matches_reference_parameter_counts(lib):
    from distributed_sac_b200.core import CoreConfig, layout
    t, arena, train = layout(CoreConfig())                     # LunarLander: SURVEY 8(a) a11/a12
    n = lambda pre: sum(r * c for k, (o, r, c, tr, opt, pitch) in t.items() if k.startswith(pre))
    assert n("actor.") == 69124 and n("q1.") == 68865 and n("q1_target.") == 68865
    assert n("actor.") + n("q1.") + n("q2.") + 1 == 206855
    assert t["actor.2.weight"][1:3] == (4, 256) and t["q1.0.weight"][1:3] == (256, 10)
    assert all(off % 4 == 0 for off, *_ in t.values())          # 16-byte aligned tensors (TMA / float4)
    assert t["q1.0.weight"][5] == 12 and t["actor.0.weight"][5] == 8 and t["q1.1.weight"][5] == 256   # padded first-layer pitch
    assert train < arena and t["log_alpha"][3] == 1 and t["q2_target.2.bias"][3] == 0
    t, arena, train = layout(CoreConfig(state_dim=39, act_dim=4, actor_hidden=[400] * 3, critic_hidden=[400] * 3,
                                        batch=1280, num_tasks=10))
    assert n("actor.") == 344008 and n("q1.") == 342801 and t["log_alpha"][1] == 10


def test_layout_rejects_bad_configs(lib):
    from distributed_sac_b200.core import CoreConfig, layout
    for bad in (dict(act_dim=0), dict(act_dim=9), dict(batch=0), dict(batch=4096), dict(num_tasks=3, batch=256),
                dict(actor_hidden=[]), dict(replicas=0), dict(precision=7)):
        with pytest.raises(RuntimeError, match="b200sac error"):
            layout(CoreConfig(**bad))


def test_cfg_decoder_and_key_maps(tmp_path):
    from distributed_sac_b200 import names
    from distributed_sac_b200.learner import cfg_read
    p = tmp_path / "c.json"
    p.write_text(json.dumps({"batch_size": "256", "device": "cuda", "nested": {"x": ["7", "a"]}, "lr": 3e-4}))
    c = cfg_read(str(p))
    assert c["batch_size"] == 256 and c["nested"]["x"] == [7, "a"] and c["device"] == "cuda" and c["lr"] == 3e-4
    assert names.actor_key_map("LL", 3) == {
        "layer_intermediate.0.weight": "actor.0.weight", "layer_intermediate.0.bias": "actor.0.bias",
        "layer_intermediate.1.weight": "actor.1.weight", "layer_intermediate.1.bias": "actor.1.bias",
        "mu_log_std_layer.weight": "actor.2.weight", "mu_log_std_layer.bias": "actor.2.bias"}
    assert names.critic_key_map("MS", 4, 2, True)["Q_function_2.6.bias"] == "q2_target.3.bias"
    assert names.critic_key_map("VS", 4, 1)["layer_module.2.weight"] == "q1.3.weight"


def test_product_fails_loudly_without_cuda(monkeypatch):
    import torch
    monkeypatch.setattr(torch.cuda, "is_available", lambda: False)      # a host with a GPU checks the same guard
    from distributed_sac_b200.core import CoreConfig, SacCore
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        SacCore(CoreConfig())


def test_publication_ranges_and_unpack_without_a_gpu():
    """Host side of the publication path (core.publish_begin / publish_wait): adjacent tensors are merged into one copy range,
    padded first-layer pitches and the (K,in,out) mixture layout are undone, and every returned tensor owns its memory."""
    import ctypes as C
    import numpy as np
    from distributed_sac_b200.core import CoreConfig, SacCore, layout

    cfg = CoreConfig(state_dim=39, act_dim=4, actor_hidden=[16, 12], critic_hidden=[16, 12], batch=60, num_tasks=10, care=True,
                     num_encoders=3, mix_hidden=[8], mix_out=6, ctx_in=20, ctx_hidden=[7], ctx_out=5)
    table, arena, _trainable = layout(cfg)
    flat = np.arange(arena, dtype=np.float32)

    calls = {}

    class StubLib:
        def b200sac_publish_begin(self, h, replica, n, offs, cnts, stream):
            calls["ranges"] = [(offs[i], cnts[i]) for i in range(n)]
            return 0

        def b200sac_publish_wait(self, h, ptr, n):
            packed = np.concatenate([flat[o:o + c] for o, c in calls["ranges"]])
            calls["buf"] = packed                                   # keep alive
            C.cast(ptr, C.POINTER(C.POINTER(C.c_float)))[0] = packed.ctypes.data_as(C.POINTER(C.c_float))
            C.cast(n, C.POINTER(C.c_int64))[0] = packed.size
            return 0

    core = object.__new__(SacCore)
    core.lib, core._h, core.cfg, core.table = StubLib(), None, cfg, table
    import distributed_sac_b200.core as core_mod
    real_stream = core_mod._stream
    core_mod._stream = lambda: None
    try:
        names = [n for n in table if n.startswith("actor.")] + [n for n in table if n.startswith("cse.")]
        core.publish_begin(names)
        got = core.publish_wait()
    finally:
        core_mod._stream = real_stream
    # actor and cse blocks are each contiguous, and q1/q2 lie between them: exactly two ranges
    assert len(calls["ranges"]) == 2
    assert set(got) == set(names)
    for n, t in got.items():
        off, rows, cols, _tr, _opt, pitch = table[n]
        ref = flat[off:off + rows * pitch].reshape(rows, pitch)[:, :cols]
        if ".mix." in n and n.endswith(".W"):
            K = cfg.num_encoders
            assert t.shape == (K, cols, rows // K)
            assert np.array_equal(t.numpy(), ref.reshape(K, rows // K, cols).transpose(0, 2, 1))
        elif ".mix." in n:
            assert t.shape == (cfg.num_encoders, 1, rows // cfg.num_encoders)
        else:
            assert np.array_equal(t.numpy().reshape(rows, cols), ref)
        assert t.numpy().base is None or not np.shares_memory(t.numpy(), calls["buf"])
    w0 = table["actor.0.weight"]
    assert w0[5] >= w0[2] and w0[5] % 4 == 0                       # padded pitch of the first layer is hidden from the caller


class BlobStubLib:
    """CPU stand-in for b200sac_blob_*: emulates the device gather (payload float j = arena[src[j]] -> image bytes at dst[j])."""

    def __init__(self, arena):
        self.arena = arena

    def b200sac_blob_template(self, h, replica, image, image_bytes, n_floats, src, dst):
        import ctypes as C
        import numpy as np
        self.image = np.ctypeslib.as_array(C.cast(image, C.POINTER(C.c_uint8)), shape=(image_bytes,)).copy()
        self.src = np.ctypeslib.as_array(C.cast(src, C.POINTER(C.c_int32)), shape=(n_floats,)).copy()
        self.dst = np.ctypeslib.as_array(C.cast(dst, C.POINTER(C.c_int32)), shape=(n_floats,)).copy()
        return 0

    def b200sac_blob_begin(self, h, stream):
        import numpy as np
        out = self.image.copy()
        vals = np.ascontiguousarray(self.arena[self.src], dtype=np.float32).view(np.uint8).reshape(-1, 4)
        for b in range(4):
            out[self.dst + b] = vals[:, b]
        self.out = out
        return 0

    def b200sac_blob_wait(self, h, ptr, n):
        import ctypes as C
        C.cast(ptr, C.POINTER(C.c_void_p))[0] = self.out.ctypes.data
        C.cast(n, C.POINTER(C.c_int64))[0] = self.out.size
        return 0


def test_parameters_blob_device_image_round_trips():
    """Learner.parameters_blob(): the pickle stream is built once from tensors of the published shapes and registered as a byte
    image + index maps (core.blob_template); a publication only gathers arena floats into the payload positions.  With the
    gather emulated on the CPU, unpickling must give exactly what a plain pickle.dumps of the state_dict gives -- through the
    padded first-layer pitch and the CARE (K,in,out) mixture layout."""
    import pickle
    import numpy as np
    import torch
    import distributed_sac_b200.core as core_mod
    from distributed_sac_b200 import names
    from distributed_sac_b200.core import CoreConfig, SacCore, layout
    from distributed_sac_b200.learner import _BaseLearner

    cfg = CoreConfig(state_dim=39, act_dim=4, actor_hidden=[16, 12], critic_hidden=[16, 12], batch=60, num_tasks=10, care=True,
                     num_encoders=3, mix_hidden=[8], mix_out=6, ctx_in=20, ctx_hidden=[7], ctx_out=5)
    table, arena, _trainable = layout(cfg)
    rng = np.random.default_rng(0)
    flat = rng.standard_normal(arena).astype(np.float32)
    core = object.__new__(SacCore)
    core.lib, core._h, core.cfg, core.table = BlobStubLib(flat), None, cfg, table
    lrn = _BaseLearner.__new__(_BaseLearner)
    lrn.core = core
    lrn._published = ("actor", "cse")
    km = {"actor": {f"ref.{n}": n for n in table if n.startswith("actor.")},
          "cse": {f"ref.{n}": n for n in table if n.startswith("cse.")}}
    lrn._key_map = lambda net: km[net]
    real_stream = core_mod._stream
    core_mod._stream = lambda: None
    try:
        for rnd in range(3):
            flat[:] = rng.standard_normal(arena).astype(np.float32)
            if rnd == 1:
                flat[:] = 0.0                                       # all-zero payloads must not confuse the template
            blob = lrn.parameters_blob(blocking=True)
            got = pickle.loads(blob)
            assert set(got) == {"actor", "cse"}
            for net, m in km.items():
                assert set(got[net]) == set(m)
                for ref, canon in m.items():
                    off, rows, cols, _tr, _opt, pitch = table[canon]
                    want = core._view(canon, flat, off)
                    t = got[net][ref]
                    assert isinstance(t, torch.Tensor) and t.dtype == torch.float32 and tuple(t.shape) == want.shape, (canon, t.shape, want.shape)
                    assert np.array_equal(t.numpy(), want), canon
            plain = pickle.loads(pickle.dumps({net: {ref: torch.from_numpy(np.ascontiguousarray(core._view(c_, flat, table[c_][0])))
                                                     for ref, c_ in m.items()} for net, m in km.items()}))
            assert all(torch.equal(plain[net][k], got[net][k]) for net in km for k in km[net])
            _blob, extra = core.blob_wait()                          # (the stub keeps the last image) the logger's temperature
            assert np.array_equal(extra["log_alpha"], flat[table["log_alpha"][0]:table["log_alpha"][0] + table["log_alpha"][1]])
    finally:
        core_mod._stream = real_stream
    mixw = [n for n in table if ".mix." in n and n.endswith(".W")]
    assert mixw and table["actor.0.weight"][5] > table["actor.0.weight"][2]      # both layout twists were exercised
