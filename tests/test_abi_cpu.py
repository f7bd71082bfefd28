"""CPU-only checks of the C-ABI library and the host-side logic (no compute calls without a GPU)."""
import ctypes
import os
import re

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _declared_symbols():
    src = open(os.path.join(ROOT, "include", "cadre_b200.h")).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    return sorted(set(re.findall(r"\b(cadre_[a-z0-9_]+)\s*\(", src)))


def test_library_builds_and_exports_every_declared_symbol():
    import __graft_entry__
    __graft_entry__.build()
    from cadre_b200 import _lib
    lib = _lib.lib()
    syms = _declared_symbols()
    assert len(syms) >= 20
    for s in syms:
        assert hasattr(lib, s), f"{s} declared in include/cadre_b200.h but not exported"
    assert lib.cadre_version().decode().startswith("cadre_b200 sm_100a")
    assert lib.cadre_enc_dtype() in (0, 1)


def test_struct_mirrors_match_header_sizes():
    from cadre_b200 import _lib, ppo
    from cadre_b200.encoder import EncoderWeights
    # pointer-heavy structs: sizes follow from the header layout on LP64
    assert ctypes.sizeof(ppo.StorageRefC) == 9 * 8
    assert ctypes.sizeof(ppo.PpoConfigC) == 24
    assert ctypes.sizeof(EncoderWeights) == (2 + 38 + 14) * 8 + 8
    assert ctypes.sizeof(_lib.GemmArgs) % 8 == 0


def test_no_cpu_fallback():
    """Without a CUDA device every product entry point must fail loudly."""
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    from cadre_b200 import CadreError
    from cadre_b200.encoder import Encoder
    from cadre_b200.ppo import PpoEngine
    from cadre_b200.storage import RolloutStorage
    with pytest.raises(CadreError):
        Encoder({}, device="cpu")
    with pytest.raises(CadreError):
        PpoEngine(1, 4, device="cpu")
    st = RolloutStorage(8, 2, 530, 8, 530, True, 0.99, 0.95)
    with pytest.raises(CadreError):
        st.compute_returns(torch.zeros(1, 1))
    from cadre_b200.models import create_model
    with pytest.raises(CadreError):
        create_model({"device_num": -1, "vae_params": "CoPM", "measurement_dim": 18}, load_vae=False)


def test_allreduce_entry_points_validate_their_arguments():
    """cadre_allreduce_*: argument errors and a missing CUDA device come back as error codes + messages (no crash, no
    silent success); the collective wrapper refuses to work without an initialised process group."""
    from cadre_b200 import CadreError, _lib
    from cadre_b200.collective import SwitchAllReduce
    lib = _lib.lib()
    assert lib.cadre_allreduce_flag_bytes() >= 16 * 16 * 4
    h = ctypes.c_void_p()
    two = (ctypes.c_void_p * 2)(None, None)
    # world of 1, rank out of range, count not a multiple of 4 floats, null peer mappings
    for rank, world, count in ((0, 1, 1024), (2, 2, 1024), (0, 2, 1023), (0, 2, 1024)):
        rc = lib.cadre_allreduce_create(ctypes.byref(h), rank, world, two, None, two, ctypes.c_int64(count))
        assert rc != 0 and lib.cadre_last_error()
    assert lib.cadre_allreduce_sum(None, ctypes.c_int64(0), ctypes.c_int64(4), 1, None) != 0
    assert b"handle" in lib.cadre_last_error()
    assert lib.cadre_allreduce_check(None) != 0
    assert lib.cadre_allreduce_set_blocks(None, 32) != 0
    with pytest.raises(CadreError, match="process group"):
        SwitchAllReduce(1024, "cuda:0")


def test_gemm_rejects_an_empty_contraction_and_a_misaligned_fp32_mask():
    """cadre_gemm refuses, before it builds a tensor map or launches anything: K = 0, and an fp32-output ReLU-backward
    mask that the epilogue could not read as float4 rows (base not 16-byte aligned, ldm or mask_bs not a multiple of
    4). Every call also asks for the retired LSTM-cell epilogue (epi = 1), which launch_gemm rejects right after these
    checks: no call here reaches a tensor map or a launch, with or without a device, and legal masks stop there."""
    from cadre_b200 import _lib
    lib = _lib.lib()

    def call(**kw):
        a = _lib.GemmArgs()
        a.kind, a.batch, a.M, a.N, a.K, a.alpha, a.out_f32, a.epi = 1, 2, 256, 128, 128, 1.0, 1, 1
        a.A, a.B, a.out = 0x10000, 0x20000, 0x30000          # never dereferenced
        a.lda, a.ldb, a.ldc, a.a_bs, a.b_bs, a.out_bs = 128, 128, 128, 256 * 128, 128 * 128, 256 * 128
        for k, v in kw.items():
            setattr(a, k, v)
        rc = lib.cadre_gemm(ctypes.byref(a), None)
        return rc, lib.cadre_last_error().decode()

    rc, msg = call(K=0)
    assert rc != 0 and "gemm K must be positive" in msg, msg
    bad_masks = (dict(mask=0x40004, ldm=128, mask_bs=256 * 128),   # 4-byte aligned base
                 dict(mask=0x40000, ldm=130, mask_bs=256 * 130),   # ldm not a multiple of 4
                 dict(mask=0x40000, ldm=128, mask_bs=256 * 128 + 2))
    for kw in bad_masks:
        rc, msg = call(**kw)
        assert rc != 0 and "fp32 mask must be 16-byte aligned" in msg, (kw, msg)
    # legal masks pass: an aligned fp32 one, and any 16-bit mask (the epilogue reads those per element)
    for kw in (dict(mask=0x40000, ldm=128, mask_bs=256 * 128),
               dict(kind=0, out_f32=0, mask=0x40002, ldm=129, mask_bs=3)):
        rc, msg = call(**kw)
        assert rc != 0 and "LSTM-cell epilogue" in msg, (kw, msg)


def test_product_package_does_not_import_oracle():
    pkg = os.path.join(ROOT, "cadre_b200")
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h")):
                txt = open(os.path.join(dirpath, f)).read()
                assert "oracle" not in txt.replace("# oracle", ""), f"{f} references the oracle"


def test_param_layout_roundtrip_and_order():
    from cadre_b200 import ppo_params as P
    from oracle import restate as R
    sd = R.ppo_fixture_state(1)
    flat = P.pack_state(sd)
    back = P.unpack_state(flat)
    assert all(torch.equal(back[m][n], sd[m][n]) for m in sd for n in sd[m])
    assert P.MODULE_ORDER == R.PPO_MODULE_ORDER
    assert sum(t.numel() for d in sd.values() for t in d.values()) == P.NUM_REFERENCE_PARAMS == 19382808
    for m in P.MODULE_ORDER:
        assert P.module_param_names(m) == [n for n, _ in R.ppo_module_param_shapes(m)]
    # gate interleave: row 4u+g of the flat W_ih is gate g, unit u of the reference tensor
    w = sd["steer_lstm_2"]["rnn.weight_ih"]
    view, perm = P.tensor_view(flat, "steer_lstm_2", "rnn.weight_ih")
    assert perm and torch.equal(view[4 * 7 + 2], w[2 * 530 + 7])
    # offsets are 16-byte aligned (TMA) and the header constants agree
    hdr = open(os.path.join(ROOT, "cadre_b200", "csrc", "ppo_layout.h")).read()
    assert "constexpr int LDF = 532" in hdr and "constexpr int B3A_LD = 36" in hdr
    assert all(o % 4 == 0 for o in P.OFF.values())


def test_flat_module_surface():
    from cadre_b200.models import FlatParams, Shared_grad_buffers, ModelDict, get_vae_output, init_state
    from oracle import restate as R
    sd = R.ppo_fixture_state(0)
    owner = FlatParams("cpu", sd)
    md = ModelDict(owner)
    assert list(md.keys()) == R.PPO_MODULE_ORDER
    names = [n for n, _ in md["steer_ppo_0"].named_parameters()]
    assert names[0] == "control.linear.0.weight" and names[-1] == "critic.4.bias"
    assert torch.equal(md["throttle_lstm_3"].state_dict()["rnn.weight_hh"], sd["throttle_lstm_3"]["rnn.weight_hh"])
    other = FlatParams("cpu", R.ppo_fixture_state(2))
    md["steer_ppo_1"].load_state_dict(ModelDict(other)["steer_ppo_1"].state_dict())
    assert torch.equal(md["steer_ppo_1"].state_dict()["critic.4.weight"], other.state()["steer_ppo_1"]["critic.4.weight"])
    owner.grads.fill_(1.0)
    bufs = Shared_grad_buffers(md)
    bufs.add_gradient(md)
    bufs.add_gradient(md)
    assert bufs.grads.max().item() == 2.0 and bufs.count == 2       # summed, never averaged
    bufs.reset()
    assert bufs.grads.abs().max().item() == 0.0
    assert get_vae_output({"vae_params": "CoPM", "measurement_dim": 18})[0] == 530
    st = init_state(seed=3)
    w = st["steer_lstm_0"]["rnn.weight_ih"]
    assert torch.allclose(w.t() @ w, torch.eye(530), atol=1e-4)       # orthogonal init (models.py:134)
    assert st["steer_ppo_0"]["control.linear.4.weight"].abs().max() < 0.05   # gain 0.01 (distributions.py:32)


def test_storage_semantics_match_reference_quirks():
    from cadre_b200.storage import RolloutStorage
    from oracle import restate as R
    st = RolloutStorage(num_steps=6, mini_batch_num=2, feature_dims=530, seq_length=8, hidden_size=530, use_gae=True,
                        gamma=0.99, tau=0.95)
    assert st.command.dtype == torch.int32 and st.action.dtype == torch.int64 and st.obs.shape == (7, 8, 530)
    for i in range(8):          # cursor wraps modulo num_steps+1 (after_update is never called by train.py)
        st.insert(torch.full((8, 530), float(i)), torch.tensor(i), torch.tensor([[0.5]]), torch.tensor([[1.0]]),
                  torch.tensor(2.0), torch.tensor([[1.0]]), (torch.ones(1, 530), torch.ones(1, 530)), i % 4)
    assert st.step == 1 and st.obs[0, 0, 0].item() == 7.0 and st.obs[6, 0, 0].item() == 6.0
    assert st.hn[1].sum().item() == 530.0 and st.hn[0].sum().item() == 0.0
    obs, cmd = st.get_last()
    assert obs.shape == (8, 530) and cmd == 6 % 4
    torch.manual_seed(3)
    got = [mb.indices for mb in st.feed_forward_generator(torch.zeros(6, 1))]
    torch.manual_seed(3)
    assert got == R.minibatch_indices(6, 2)
    mb = next(iter(st.feed_forward_generator(torch.zeros(6, 1))))
    tup = tuple(mb)
    assert tup[0].shape == (8 * 3, 530) and tup[7][0].shape == (3, 530) and tup[8].shape == (3, 1)
    # time-major obs: row t*mb + n  (storage.py:100-104)
    assert torch.equal(tup[0][3], st.obs[mb.indices[0], 1])


def test_config_and_synthetic_env_contract():
    from cadre_b200.config import load_config
    from cadre_b200.synthetic_env import SyntheticEnv
    cfg = load_config()
    assert cfg.rollout_cfg.num_steps == 200 and cfg.rollout_cfg.feature_dims == 530 and cfg.train_cfg.lr == 3e-4
    assert cfg.agent_cfg.STEER_CONTROL[0] == -0.5 and cfg.agent_cfg.STEER_CONTROL[32] == -1.0
    assert cfg.agent_cfg.THROTTLE_CONTROL[2] == [0.6, 0] and cfg.train_cfg.max_grad_norm == 250
    env = SyntheticEnv(dict(cfg.env_cfg, rank=1))
    t = env.reset()
    assert t["rgb"].shape == (8, 144, 256, 3) and t["rgb"].dtype == np.uint8
    assert t["route_fig"].shape == (8, 256, 144) and t["measurements"].shape == (8, 3) and 0 <= t["command"] < 4
    t2, r, done, info = env.step([0.0, 0.6, 0.0])
    assert np.array_equal(t2["rgb"][:7], t["rgb"][1:]) and r.shape == (2,) and len(info["action_done"]) == 2


def test_sync_primitive_shims_keep_the_reference_interface():
    """ppo_agent/utils.py:31-70, 108-126: Counter / TrafficLight as used by train.py:101-110 and chief.py:12-24."""
    from cadre_b200.utils import Counter, TrafficLight
    c, light = Counter(), TrafficLight()
    assert c.get() == 0 and light.get() is False
    c.increment(), c.increment()
    assert c.get() == 2
    c.reset()
    assert c.get() == 0
    light.switch()
    assert light.get() is True
    light.switch()
    assert light.get() is False


def test_batched_actor_window_check_on_the_synthetic_env():
    """cadre_b200.actor.BatchedActor host logic (no GPU): the one-frame check recognises a window that slid by one
    (env_wrapper.py:900-904 semantics of SyntheticEnv.step) and rejects a reset / repeated / foreign window."""
    import numpy as np
    from cadre_b200.actor import BatchedActor
    from cadre_b200.synthetic_env import SyntheticEnv
    env, other = SyntheticEnv(dict(rank=0)), SyntheticEnv(dict(rank=1))
    actor = BatchedActor.__new__(BatchedActor)          # host-side state only
    actor.E, actor.verify_window, actor._last = 1, True, [None]

    def remember(t):
        actor._last[0] = (np.array(t["rgb"][-1], copy=True), np.array(t["route_fig"][-1], copy=True),
                          np.array(t["measurements"][-1], copy=True))
    t0 = env.reset()
    assert not actor._slid_by_one(0, t0)                # nothing seen yet
    remember(t0)
    t1, *_ = env.step([0.0, 0.0, 0.0])
    assert actor._slid_by_one(0, t1)                    # newest frame of t0 is now the second newest
    assert not actor._slid_by_one(0, t0) or np.array_equal(t0["rgb"][-2], t0["rgb"][-1])   # (reset primes 8 equal frames)
    remember(t1)
    t2, *_ = env.step([0.0, 0.0, 0.0])
    assert actor._slid_by_one(0, t2) and not actor._slid_by_one(0, t1)
    assert not actor._slid_by_one(0, other.reset())     # a different environment's window
    actor.reset(0)
    assert not actor._slid_by_one(0, t2)
