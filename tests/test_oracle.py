"""The oracle (oracle/restate.py) against (i) the committed goldens produced by the unmodified reference
(oracle/make_golden.py) and (ii) the live reference, bit for bit, when /root/reference is present."""
import os

import numpy as np
import pytest
import torch

from oracle import ref_shim, restate as R

THREADS = 8
needs_ref = pytest.mark.skipif(not ref_shim.available(), reason="reference tree not present on this box")


@pytest.fixture(autouse=True)
def _threads():
    torch.set_num_threads(THREADS)


def _load(golden_dir, name):
    return np.load(os.path.join(golden_dir, name))


# ---------------------------------------------------------------------------------------------- GAE
@pytest.mark.parametrize("i,T,seed", [(0, 200, 0), (1, 200, 1), (2, 800, 2), (3, 7, 3)])
def test_gae_matches_golden(golden_dir, i, T, seed):
    g = _load(golden_dir, "gae.npz")
    rs = np.random.RandomState(seed)
    st = R.synthetic_storage(rs, T=T, feature_dims=8, seq=1)
    if i == 1:
        st["masks"][::5] = 0.0
    returns, vp = R.compute_returns(st["rewards"], st["value_preds"], st["masks"], torch.tensor([[0.37 * (i + 1)]]))
    assert np.array_equal(returns.numpy(), g[f"returns_{i}"])          # bit-exact, same op order
    adv = R.normalized_advantages(returns, vp)
    assert np.array_equal(adv.numpy(), g[f"adv_{i}"])


# ---------------------------------------------------------------------------------------------- indices
@pytest.mark.parametrize("seed", [0, 1, 7])
def test_minibatch_indices_match_golden(golden_dir, seed):
    g = _load(golden_dir, "indices.npz")[f"idx_{seed}"]
    torch.manual_seed(seed)
    rows = []
    for _ in range(R.PPO_EPOCH):
        steer, throttle = R.minibatch_indices(), R.minibatch_indices()
        # zip() of two lazy generators: steer draws its permutation first, then throttle (train.py:94-96)
        for a, b in zip(steer, throttle):
            rows.append(np.stack([np.array(a), np.array(b)]))
    assert np.array_equal(np.stack(rows), g)


# ---------------------------------------------------------------------------------------------- encoder
@pytest.mark.parametrize("tag,peaky", [("base", False), ("peaky", True)])
def test_encoder_matches_golden(golden_dir, tag, peaky):
    g = _load(golden_dir, "encoder.npz")
    sd = R.danet_fixture_state(0, peaky=peaky)
    tick = R.synthetic_tick(np.random.RandomState(1000))
    x = torch.from_numpy(R.pre_process(tick["rgb"], tick["route_fig"].copy()))
    with torch.no_grad():
        l4 = R.backbone(x, sd)
        da = R.da_head(l4, sd)
        lat = R.encoder_latent(x, sd)
    assert np.array_equal(l4[:, :8].numpy(), g[f"{tag}_l4_slice"])
    assert np.array_equal(lat.numpy(), g[f"{tag}_latent"])
    # (sum, L2 norm, max |x|) of the whole backbone output and of the attention head (PAM + CAM branches)
    for t, key in ((l4, "l4_stats"), (da, "da_stats")):
        t = t.double().flatten()
        np.testing.assert_allclose([t.sum().item(), t.norm().item(), t.abs().max().item()], g[f"{tag}_{key}"],
                                   rtol=1e-12, atol=0)
    # the peaky fixture must actually be far from a uniform softmax to stress the attention kernels
    if peaky:
        assert np.abs(g["peaky_latent"] - g["base_latent"]).max() > 1e-3


def test_agent_feature_matches_golden(golden_dir):
    g = _load(golden_dir, "agent_feature.npz")
    sd = R.danet_fixture_state(0)
    rs = np.random.RandomState(2000)
    tick = R.synthetic_tick(rs)
    tick["route_fig"][3] = (rs.rand(256, 144) * 200).astype(np.uint8)
    tick["route_fig"][5] = 0
    with torch.no_grad():
        feat = R.agent_latent_feature(tick["rgb"], tick["route_fig"], tick["measurements"], sd)
    assert feat.dtype == torch.float32 and tuple(feat.shape) == (8, 530)
    assert np.array_equal(feat.numpy(), g["feature"])
    # bootstrap values for each command: LSTM unroll over the 8 frames with zero state, critic head
    ppo = R.ppo_fixture_state(0)
    h0 = torch.zeros(1, 530)
    for c in range(4):
        with torch.no_grad():
            fs, _ = R.lstm_forward(feat, h0, h0, ppo[f"steer_lstm_{c}"])
            ft, _ = R.lstm_forward(feat, h0, h0, ppo[f"throttle_lstm_{c}"])
            vs = R._mlp3(fs, ppo[f"steer_ppo_{c}"], "critic.")
            vt = R._mlp3(ft, ppo[f"throttle_ppo_{c}"], "critic.")
        assert np.array_equal(np.array([vs.item(), vt.item()], dtype=np.float32), g["values"][c])


# ---------------------------------------------------------------------------------------------- update
def _worker_samples(w):
    rs = np.random.RandomState(100 + w)
    st_s = R.synthetic_storage(rs, actions=R.STEER_ACTIONS)
    st_t = R.synthetic_storage(rs, actions=R.THROTTLE_ACTIONS)
    if w == 1:
        for st in (st_s, st_t):
            st["hn"] = torch.from_numpy(rs.randn(201, 530).astype(np.float32) * 0.3)
            st["cn"] = torch.from_numpy(rs.randn(201, 530).astype(np.float32) * 0.3)
    out = []
    for st, nv in ((st_s, 0.1), (st_t, -0.2)):
        st["returns"], st["value_preds"] = R.compute_returns(st["rewards"], st["value_preds"], st["masks"],
                                                             torch.tensor([[nv]]))
        out.append((st, R.normalized_advantages(st["returns"], st["value_preds"])))
    torch.manual_seed(500 + w)
    idx_s = R.minibatch_indices()[0]
    idx_t = R.minibatch_indices()[0]
    return R.gather_minibatch(out[0][0], out[0][1], idx_s), R.gather_minibatch(out[1][0], out[1][1], idx_t)


def test_update_and_chief_match_golden(golden_dir):
    g = _load(golden_dir, "update.npz")
    sd = R.ppo_fixture_state(0)
    params = {m: {n: t.clone().requires_grad_(True) for n, t in d.items()} for m, d in sd.items()}
    summed = {m: {n: torch.zeros_like(t) for n, t in d.items()} for m, d in sd.items()}
    for w in range(2):
        s_samp, t_samp = _worker_samples(w)
        losses = R.update_policy(s_samp, t_samp, params)
        np.testing.assert_allclose(np.array(losses), g["losses"][w], rtol=1e-6)
        k = 0
        for m in R.PPO_MODULE_ORDER:
            for n, _ in R.ppo_module_param_shapes(m):
                gr = params[m][n].grad
                if w == 0:
                    sl = gr.flatten()[:32].numpy()
                    np.testing.assert_allclose(sl, g["w0_grad_slices"][k][:len(sl)], rtol=2e-4, atol=1e-9)
                    np.testing.assert_allclose(gr.double().norm().item(), g["w0_grad_stats"][k][1], rtol=1e-5)
                summed[m][n] += gr
                k += 1
    adam = {m: {n: {"exp_avg": torch.zeros_like(t), "exp_avg_sq": torch.zeros_like(t)} for n, t in d.items()}
            for m, d in sd.items()}
    before = {m: {n: t.detach().clone() for n, t in d.items()} for m, d in params.items()}
    R.chief_step(params, summed, adam, step=1)
    k = 0
    for m in R.PPO_MODULE_ORDER:
        for n, _ in R.ppo_module_param_shapes(m):
            p = params[m][n].detach()
            # first Adam step moves every weight by ~lr*sign(g): compare parameters tightly, deltas by norm
            sl = p.flatten()[:32].numpy()
            np.testing.assert_allclose(sl, g["post_param_slices"][k][:len(sl)], rtol=0, atol=2e-6)
            np.testing.assert_allclose((p - before[m][n]).double().norm().item(), g["post_delta_stats"][k][1],
                                       rtol=2e-3)
            k += 1
    assert k == 128
    assert sum(t.numel() for d in sd.values() for t in d.values()) == 19382808


# ---------------------------------------------------------------------------------------------- live reference
@needs_ref
def test_restatement_bit_exact_vs_live_reference_encoder():
    sd = R.danet_fixture_state(3)
    net, _ = ref_shim.build_reference_danet(sd)
    tick = R.synthetic_tick(np.random.RandomState(77), seq=2)
    x = torch.from_numpy(R.pre_process(tick["rgb"], tick["route_fig"].copy()))
    with torch.no_grad():
        assert torch.equal(net.get_latent_feature(x, "concate"), R.encoder_latent(x, sd))
        l4 = net.backbone(x)
        f = net.da_head.conv5a(l4)
        assert torch.equal(net.da_head.sa(f), R.pam(f, sd))
        assert torch.equal(net.da_head.sc(f), R.cam(f, sd))


@needs_ref
def test_restatement_bit_exact_vs_live_reference_update():
    ref_shim.install()
    from ppo_agent.models import LSTM, Model
    sd = R.ppo_fixture_state(5)
    lstm = LSTM(530, hid_size=530)
    lstm.load_state_dict(sd["steer_lstm_2"])
    model = Model(530, 33)
    model.load_state_dict(sd["steer_ppo_2"])
    rs = np.random.RandomState(5)
    x = torch.from_numpy(rs.randn(8 * 6, 530).astype(np.float32))
    h0 = torch.from_numpy(rs.randn(6, 530).astype(np.float32))
    c0 = torch.from_numpy(rs.randn(6, 530).astype(np.float32))
    act = torch.from_numpy(rs.randint(0, 33, size=(6, 1)))
    with torch.no_grad():
        fr, _ = lstm(x, (h0, c0))
        fo, _ = R.lstm_forward(x, h0, c0, sd["steer_lstm_2"])
        assert torch.equal(fr, fo)
        for a, b in zip(model.evaluate_actions(fr, act), R.evaluate_actions(fo, act, sd["steer_ppo_2"])):
            assert torch.equal(a, b)
