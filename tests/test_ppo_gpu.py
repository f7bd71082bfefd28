"""PPO path parity on the B200 (through the C ABI): GAE, routed forward, losses, gradients, clip + Adam,
against reference-generated goldens and the CPU oracle. Tolerances (BASELINE north_star): GAE 1e-5 relative
fp32; losses 1e-3 relative; parameters after the step by relative L2 (TF32 tensor-core operands)."""
import os
from types import SimpleNamespace

import numpy as np
import pytest
import torch

from oracle import restate as R

pytestmark = pytest.mark.gpu
DEV = "cuda:0"


def rel(got, ref):
    got, ref = got.double().flatten().cpu(), ref.double().flatten().cpu()
    return ((got - ref).norm() / (ref.norm() + 1e-30)).item()


# ------------------------------------------------------------------------------------------------ GAE
@pytest.mark.parametrize("i,T,seed", [(0, 200, 0), (1, 200, 1), (2, 800, 2), (3, 7, 3)])
def test_gae_matches_reference_golden(golden_dir, i, T, seed):
    from cadre_b200 import ppo
    g = np.load(os.path.join(golden_dir, "gae.npz"))
    st = R.synthetic_storage(np.random.RandomState(seed), T=T, feature_dims=8, seq=1)
    if i == 1:
        st["masks"][::5] = 0.0
    r, v, m = (st[k].view(1, -1).to(DEV).contiguous() for k in ("rewards", "value_preds", "masks"))
    ret, adv = torch.zeros_like(r), torch.zeros(1, T, device=DEV)
    ppo.gae(r, v, m, torch.tensor([0.37 * (i + 1)], device=DEV), ret, adv)
    ref_ret = torch.from_numpy(g[f"returns_{i}"])[:T, 0]
    np.testing.assert_allclose(ret[0, :T].cpu().numpy(), ref_ret.numpy(), rtol=1e-5, atol=1e-5)
    assert rel(adv[0], torch.from_numpy(g[f"adv_{i}"])[:, 0]) < 1e-5
    assert v[0, T].item() == pytest.approx(0.37 * (i + 1))      # value_preds[-1] = next_value (storage.py:70)


@pytest.mark.parametrize("T", [2, 31, 32, 33, 255, 256, 257, 800, 1023, 1024, 1025, 3000])
def test_gae_all_kernel_variants_match_oracle(T):
    """Sequence lengths on both sides of every kernel switch (register-resident <= 256, <= 1024, general loop)
    and of the 32-lane chunking, with ~10 % episode boundaries; with and without advantage normalisation."""
    from cadre_b200 import ppo
    E = 5
    gen = torch.Generator().manual_seed(T)
    r = torch.rand(E, T + 1, generator=gen)
    v = torch.randn(E, T + 1, generator=gen)
    m = (torch.rand(E, T + 1, generator=gen) > 0.1).float()
    nv = torch.randn(E, generator=gen)
    for normalize in (True, False):
        vd = v.to(DEV).clone()
        ret, adv = torch.zeros(E, T + 1, device=DEV), torch.zeros(E, T, device=DEV)
        ppo.gae(r.to(DEV), vd, m.to(DEV), nv.to(DEV), ret, adv, normalize=normalize)
        for e in range(E):
            ref_ret, vp = R.compute_returns(r[e].view(-1, 1), v[e].view(-1, 1).clone(), m[e].view(-1, 1), nv[e].view(1, 1))
            np.testing.assert_allclose(ret[e, :T].cpu().numpy(), ref_ret[:T, 0].numpy(), rtol=1e-5, atol=1e-5)
            ref_adv = R.normalized_advantages(ref_ret, vp) if normalize else (ref_ret[:-1] - vp[:-1])
            assert rel(adv[e], ref_adv[:, 0]) < 2e-5
            assert vd[e, T].item() == pytest.approx(nv[e].item())


@pytest.mark.parametrize("T", [257, 500, 512, 513, 800, 1000, 1024])
def test_gae_many_sequences_long_T(T):
    """256 < T <= 1024 (two-warp blocks, cp.async staging): several waves
    of sequences, ragged T, ~10 % episode boundaries; a sample of sequences vs the oracle."""
    from cadre_b200 import ppo
    E = 8 * 148 * 3 + 5
    g = torch.Generator(device=DEV).manual_seed(T)
    r = torch.rand(E, T + 1, device=DEV, generator=g)
    v = torch.randn(E, T + 1, device=DEV, generator=g)
    m = (torch.rand(E, T + 1, device=DEV, generator=g) > 0.1).float()
    nv = torch.randn(E, device=DEV, generator=g)
    for normalize in (True, False):
        vd = v.clone()
        ret, adv = torch.zeros(E, T + 1, device=DEV), torch.zeros(E, T, device=DEV)
        ppo.gae(r, vd, m, nv, ret, adv, normalize=normalize)
        for e in (0, 1, 7, 8, 1183, 1184, 1185, 2367, 2368, E - 2, E - 1):
            ref_ret, vp = R.compute_returns(r[e].cpu().view(-1, 1), v[e].cpu().view(-1, 1).clone(),
                                            m[e].cpu().view(-1, 1), nv[e].cpu().view(1, 1))
            np.testing.assert_allclose(ret[e, :T].cpu().numpy(), ref_ret[:T, 0].numpy(), rtol=1e-5, atol=1e-5)
            ref_adv = R.normalized_advantages(ref_ret, vp) if normalize else (ref_ret[:-1] - vp[:-1])
            assert rel(adv[e], ref_adv[:, 0]) < 2e-5
            assert vd[e, T].item() == pytest.approx(nv[e].item())
    assert torch.isfinite(adv).all() and torch.isfinite(ret).all()


def test_gae_large_sweep_properties():
    """65 536 sequences x 1 024 steps (1.3 GB): linearity in the rewards and the all-masked closed form."""
    from cadre_b200 import ppo
    E, T = 65536, 1024
    g = torch.Generator(device=DEV).manual_seed(0)
    r = torch.rand(E, T + 1, device=DEV, generator=g)
    v = torch.randn(E, T + 1, device=DEV, generator=g)
    m = (torch.rand(E, T + 1, device=DEV, generator=g) > 0.02).float()
    nv = torch.randn(E, device=DEV, generator=g)
    out = [torch.zeros(E, T + 1, device=DEV) for _ in range(3)]
    adv = torch.zeros(E, T, device=DEV)
    ppo.gae(r, v.clone(), m, nv, out[0], adv, normalize=False)
    ppo.gae(2 * r, (2 * v).clone(), m, 2 * nv, out[1], adv, normalize=False)
    assert rel(out[1][:, :T], 2 * out[0][:, :T]) < 1e-6                      # linear in (r, V)
    ppo.gae(r, v.clone(), torch.zeros_like(m), nv, out[2], adv, normalize=False)
    assert torch.allclose(out[2][:, :T], r[:, :T], atol=1e-6)                # mask 0: returns_t = r_t
    # spot check 8 random sequences against the oracle loop
    for e in (0, 1, 777, 65535):
        ret, _ = R.compute_returns(r[e].cpu().view(-1, 1), v[e].cpu().view(-1, 1), m[e].cpu().view(-1, 1),
                                   nv[e].cpu().view(1, 1))
        np.testing.assert_allclose(out[0][e, :T].cpu().numpy(), ret[:T, 0].numpy(), rtol=2e-5, atol=2e-5)


# ------------------------------------------------------------------------------------------------ update
def _worker(w):
    rs = np.random.RandomState(100 + w)
    st_s = R.synthetic_storage(rs, actions=R.STEER_ACTIONS)
    st_t = R.synthetic_storage(rs, actions=R.THROTTLE_ACTIONS)
    if w == 1:
        for st in (st_s, st_t):
            st["hn"] = torch.from_numpy(rs.randn(201, 530).astype(np.float32) * 0.3)
            st["cn"] = torch.from_numpy(rs.randn(201, 530).astype(np.float32) * 0.3)
    advs = []
    for st, nv in ((st_s, 0.1), (st_t, -0.2)):
        st["returns"], st["value_preds"] = R.compute_returns(st["rewards"], st["value_preds"], st["masks"],
                                                             torch.tensor([[nv]]))
        advs.append(R.normalized_advantages(st["returns"], st["value_preds"]))
    torch.manual_seed(500 + w)
    return (st_s, st_t), advs, (R.minibatch_indices()[0], R.minibatch_indices()[0])


def _dev(st):
    return SimpleNamespace(**{k: v.to(DEV).contiguous() for k, v in st.items()})


@pytest.fixture(scope="module")
def two_worker_update():
    from cadre_b200 import ppo, ppo_params
    torch.set_num_threads(8)
    sd = R.ppo_fixture_state(0)
    cpu = [_worker(w) for w in range(2)]
    storages = [(_dev(c[0][0]), _dev(c[0][1])) for c in cpu]
    advs = [(c[1][0].to(DEV).contiguous(), c[1][1].to(DEV).contiguous()) for c in cpu]
    idx = np.array([[c[2][0], c[2][1]] for c in cpu], dtype=np.int32)
    flat = ppo_params.pack_state(sd, DEV)
    grads = torch.zeros_like(flat)
    eng = ppo.PpoEngine(2, 100, device=DEV)
    ev = eng.evaluate(storages, advs, idx, flat).cpu()
    losses = eng.update(storages, advs, idx, flat, grads).cpu()
    eng.check()             # no hand-off of the persistent recurrence kernels timed out
    # oracle: per-worker update_policy, gradients summed like Shared_grad_buffers.add_gradient
    params = {m: {n: t.clone().requires_grad_(True) for n, t in d.items()} for m, d in sd.items()}
    summed = {m: {n: torch.zeros_like(t) for n, t in d.items()} for m, d in sd.items()}
    ref_losses = []
    for w in range(2):
        s = R.gather_minibatch(cpu[w][0][0], cpu[w][1][0], cpu[w][2][0])
        t = R.gather_minibatch(cpu[w][0][1], cpu[w][1][1], cpu[w][2][1])
        ref_losses.append(R.update_policy(s, t, params))
        for m in params:
            for n in params[m]:
                summed[m][n] += params[m][n].grad
    return dict(eng=eng, flat=flat, grads=grads, losses=losses, ev=ev, cpu=cpu, sd=sd, summed=summed,
                ref_losses=ref_losses, ppo_params=ppo_params)


def test_losses_match_reference_golden(two_worker_update, golden_dir):
    u = two_worker_update
    g = np.load(os.path.join(golden_dir, "update.npz"))
    for w in range(2):
        L = u["losses"][w].sum(0)
        got = np.array([0.1 * L[0].item(), L[1].item(), 0.01 * L[2].item()])
        np.testing.assert_allclose(got, g["losses"][w], rtol=1e-3)                 # reference run (golden)
        np.testing.assert_allclose(got, np.array(u["ref_losses"][w]), rtol=1e-3)   # oracle


def test_forward_rows_match_oracle(two_worker_update):
    u = two_worker_update
    sd = u["sd"]
    for head_i, head in enumerate(("steer", "throttle")):
        ref = []
        for w in range(2):
            obs, action, _, _, _, _, _, (hn, cn), command = R.gather_minibatch(u["cpu"][w][0][head_i],
                                                                               u["cpu"][w][1][head_i],
                                                                               u["cpu"][w][2][head_i])
            acc = torch.zeros(100, 3)
            with torch.no_grad():
                for c in range(4):
                    feat, _ = R.lstm_forward(obs.clone(), hn, cn, sd[f"{head}_lstm_{c}"])
                    v, lp, en = R.evaluate_actions(feat, action, sd[f"{head}_ppo_{c}"])
                    acc += torch.cat([v, lp, en], 1) * (command == c)
            ref.append(acc)
        ref = torch.cat(ref, 0)
        got = u["ev"][head_i, :, :3]
        assert rel(got[:, 0], ref[:, 0]) < 2e-3        # value (TF32 operands)
        assert rel(got[:, 1], ref[:, 1]) < 1e-3        # log-prob of the stored action
        assert rel(got[:, 2], ref[:, 2]) < 1e-4        # entropy


def test_gradients_match_oracle_and_golden(two_worker_update, golden_dir):
    u = two_worker_update
    P = u["ppo_params"]
    g = P.unpack_state(u["grads"].cpu())
    names = [(m, n) for m in P.MODULE_ORDER for n in P.module_param_names(m)]
    got = torch.cat([g[m][n].flatten() for m, n in names])
    ref = torch.cat([u["summed"][m][n].flatten() for m, n in names])
    assert rel(got, ref) < 2e-2                                                   # all 19.4 M gradients
    per = sorted(rel(g[m][n], u["summed"][m][n]) for m, n in names)
    assert per[len(per) // 2] < 5e-3 and per[-1] < 5e-2       # worst single tensor (ReLU-mask flips, DESIGN.md §2)
    # layout padding never receives gradient
    probe = torch.zeros(P.TOTAL)
    for m, n in names:
        P.tensor_view(probe, m, n)[0].fill_(1.0)
    assert u["grads"].cpu()[probe == 0].abs().max().item() == 0.0
    # the reference run's own numbers (golden): per-module norms of the summed gradient (chief.py:19, clip_grad_norm_)
    gold = np.load(os.path.join(golden_dir, "update.npz"))
    got_norms = [torch.sqrt(sum((g[m][n].double() ** 2).sum() for n in P.module_param_names(m))).item()
                 for m in P.MODULE_ORDER]
    np.testing.assert_allclose(got_norms, gold["module_grad_norms"], rtol=1e-2)


def test_worker0_gradient_slices_match_reference_golden(two_worker_update, golden_dir):
    """update.npz `w0_grad_slices` / `w0_grad_stats`: worker 0's own gradient from the reference run (first 32 elements,
    [sum, norm, absmax] of all 128 tensors), against a one-worker CUDA update on the same minibatch."""
    from cadre_b200 import ppo
    u = two_worker_update
    P = u["ppo_params"]
    gold = np.load(os.path.join(golden_dir, "update.npz"))
    c = u["cpu"][0]
    storages = [(_dev(c[0][0]), _dev(c[0][1]))]
    advs = [(c[1][0].to(DEV).contiguous(), c[1][1].to(DEV).contiguous())]
    idx = np.array([[c[2][0], c[2][1]]], dtype=np.int32)
    grads = torch.zeros_like(u["flat"])
    ppo.PpoEngine(1, 100, device=DEV).update(storages, advs, idx, u["flat"], grads)
    g = P.unpack_state(grads.cpu())
    k = 0
    num = den = 0.0
    for m in P.MODULE_ORDER:
        for n in P.module_param_names(m):
            t = g[m][n].flatten().double()
            ref_sl = torch.from_numpy(gold["w0_grad_slices"][k][:min(32, t.numel())]).double()
            num += ((t[:len(ref_sl)] - ref_sl) ** 2).sum().item()
            den += (ref_sl ** 2).sum().item()
            ref_sum, ref_norm, ref_max = gold["w0_grad_stats"][k]
            assert abs(t.norm().item() - ref_norm) <= 2e-2 * ref_norm + 1e-9, (m, n)
            assert abs(t.abs().max().item() - ref_max) <= 5e-2 * ref_max + 1e-9, (m, n)
            k += 1
    assert k == 128 and (num / den) ** 0.5 < 2e-2


def test_unrouted_experts_get_exactly_zero_gradient():
    """agent.py:170-182 masks every row by its command, so an expert no row is routed to receives a zero gradient
    (autograd of `x * False`). Here such experts are never visited; every element of their 8 x 16 tensors must be
    EXACTLY 0.0 while the visited experts' gradients are not."""
    from cadre_b200 import ppo, ppo_params as P
    rs = np.random.RandomState(9)
    sts = []
    for a, cmds in ((R.STEER_ACTIONS, (0, 1)), (R.THROTTLE_ACTIONS, (3,))):
        st = R.synthetic_storage(rs, T=64, actions=a)
        st["command"] = torch.from_numpy(rs.choice(cmds, size=(65, 1)).astype(np.int32))
        st["returns"] = torch.from_numpy(rs.randn(65, 1).astype(np.float32))
        sts.append(st)
    adv = [torch.from_numpy(rs.randn(64, 1).astype(np.float32)) for _ in range(2)]
    idx = np.array([[list(rs.permutation(64)[:32]), list(rs.permutation(64)[:32])]], dtype=np.int32)
    flat = P.pack_state(R.ppo_fixture_state(0), DEV)
    grads = torch.full_like(flat, 123.0)                                   # stale values must be overwritten
    eng = ppo.PpoEngine(1, 32, device=DEV)
    eng.update([(_dev(sts[0]), _dev(sts[1]))], [(adv[0].to(DEV), adv[1].to(DEV))], idx, flat, grads)
    eng.check()
    g = P.unpack_state(grads.cpu())
    visited = {"steer": (0, 1), "throttle": (3,)}
    for head in ("steer", "throttle"):
        for c in range(4):
            for m in (f"{head}_lstm_{c}", f"{head}_ppo_{c}"):
                tot = sum(t.abs().sum().item() for t in g[m].values())
                if c in visited[head]:
                    assert tot > 0.0, m
                else:
                    assert all(t.abs().max().item() == 0.0 for t in g[m].values()), m


def test_clip_adam_matches_oracle(two_worker_update):
    u = two_worker_update
    P = u["ppo_params"]
    flat, grads = u["flat"].clone(), u["grads"]
    m1, m2 = torch.zeros_like(flat), torch.zeros_like(flat)
    # feed the ORACLE's summed gradient so that this test isolates the clip + Adam kernels
    gflat = P.pack_state(u["summed"], DEV)
    u["eng"].adam_step(flat, gflat, m1, m2, step=1)
    sd = u["sd"]
    adam = {m: {n: {"exp_avg": torch.zeros_like(t), "exp_avg_sq": torch.zeros_like(t)} for n, t in d.items()}
            for m, d in sd.items()}
    pref = {m: {n: t.detach().clone() for n, t in d.items()} for m, d in sd.items()}
    R.chief_step(pref, u["summed"], adam, step=1)
    post = P.unpack_state(flat.cpu())
    names = [(m, n) for m in P.MODULE_ORDER for n in P.module_param_names(m)]
    a = torch.cat([post[m][n].flatten() for m, n in names])
    b = torch.cat([pref[m][n].flatten() for m, n in names])
    a0 = torch.cat([sd[m][n].flatten() for m, n in names])
    assert rel(a, b) < 1e-6 and rel(a - a0, b - a0) < 1e-3
    norms = u["eng"].module_norms()
    for m in sd:
        ref_n = torch.sqrt(sum((u["summed"][m][n].double() ** 2).sum() for n in sd[m])).item()
        assert norms[m] == pytest.approx(ref_n, rel=1e-5)
    # a second step with a huge gradient exercises the clip branch (coef < 1) per module
    big = gflat * 1e5
    u["eng"].adam_step(flat, big, m1, m2, step=2)
    grads2 = {m: {n: u["summed"][m][n] * 1e5 for n in sd[m]} for m in sd}
    R.chief_step(pref, grads2, adam, step=2)
    post = P.unpack_state(flat.cpu())
    a = torch.cat([post[m][n].flatten() for m, n in names])
    b = torch.cat([pref[m][n].flatten() for m, n in names])
    assert rel(a, b) < 1e-6


def _delta_agreement(d_got, d_ref):
    """How well two first-Adam-step updates agree. The first step moves every weight by ~ lr * sign(g) (bias-corrected
    m / sqrt(v) = g / |g|), so the relative L2 of the DELTAS is sqrt(4 * fraction of sign flips) - a far sharper
    measure than the relative L2 of theta (|delta| ~ 3e-4 on |theta| ~ 4e-2 would let a no-op Adam pass)."""
    d_got, d_ref = d_got.double().flatten().cpu(), d_ref.double().flatten().cpu()
    rel_d = ((d_got - d_ref).norm() / d_ref.norm()).item()
    moved = d_ref.abs() > 0
    flips = ((torch.sign(d_got) != torch.sign(d_ref)) & moved).double().mean().item()
    return rel_d, flips


# Stated tolerance for post-step parameters (north_star: "post-step parameters within a stated tf32 tolerance"):
#   relative L2 of delta-theta <= DELTA_REL, i.e. at most DELTA_REL^2 / 4 of the 19.4 M weights step the other way
#   (those are weights whose gradient is within TF32 noise of zero).
DELTA_REL = 0.2     # measured on B200: 0.096 (2 workers x 100 rows), 0.127 (cfg 3), 0.161 (cfg 5: 0.7 % sign flips)


def test_delta_theta_matches_oracle(two_worker_update):
    """CUDA gradients -> CUDA clip + Adam against the oracle's chief step on the oracle's gradients: the UPDATE itself
    (delta theta), not theta."""
    u = two_worker_update
    P = u["ppo_params"]
    flat = u["flat"].clone()
    m1, m2 = torch.zeros_like(flat), torch.zeros_like(flat)
    u["eng"].adam_step(flat, u["grads"], m1, m2, step=1)
    sd = u["sd"]
    adam = {m: {n: {"exp_avg": torch.zeros_like(t), "exp_avg_sq": torch.zeros_like(t)} for n, t in d.items()}
            for m, d in sd.items()}
    pref = {m: {n: t.detach().clone() for n, t in d.items()} for m, d in sd.items()}
    R.chief_step(pref, u["summed"], adam, step=1)
    post = P.unpack_state(flat.cpu())
    names = [(m, n) for m in P.MODULE_ORDER for n in P.module_param_names(m)]
    d_got = torch.cat([(post[m][n] - sd[m][n]).flatten() for m, n in names])
    d_ref = torch.cat([(pref[m][n] - sd[m][n]).flatten() for m, n in names])
    rel_d, flips = _delta_agreement(d_got, d_ref)
    print(f"delta-theta rel-L2 {rel_d:.4f}, sign flips {flips:.5f}")
    assert d_got.abs().max().item() <= 3e-4 * 1.001 and d_got.abs().max().item() > 2.9e-4   # Adam really stepped by lr
    assert rel_d < DELTA_REL, (rel_d, flips)


def test_post_step_statistics_match_reference_golden(two_worker_update, golden_dir):
    """update.npz `post_delta_stats` ([sum, norm, absmax] of delta theta per tensor, from the reference's own
    optimizer.step()) against the CUDA step."""
    u = two_worker_update
    P = u["ppo_params"]
    gold = np.load(os.path.join(golden_dir, "update.npz"))
    flat = u["flat"].clone()
    m1, m2 = torch.zeros_like(flat), torch.zeros_like(flat)
    u["eng"].adam_step(flat, u["grads"], m1, m2, step=1)
    post = P.unpack_state(flat.cpu())
    k = 0
    for m in P.MODULE_ORDER:
        for n in P.module_param_names(m):
            d = (post[m][n] - u["sd"][m][n]).double().flatten()
            _, ref_norm, ref_max = gold["post_delta_stats"][k]
            assert abs(d.norm().item() - ref_norm) <= 2e-2 * ref_norm + 1e-12, (m, n, d.norm().item(), ref_norm)
            assert abs(d.abs().max().item() - ref_max) <= 1e-2 * ref_max + 1e-12, (m, n)
            k += 1
    assert k == 128


def test_end_to_end_step_parameters(two_worker_update, golden_dir):
    """CUDA gradients -> CUDA clip + Adam vs the reference's post-step parameters (golden)."""
    u = two_worker_update
    P = u["ppo_params"]
    g = np.load(os.path.join(golden_dir, "update.npz"))
    flat = u["flat"].clone()
    m1, m2 = torch.zeros_like(flat), torch.zeros_like(flat)
    u["eng"].adam_step(flat, u["grads"], m1, m2, step=1)
    post = P.unpack_state(flat.cpu())
    k = 0
    num = den = 0.0
    for m in P.MODULE_ORDER:
        for n in P.module_param_names(m):
            sl = post[m][n].flatten()[:32].double()
            ref = torch.from_numpy(g["post_param_slices"][k][:len(sl)]).double()
            num += ((sl - ref) ** 2).sum().item()
            den += (ref ** 2).sum().item()
            # the first Adam step moves every weight by ~lr * sign(g): bounded by 2 * lr elementwise
            assert (sl - ref).abs().max().item() <= 2 * 3e-4 + 1e-6
            k += 1
    assert (num / den) ** 0.5 < 5e-3


# ------------------------------------------------------------------------------------------------ declared configs
def _make_worker(w, T, seed0, commands=None):
    """Storages (steer, throttle) of worker w and their normalised advantages. `commands`: optional pair (steer,
    throttle) of (storage rows, command of each row), written into the storages' command column."""
    rs = np.random.RandomState(seed0 + w)
    pair = [R.synthetic_storage(rs, T=T, actions=a) for a in (R.STEER_ACTIONS, R.THROTTLE_ACTIONS)]
    if w % 3 == 1:                                           # non-zero stored recurrent state in some workers
        for st in pair:
            st["hn"] = torch.from_numpy(rs.randn(T + 1, 530).astype(np.float32) * 0.3)
            st["cn"] = torch.from_numpy(rs.randn(T + 1, 530).astype(np.float32) * 0.3)
    if commands is not None:
        for st, (rows, cmd) in zip(pair, commands):
            st["command"][torch.as_tensor(np.asarray(rows, dtype=np.int64)), 0] = torch.as_tensor(
                np.asarray(cmd, dtype=np.int32))
    advs = []
    for st, nv in zip(pair, (0.1, -0.2)):
        st["returns"], st["value_preds"] = R.compute_returns(st["rewards"], st["value_preds"], st["masks"],
                                                             torch.tensor([[nv]]))
        advs.append(R.normalized_advantages(st["returns"], st["value_preds"]))
    return pair, advs


def _config_inputs(W, mb, T, seed0, plan=None, shift=0):
    """Inputs of one update step of W workers: storages of T steps, minibatch indices of mb rows per worker and head
    drawn like storage.py:93-97, and - with a routing `plan` (ROUTING_PLANS) - commands that give every expert exactly
    the plan's row count (commands shifted by `shift`, c -> (c + shift) % 4)."""
    idx = np.empty((W, 2, mb), dtype=np.int32)
    for w in range(W):
        torch.manual_seed(seed0 + 1000 + w)
        idx[w, 0] = R.minibatch_indices(T, T // mb)[0]
        idx[w, 1] = R.minibatch_indices(T, T // mb)[1 % (T // mb)]
    cmds = [None] * W
    if plan is not None:
        cmds = _plan_commands(_plan_counts(plan, shift), idx, seed0)
    cpu = [_make_worker(w, T, seed0, cmds[w]) for w in range(W)]
    storages = [(_dev(c[0][0]), _dev(c[0][1])) for c in cpu]
    advs = [(c[1][0].to(DEV).contiguous(), c[1][1].to(DEV).contiguous()) for c in cpu]
    counts = [np.bincount(np.concatenate([cpu[w][0][h]["command"][idx[w, h], 0].numpy() for w in range(W)]),
                          minlength=4) for h in range(2)]
    return SimpleNamespace(W=W, mb=mb, T=T, idx=idx, cpu=cpu, storages=storages, advs=advs, counts=counts)


def _stale_grads(flat):
    """A gradient buffer that holds 123.0 in every parameter element (layout padding 0.0, as in a real learner): an
    update has to overwrite every element it owns, including the exact zeros of an expert without rows."""
    from cadre_b200 import ppo_params as P
    g = torch.zeros_like(flat)
    for m in P.MODULE_ORDER:
        for n in P.module_param_names(m):
            P.tensor_view(g, m, n)[0].fill_(123.0)
    return g


def _run_config(W, mb, T, seed0, plan=None):
    """One update step of W workers (storages of T steps, minibatches of mb rows drawn like storage.py:93-97) on the
    GPU and in the oracle (per-worker update_policy, gradients summed like Shared_grad_buffers.add_gradient, chief
    step); `plan` fixes every expert's row count (ROUTING_PLANS). Checks the losses per worker and head and the
    module norms, and returns the inputs, the engine, the CUDA losses / gradients / post-step parameters, the oracle's
    summed gradients and the agreement figures."""
    from cadre_b200 import ppo, ppo_params as P
    torch.set_num_threads(min(16, os.cpu_count() or 1))
    sd = R.ppo_fixture_state(0)
    x = _config_inputs(W, mb, T, seed0, plan)
    cpu, idx = x.cpu, x.idx
    flat = P.pack_state(sd, DEV)
    grads = _stale_grads(flat)
    eng = ppo.PpoEngine(W, mb, device=DEV)
    losses = eng.update(x.storages, x.advs, idx, flat, grads).cpu()
    eng.check()
    post_flat = flat.clone()
    m1, m2 = torch.zeros_like(flat), torch.zeros_like(flat)
    eng.adam_step(post_flat, grads, m1, m2, step=1)
    # oracle
    params = {m: {n: t.clone().requires_grad_(True) for n, t in d.items()} for m, d in sd.items()}
    summed = {m: {n: torch.zeros_like(t) for n, t in d.items()} for m, d in sd.items()}
    for w in range(W):
        samples = [R.gather_minibatch(cpu[w][0][h], cpu[w][1][h], list(idx[w, h])) for h in range(2)]
        ref_heads = []
        ref_l = R.update_policy(samples[0], samples[1], params, head_losses=ref_heads)
        L = losses[w].sum(0)
        got = np.array([0.1 * L[0].item(), L[1].item(), 0.01 * L[2].item()])
        np.testing.assert_allclose(got, np.array(ref_l), rtol=1e-3, err_msg=f"worker {w}")
        np.testing.assert_allclose(losses[w].numpy(), np.array(ref_heads), rtol=1e-3, err_msg=f"worker {w} per head")
        for m in params:
            for n in params[m]:
                summed[m][n] += params[m][n].grad
    adam = {m: {n: {"exp_avg": torch.zeros_like(t), "exp_avg_sq": torch.zeros_like(t)} for n, t in d.items()}
            for m, d in sd.items()}
    pref = {m: {n: t.detach().clone() for n, t in d.items()} for m, d in sd.items()}
    R.chief_step(pref, summed, adam, step=1)
    names = [(m, n) for m in P.MODULE_ORDER for n in P.module_param_names(m)]
    visited = {m for m in sd if x.counts[P.expert_of(m) // 4][P.expert_of(m) % 4] > 0}
    g = P.unpack_state(grads.cpu())
    post = P.unpack_state(post_flat.cpu())
    cat = lambda d: torch.cat([d[m][n].flatten() for m, n in names])   # noqa: E731
    g_rel = rel(cat(g), cat(summed))
    per = sorted(rel(g[m][n], summed[m][n]) for m, n in names)
    per_visited = sorted(rel(g[m][n], summed[m][n]) for m, n in names if m in visited)
    th_rel = rel(cat(post), cat(pref))
    d_rel, flips = _delta_agreement(cat(post) - cat(sd), cat(pref) - cat(sd))
    norms = eng.module_norms()
    for m in sd:
        ref_n = torch.sqrt(sum((summed[m][n].double() ** 2).sum() for n in sd[m])).item()
        assert norms[m] == pytest.approx(ref_n, rel=2e-2), m
    print(f"{plan or 'uniform'} W={W} mb={mb} T={T}: grad rel-L2 {g_rel:.4e} (median visited tensor "
          f"{per_visited[len(per_visited) // 2]:.2e}, worst {per_visited[-1]:.2e}), theta rel-L2 {th_rel:.2e}, "
          f"delta-theta rel-L2 {d_rel:.4f} (sign flips {flips:.5f})")
    return SimpleNamespace(x=x, sd=sd, eng=eng, flat=flat, grads=grads, losses=losses, post_flat=post_flat, g=g,
                           summed=summed, visited=visited, g_rel=g_rel, per=per, per_visited=per_visited,
                           th_rel=th_rel, d_rel=d_rel, norms=norms)


def test_cfg3_update_step_four_workers():
    """BASELINE config 3 (the shape bench.py times): 4 workers x minibatches of 100 rows x 2 heads from T = 200."""
    u = _run_config(W=4, mb=100, T=200, seed0=300)
    assert u.g_rel < 2e-2 and u.per[len(u.per) // 2] < 5e-3 and u.per[-1] < 5e-2
    assert u.th_rel < 2e-3 and u.d_rel < DELTA_REL


def test_cfg5_update_step_eight_workers_T800():
    """BASELINE config 5 per GPU: 8 environments x minibatches of 400 rows x 2 heads from T = 800 (3200 rows per head:
    several 128-row tiles per expert, the tensor-core-bound regime of the TF32 GEMMs)."""
    u = _run_config(W=8, mb=400, T=800, seed0=700)
    assert u.g_rel < 2e-2 and u.per[len(u.per) // 2] < 5e-3 and u.per[-1] < 5e-2
    assert u.th_rel < 2e-3 and u.d_rel < DELTA_REL


def test_cfg5_gae_128_sequences_T800():
    """cfg 5's GAE launch: 128 sequences (64 envs x 2 heads) x 800 steps in one call, every sequence vs the oracle."""
    from cadre_b200 import ppo
    E, T = 128, 800
    gen = torch.Generator().manual_seed(5)
    r = torch.rand(E, T + 1, generator=gen)
    v = torch.randn(E, T + 1, generator=gen)
    m = (torch.rand(E, T + 1, generator=gen) > 0.02).float()
    nv = torch.randn(E, generator=gen)
    vd = v.to(DEV).clone()
    ret, adv = torch.zeros(E, T + 1, device=DEV), torch.zeros(E, T, device=DEV)
    ppo.gae(r.to(DEV), vd, m.to(DEV), nv.to(DEV), ret, adv)
    for e in range(E):
        ref_ret, vp = R.compute_returns(r[e].view(-1, 1), v[e].view(-1, 1).clone(), m[e].view(-1, 1), nv[e].view(1, 1))
        np.testing.assert_allclose(ret[e, :T].cpu().numpy(), ref_ret[:T, 0].numpy(), rtol=1e-5, atol=1e-5)
        assert rel(adv[e], R.normalized_advantages(ref_ret, vp)[:, 0]) < 2e-5


# ------------------------------------------------------------------------------------------------ routing
# The update routes rows instead of masking them (agent.py:170-182 -> route_kernel), and almost every later launch
# sizes its work from the per-expert row counts: the x-part GEMM's tile list, the LSTM kernels' 128-row tiles and
# their 32-row zero fill, head_kernel's CTAs and active-expert count, the K of the weight-gradient GEMMs rounded up to
# whole k-blocks. Uniform random commands give every expert about R / 4 rows; these plans put the counts at the edges.
SKEWED_P = (0.05, 0.05, 0.05, 0.85)    # driving: one command (lane following) dominates
ROUTING_PLANS = {  # name: (W, mb, steer rows of commands 0..3, throttle rows of commands 0..3); None: seeded draw
    "one_expert": (4, 100, (0, 0, 0, 400), (400, 0, 0, 0)),           # capacity worst case; 3 empty experts per head
    "tile_edges": (4, 100, (128, 129, 127, 16), (31, 33, 256, 80)),   # 128- / 32-row edges; 9 * 31 pads to 35.6 rows
    "kblock_edges": (4, 100, (95, 7, 8, 290), (1, 0, 399, 0)),        # 9 * count = 63 / 72; 95 pads to 99.6 rows
    "skewed": (4, 100, None, None),                                   # multinomial(R, SKEWED_P) per head
    "cfg5_one_expert": (8, 400, (0, 0, 3200, 0), (3199, 1, 0, 0)),    # 25 row tiles; 4 route_kernel chunks
    "actor_shape": (1, 64, (0, 64, 0, 0), (0, 64, 0, 0)),             # BatchedActor: every env on one command
}


def _plan_seed(plan):
    return 3000 + 100 * list(ROUTING_PLANS).index(plan)


def _plan_counts(plan, shift=0):
    """[steer, throttle] rows per command of a plan; `shift` moves command c's rows to (c + shift) % 4."""
    W, mb, *heads = ROUTING_PLANS[plan]
    rs = np.random.RandomState(17)
    counts = [rs.multinomial(W * mb, SKEWED_P) if c is None else np.asarray(c) for c in heads]
    assert all(c.sum() == W * mb for c in counts), plan
    return [np.roll(c, shift) for c in counts]


def _plan_commands(counts, idx, seed):
    """Per worker: ((rows, commands) of steer, (rows, commands) of throttle) such that head h routes exactly
    counts[h][c] minibatch rows to command c. Each head's command list is shuffled with a seeded RNG, so every
    expert's rows are spread over workers and minibatch positions (flat row r = w * mb + i)."""
    W, mb = idx.shape[0], idx.shape[2]
    rs = np.random.RandomState(seed)
    per_head = [rs.permutation(np.repeat(np.arange(4), counts[h])).reshape(W, mb) for h in range(2)]
    return [tuple((idx[w, h], per_head[h][w]) for h in range(2)) for w in range(W)]


@pytest.fixture(scope="module", params=list(ROUTING_PLANS))
def routed_update(request):
    """One update + clip + Adam step of a routing plan on the GPU and in the oracle (_run_config)."""
    W, mb = ROUTING_PLANS[request.param][:2]
    u = _run_config(W, mb, 2 * mb, _plan_seed(request.param), plan=request.param)
    u.plan = request.param
    return u


# Median tensor error over the visited experts: 5e-3, as for the declared configs. With one expert per head
# (one_expert, actor_shape) it is the median of two experts' 32 tensors, 24 of which sit behind ReLU masks, and which
# rows flip a mask at a pre-activation within rounding error of zero sets their error. Measured on B200: 8.0e-3
# (one_expert) and 4.1e-3 (actor_shape). Rounding only the fp32 oracle's operands to fp16 / TF32 moves the oracle's own
# gradient by a median 3.1e-3 / 4.1e-3 (worst 4.7e-2 / 4.1e-2) on the same inputs, and the 400-row update equals the
# sum of its four single-tile parts to 3.5e-6, so this is the sensitivity of the gradient, not a routing error.
MEDIAN_REL_ONE_EXPERT_PER_HEAD = 1.5e-2
# Last layers: no ReLU mask lies between them and the loss, so they carry the forward error only (<= 7.4e-4 measured).
# One row of 400 routed to the wrong expert moves them by ~5 %.
LAST_LAYERS = ("control.linear.4.weight", "control.linear.4.bias", "critic.4.weight", "critic.4.bias")
LAST_LAYER_REL = 5e-3


def test_routed_update_matches_oracle(routed_update):
    """Losses per worker and head and module norms (checked in _run_config), the gradients of the visited experts
    (overall, median and worst tensor, last layers) and delta-theta against the oracle. An expert without rows gets an
    EXACTLY zero gradient and module norm (the buffer held 123.0 before the update), and clip + Adam leave its
    parameters bit for bit unchanged."""
    from cadre_b200 import ppo_params as P
    u = routed_update
    pv = u.per_visited
    n_experts = len({P.expert_of(m) for m in u.visited})
    median_bound = MEDIAN_REL_ONE_EXPERT_PER_HEAD if n_experts == 2 else 5e-3
    last = max(rel(u.g[m][n], u.summed[m][n]) for m in u.visited if "_ppo_" in m for n in LAST_LAYERS)
    print(f"{u.plan}: worst last-layer tensor {last:.2e}")
    assert u.g_rel < 2e-2 and pv[len(pv) // 2] < median_bound and pv[-1] < 5e-2, (u.g_rel, pv[len(pv) // 2], pv[-1])
    assert last < LAST_LAYER_REL, last
    assert u.d_rel < DELTA_REL, u.d_rel
    for m in P.MODULE_ORDER:
        if m in u.visited:
            continue
        assert u.norms[m] == 0.0, m
        for n in P.module_param_names(m):
            assert u.g[m][n].abs().max().item() == 0.0, (m, n)
            assert torch.equal(P.tensor_view(u.post_flat, m, n)[0], P.tensor_view(u.flat, m, n)[0]), (m, n)


def _oracle_rows(u, h):
    """[value, log-prob of the stored action, entropy] of every minibatch row of head h in (worker, minibatch
    position) order, each row through the LSTM + actor-critic of its own command."""
    head = R.HEADS[h]
    out = []
    for w in range(u.x.W):
        obs, action, _, _, _, _, _, (hn, cn), command = R.gather_minibatch(u.x.cpu[w][0][h], u.x.cpu[w][1][h],
                                                                           list(u.x.idx[w, h]))
        n = command.shape[0]
        rows = torch.zeros(n, 3)
        with torch.no_grad():
            for c in range(4):
                sel = command[:, 0] == c
                if not sel.any():
                    continue
                xs = obs.view(8, n, -1)[:, sel].reshape(-1, obs.shape[-1])     # time-major, this expert's rows
                feat, _ = R.lstm_forward(xs, hn[sel], cn[sel], u.sd[f"{head}_lstm_{c}"])
                v, lp, en = R.evaluate_actions(feat, action[sel], u.sd[f"{head}_ppo_{c}"])
                rows[sel] = torch.cat([v, lp, en], 1)
        out.append(rows)
    return torch.cat(out)


def test_routed_forward_rows_match_oracle(routed_update):
    """`evaluate` on the plan's rows against the oracle, per row. Besides the relative L2 over all rows, the worst
    row is bounded: a row routed to the wrong expert or written to the wrong slot moves its value by O(1), which a
    relative L2 over thousands of rows can hide."""
    u = routed_update
    ev = u.eng.evaluate(u.x.storages, u.x.advs, u.x.idx, u.flat).cpu()
    u.eng.check()
    for h in range(2):
        ref = _oracle_rows(u, h).double()
        got = ev[h, :, :3].double()
        rels = [rel(got[:, k], ref[:, k]) for k in range(3)]
        worst = ((got - ref).abs().max(0).values / ref.pow(2).mean(0).sqrt()).tolist()
        print(f"{u.plan} {R.HEADS[h]}: rel-L2 value / log-prob / entropy {rels[0]:.2e} / {rels[1]:.2e} / "
              f"{rels[2]:.2e}, worst row / rms {worst[0]:.2e} / {worst[1]:.2e} / {worst[2]:.2e}")
        assert rels[0] < 2e-3 and rels[1] < 1e-3 and rels[2] < 1e-4, (R.HEADS[h], rels)
        assert worst[0] < 2e-2 and worst[1] < 2e-2 and worst[2] < 1e-3, (R.HEADS[h], worst)


def _differing_modules(a, b):
    from cadre_b200 import ppo_params as P
    return [m for m in P.MODULE_ORDER
            if any(not torch.equal(P.tensor_view(a, m, n)[0], P.tensor_view(b, m, n)[0]) for n in P.module_param_names(m))]


def _fresh_engine_update(storages, advs, idx, flat, evaluate=False):
    """losses, gradients (and `evaluate` rows) of a newly created engine's first update on these inputs"""
    from cadre_b200 import ppo
    eng = ppo.PpoEngine(idx.shape[0], idx.shape[2], device=DEV)
    grads = _stale_grads(flat)
    losses = eng.update(storages, advs, idx, flat, grads)
    eng.check()
    ev = eng.evaluate(storages, advs, idx, flat) if evaluate else None
    eng.check()
    return losses, grads, ev


# one engine, in this order; shift 1 moves every command c to c + 1 (the 400-row expert too)
REUSE_SEQUENCE = (("one_expert", 0), ("tile_edges", 0), ("kblock_edges", 0), ("skewed", 0), ("one_expert", 1),
                  ("tile_edges", 1))


def test_engine_reused_across_routings_is_bit_exact():
    """The update is bit-deterministic (fixed reduction orders, no float atomics), so an engine that has run other
    routings must give the bits of a fresh engine. Each shrink happens inside one expert, whose scratch rows past the
    new count still hold the previous update's values: throttle command 0 goes 400 -> 31 rows (one_expert ->
    tile_edges: the fp16 LSTM weight-gradient GEMMs read rows up to 35, past the BPTT kernel's zero fill up to 32),
    steer command 0 128 -> 95 (tile_edges -> kblock_edges: rows up to 99, zero fill up to 96), and throttle command 1
    400 -> 31 in the shifted pair. An `evaluate` runs between the updates."""
    from cadre_b200 import ppo, ppo_params as P
    flat = P.pack_state(R.ppo_fixture_state(0), DEV)
    eng = ppo.PpoEngine(4, 100, device=DEV)
    grads = _stale_grads(flat)
    prev = "new engine"
    for k, (plan, shift) in enumerate(REUSE_SEQUENCE):
        x = _config_inputs(4, 100, 200, 5000 + 100 * k, plan, shift)
        step = f"{prev} -> {plan}" + (f" (commands + {shift})" if shift else "")
        losses = eng.update(x.storages, x.advs, x.idx, flat, grads)
        eng.check()
        ref_losses, ref_grads, ref_ev = _fresh_engine_update(x.storages, x.advs, x.idx, flat, evaluate=True)
        assert torch.equal(losses, ref_losses), step
        assert torch.equal(grads, ref_grads), (step, _differing_modules(grads, ref_grads))
        ev = eng.evaluate(x.storages, x.advs, x.idx, flat)
        eng.check()
        assert torch.equal(ev, ref_ev), step
        prev = plan + (f" (commands + {shift})" if shift else "")


def test_staged_updates_across_routings_are_bit_exact():
    """update_staged takes its minibatch indices from the device-side table and advances the step counter itself.
    Three staged steps, no Adam step in between: slice A (storage rows 0..99, which carry one command per head: all
    400 rows of a head in one expert), slice B (rows 100..199: that expert gets 31 rows, the other three 129 / 127 /
    113), A again - a shrink 400 -> 31 and a growth back inside one expert. Every step's losses and gradients equal
    a fresh engine's `update` on that slice bit for bit."""
    from cadre_b200 import ppo, ppo_params as P
    W, mb, T = 4, 100, 200
    big = (0, 3)                      # the command of slice A: steer 0, throttle 3
    rs = np.random.RandomState(41)
    cmds = []
    for h in range(2):
        order = [big[h]] + [c for c in range(4) if c != big[h]]
        tail = rs.permutation(np.repeat(order, (31, 129, 127, 113))).reshape(W, mb)
        cmds.append(np.concatenate([np.full((W, mb), big[h]), tail], 1))       # [W, T] commands of rows 0..T-1
    rows = np.arange(T)
    cpu = [_make_worker(w, T, 6000, ((rows, cmds[0][w]), (rows, cmds[1][w]))) for w in range(W)]
    storages = [(_dev(c[0][0]), _dev(c[0][1])) for c in cpu]
    advs = [(c[1][0].to(DEV).contiguous(), c[1][1].to(DEV).contiguous()) for c in cpu]
    A = np.array([[rs.permutation(mb) for _ in range(2)] for _ in range(W)], dtype=np.int32)
    B = np.array([[mb + rs.permutation(mb) for _ in range(2)] for _ in range(W)], dtype=np.int32)
    slices = np.stack([A, B, A])
    for h in range(2):                # the routing the docstring describes
        assert (cmds[h][:, :mb] == big[h]).all() and (cmds[h][:, mb:] == big[h]).sum() == 31
    flat = P.pack_state(R.ppo_fixture_state(0), DEV)
    eng = ppo.PpoEngine(W, mb, device=DEV)
    assert eng.stage(storages, advs, slices, first_adam_step=1) == 3
    staged = []
    for _ in range(3):
        grads, losses = _stale_grads(flat), torch.empty(W, 2, 3, device=DEV)
        eng.update_staged(flat, grads, losses)
        staged.append((losses, grads))
    eng.check()
    for k, name in enumerate(("A", "B", "A again")):
        ref_losses, ref_grads, _ = _fresh_engine_update(storages, advs, slices[k], flat)
        assert torch.equal(staged[k][0], ref_losses), name
        assert torch.equal(staged[k][1], ref_grads), (name, _differing_modules(staged[k][1], ref_grads))


@pytest.mark.parametrize("plan", ["one_expert", "tile_edges"])
def test_grad_groups_give_identical_gradients(plan):
    """The data-parallel learner splits the LSTM weight-gradient GEMMs into 1, 2, 4 or 8 groups of experts, each with
    one contiguous gradient range and one event; with 4 and 8 groups some groups hold only empty experts (zero-K
    GEMMs). Losses and gradients are bit-identical to one group, the ranges of groups 0 .. g-1 and of the actor-critic
    tensors (group -1) tile the flat buffer, and each range is final once its event has fired."""
    from cadre_b200 import ppo, ppo_params as P
    x = _config_inputs(4, 100, 200, _plan_seed(plan), plan)
    flat = P.pack_state(R.ppo_fixture_state(0), DEV)
    eng = ppo.PpoEngine(4, 100, device=DEV)
    side = torch.cuda.Stream(device=DEV)
    ref = None
    for groups in (1, 2, 4, 8):
        eng.set_grad_groups(groups)
        grads = _stale_grads(flat)
        losses = eng.update(x.storages, x.advs, x.idx, flat, grads)
        ids = list(range(groups)) + [-1]
        ranges = [eng.grad_range(i) for i in ids]
        snaps = []
        for i, (off, cnt, _, _) in zip(ids, ranges):   # copied by a stream that waits for this group's event only
            eng.wait_grads(i, side)
            with torch.cuda.stream(side):
                snaps.append(grads[off:off + cnt].clone())
        torch.cuda.synchronize()
        eng.check()
        end, mod = 0, 0
        for off, cnt, m0, m1 in ranges:
            assert (off, m0) == (end, mod) and cnt > 0 and m1 > m0, (groups, ranges)
            end, mod = off + cnt, m1
        assert (end, mod) == (P.TOTAL, 16), (groups, ranges)
        for i, (off, cnt, _, _), s in zip(ids, ranges, snaps):
            assert torch.equal(s, grads[off:off + cnt]), (groups, i)
        if ref is None:
            ref = (losses, grads)
        else:
            assert torch.equal(losses, ref[0]), groups
            assert torch.equal(grads, ref[1]), (groups, _differing_modules(grads, ref[1]))
