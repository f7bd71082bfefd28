"""Encoder parity on the B200: CUDA path (through the C ABI) vs reference-generated goldens and the oracle.
Tolerance (BASELINE north_star): encoder features within 1e-2 relative (bf16 operands, fp32 accumulate)."""
import os

import numpy as np
import pytest
import torch

from oracle import restate as R

pytestmark = pytest.mark.gpu

REL_FEATURE = 1e-2


def rel_l2(got, ref):
    got, ref = got.double().flatten(), ref.double().flatten()
    return ((got - ref).norm() / (ref.norm() + 1e-30)).item()


@pytest.fixture(scope="module")
def encoders():
    from cadre_b200.encoder import Encoder
    return {tag: Encoder(R.danet_fixture_state(0, peaky=pk), "cuda:0", max_batch=32)
            for tag, pk in (("base", False), ("peaky", True))}


@pytest.mark.parametrize("tag", ["base", "peaky"])
def test_latent_matches_reference_golden(encoders, golden_dir, tag):
    g = np.load(os.path.join(golden_dir, "encoder.npz"))
    tick = R.synthetic_tick(np.random.RandomState(1000))
    x = torch.from_numpy(R.pre_process(tick["rgb"], tick["route_fig"].copy())).cuda()
    enc = encoders[tag]
    lat = enc.forward_f32(x).cpu()
    ref = torch.from_numpy(g[f"{tag}_latent"])
    assert torch.isfinite(lat).all()
    assert rel_l2(lat, ref) < REL_FEATURE, rel_l2(lat, ref)
    # layer-4 activations (first 8 channels) against the reference's
    l4 = enc.debug_buffer(0, 8).view(8, 5, 8, 512).float().cpu().permute(0, 3, 1, 2)[:, :8]
    assert rel_l2(l4, torch.from_numpy(g[f"{tag}_l4_slice"])) < 2e-2


def test_u8_ingest_and_measurements_match_reference_golden(encoders, golden_dir):
    g = np.load(os.path.join(golden_dir, "agent_feature.npz"))
    rs = np.random.RandomState(2000)
    tick = R.synthetic_tick(rs)
    tick["route_fig"][3] = (rs.rand(256, 144) * 200).astype(np.uint8)   # non-binary: uint8 truncation quirk
    tick["route_fig"][5] = 0                                             # max == 0 branch
    feat = encoders["base"].forward_u8(torch.from_numpy(tick["rgb"]).cuda(),
                                       torch.from_numpy(tick["route_fig"]).cuda(),
                                       torch.from_numpy(tick["measurements"]).cuda()).cpu()
    ref = torch.from_numpy(g["feature"])
    assert feat.shape == (8, 530)
    assert rel_l2(feat[:, :512], ref[:, :512]) < REL_FEATURE
    assert torch.equal(feat[:, 512:], ref[:, 512:])      # measurement columns are exact (f64 -> f32 cast)


@pytest.mark.parametrize("B", [1, 3, 17, 32])
def test_ragged_batches_match_oracle(encoders, B):
    torch.set_num_threads(8)
    rs = np.random.RandomState(B)
    x = torch.from_numpy(rs.rand(B, 4, 144, 256).astype(np.float32))
    with torch.no_grad():
        ref = R.encoder_latent(x, R.danet_fixture_state(0))
    lat = encoders["base"].forward_f32(x.cuda()).cpu()
    assert rel_l2(lat, ref) < REL_FEATURE


def test_batch_chunking_is_consistent(encoders):
    rs = np.random.RandomState(9)
    x = torch.from_numpy(rs.rand(40, 4, 144, 256).astype(np.float32)).cuda()   # > max_batch: two chunks
    enc = encoders["base"]
    full = enc.forward_f32(x)
    part = enc.forward_f32(x[32:].contiguous())
    assert torch.equal(full[32:], part)


@pytest.mark.parametrize("tag", ["base", "peaky"])
def test_attention_stages_match_oracle(encoders, tag):
    """Intermediate maps of the DA head (danet.py:43-69): layer4, conv5a|conv5c, PAM (fp32 CUDA-core kernel),
    CAM (tensor-core mma.sync kernel, fp16 attention weights) and their fused sum, against the oracle."""
    import torch.nn.functional as F  # noqa: F401
    enc = encoders[tag]
    sd = R.danet_fixture_state(0, peaky=(tag == "peaky"))
    B = 5
    x = torch.from_numpy(np.random.RandomState(3).rand(B, 4, 144, 256).astype(np.float32))
    enc.forward_f32(x.cuda())
    with torch.no_grad():
        l4 = R.backbone(x, sd)
        f1 = R._conv_bn_relu(l4, sd, "da_head.conv5a")
        f2 = R._conv_bn_relu(l4, sd, "da_head.conv5c")
        sa, sc = R.pam(f1, sd), R.cam(f2, sd)
        fs = R._conv_bn_relu(sa, sd, "da_head.conv51") + R._conv_bn_relu(sc, sd, "da_head.conv52")

    def nhwc(buf, c):
        return enc.debug_buffer(buf, B).view(B, 5, 8, c).float().cpu().permute(0, 3, 1, 2)
    assert rel_l2(nhwc(0, 512), l4) < 5e-3
    h5 = nhwc(2, 256)
    assert rel_l2(h5[:, :128], f1) < 5e-3 and rel_l2(h5[:, 128:], f2) < 5e-3
    assert rel_l2(nhwc(3, 128), sa) < REL_FEATURE
    assert rel_l2(nhwc(4, 128), sc) < 5e-3
    assert rel_l2(nhwc(1, 128), fs) < REL_FEATURE


def test_fused_shortcut_matches_separate_downsample_launches():
    """layer2.0 / 3.0 / 4.0: the 1x1/stride-2 shortcut as extra k-blocks of conv2 (default) against the separate
    downsample conv + residual add (CADRE_NO_SHORTCUT_FUSION=1, read when the encoder is created)."""
    from cadre_b200.encoder import Encoder
    sd = R.danet_fixture_state(0)
    x = torch.from_numpy(np.random.RandomState(5).rand(7, 4, 144, 256).astype(np.float32)).cuda()
    fused_enc = Encoder(sd, "cuda:0", max_batch=8)
    fused = fused_enc.forward_f32(x).cpu()
    os.environ["CADRE_NO_SHORTCUT_FUSION"] = "1"
    try:
        plain_enc = Encoder(sd, "cuda:0", max_batch=8)
    finally:
        del os.environ["CADRE_NO_SHORTCUT_FUSION"]
    plain = plain_enc.forward_f32(x).cpu()
    assert plain_enc.launches_per_forward == fused_enc.launches_per_forward + 3   # counted during a forward
    assert rel_l2(fused, plain) < 2e-3          # the fused form keeps the shortcut in fp32 instead of rounding it to fp16
    with torch.no_grad():
        ref = R.encoder_latent(x.cpu(), sd)
    assert rel_l2(fused, ref) < REL_FEATURE and rel_l2(plain, ref) < REL_FEATURE


def test_two_encoders_on_two_streams_match_sequential(encoders):
    """bench.py's scheduling: independent chunks on two encoder instances / two streams give the results of one
    encoder on one stream, bit for bit."""
    from cadre_b200.encoder import Encoder
    sd = R.danet_fixture_state(0)
    enc_a, enc_b = encoders["base"], Encoder(sd, "cuda:0", max_batch=32)
    g = torch.Generator().manual_seed(11)
    rgb = torch.randint(0, 256, (64, 144, 256, 3), dtype=torch.uint8, generator=g).cuda()
    route = (torch.rand(64, 256, 144, generator=g) < 0.1).to(torch.uint8).mul(255).cuda()
    meas = torch.rand(64, 3, dtype=torch.float64, generator=g).cuda()
    ref = torch.cat([enc_a.forward_u8(rgb[s:s + 32], route[s:s + 32], meas[s:s + 32]) for s in (0, 32)])
    torch.cuda.synchronize()
    out = torch.empty_like(ref)
    streams = [torch.cuda.Stream(), torch.cuda.Stream()]
    for rep in range(3):
        out.zero_()
        torch.cuda.synchronize()
        for k, (e, s) in enumerate(((enc_a, 0), (enc_b, 32))):
            with torch.cuda.stream(streams[k]):
                e.forward_u8(rgb[s:s + 32], route[s:s + 32], meas[s:s + 32], out[s:s + 32])
        torch.cuda.synchronize()
        assert torch.equal(out, ref)


# ------------------------------------------------------------------------------------------------ benchmarked shapes
def _u8_frames(n, seed):
    g = torch.Generator().manual_seed(seed)
    rgb = torch.randint(0, 256, (n, 144, 256, 3), dtype=torch.uint8, generator=g)
    route = (torch.rand(n, 256, 144, generator=g) < 0.1).to(torch.uint8).mul(255)
    meas = torch.rand(n, 3, dtype=torch.float64, generator=g)
    return rgb, route, meas


def _oracle_features(rgb, route, meas, sd, rows):
    """agent_latent_feature (agent.py:97-112) for the selected frame indices, 8 frames per call like the reference."""
    out = []
    with torch.no_grad():
        for s in range(0, len(rows), 8):
            ix = rows[s:s + 8]
            out.append(R.agent_latent_feature(rgb[ix].numpy(), route[ix].numpy().copy(), meas[ix].numpy(), sd))
    return torch.cat(out)


@pytest.fixture(scope="module")
def bench_encoders():
    """bench.py's configuration: two encoder instances with max_batch = 640."""
    from cadre_b200.encoder import Encoder
    sd = R.danet_fixture_state(0)
    return [Encoder(sd, "cuda:0", max_batch=640) for _ in range(2)]


@pytest.mark.parametrize("B", [640, 1024])
def test_bench_batch_sizes_match_oracle(bench_encoders, B):
    """BASELINE config 2's top batch sizes on the encoder bench.py uses (max_batch = 640; 1024 = chunks of 640 + 384):
    EVERY frame against the CPU oracle."""
    torch.set_num_threads(min(16, os.cpu_count() or 1))
    rgb, route, meas = _u8_frames(B, seed=B)
    feat = bench_encoders[0].forward_u8(rgb.cuda(), route.cuda(), meas.cuda()).cpu()
    ref = _oracle_features(rgb, route, meas, R.danet_fixture_state(0), list(range(B)))
    assert feat.shape == (B, 530) and torch.isfinite(feat).all()
    assert torch.equal(feat[:, 512:], ref[:, 512:])
    assert rel_l2(feat[:, :512], ref[:, :512]) < REL_FEATURE
    per_frame = ((feat[:, :512] - ref[:, :512]).double().norm(dim=1) / ref[:, :512].double().norm(dim=1))
    assert per_frame.max().item() < 2 * REL_FEATURE, per_frame.max().item()     # no single frame is off either


def test_bench_two_stream_ramp_schedule(bench_encoders):
    """The ingest's e2e schedule (cadre_b200.ingest.chunk_schedule: a geometric start-up ramp 32, 96, 288, then chunks of
    640; round 1's 128 / 512 steps ride along) alternating between two encoder instances on two streams, each writing its rows of one [N,530] feature matrix through ld_out. Bit-identical to one encoder on one
    stream, and equal to the oracle on a sample of frames from every chunk."""
    sizes = [32, 96, 288, 640, 128, 512, 224]
    n = sum(sizes)
    rgb, route, meas = _u8_frames(n, seed=77)
    d = [t.cuda() for t in (rgb, route, meas)]
    one = bench_encoders[0].forward_u8(*d).clone()
    torch.cuda.synchronize()
    out = torch.zeros(n, 530, device="cuda")
    streams = [torch.cuda.Stream(), torch.cuda.Stream()]
    s0 = 0
    for i, m in enumerate(sizes):
        with torch.cuda.stream(streams[i % 2]):
            bench_encoders[i % 2].forward_u8(d[0][s0:s0 + m], d[1][s0:s0 + m], d[2][s0:s0 + m], out[s0:s0 + m])
        s0 += m
    torch.cuda.synchronize()
    assert torch.equal(out, one)
    rows = [0, 5, 31, 32, 127, 128, 300, 415, 416, 1000, 1055, 1056, 1183, 1184, 1500, 1695, 1696, 1919]   # every chunk + edges
    torch.set_num_threads(min(16, os.cpu_count() or 1))
    ref = _oracle_features(rgb, route, meas, R.danet_fixture_state(0), rows)
    assert rel_l2(out[rows, :512].cpu(), ref[:, :512]) < REL_FEATURE


def test_features_written_through_ld_out_into_rollout_obs(bench_encoders):
    """The learner writes encoder features straight into RolloutStorage.obs (row stride 530, arbitrary base)."""
    rgb, route, meas = _u8_frames(24, seed=5)
    d = [t.cuda() for t in (rgb, route, meas)]
    obs = torch.full((4, 8, 530), -7.0, device="cuda")       # [steps, seq, 530] like storage.obs[t0:t0+4]
    plain = bench_encoders[0].forward_u8(*d)
    bench_encoders[0].forward_u8(*d, out=obs[1:4].view(24, 530))
    assert torch.equal(obs[1:4].view(24, 530), plain) and float(obs[0].min()) == -7.0


# ------------------------------------------------------------------------------------------------ dynamic range
@pytest.mark.parametrize("tag", ["xavier", "wide"])
def test_fp16_dynamic_range_fixtures(tag):
    """SURVEY §8c.3 fixtures beyond base / peaky: (xavier) the reference trainer's initialisation
    (experiments_builder.py:163-188): activations two orders of magnitude below the base fixture's; (wide) calibrated
    BatchNorm statistics spanning running_var 1e-5 .. 1e+5 with gammas up to 5. Latent within 1e-2 and no 16-bit store
    anywhere near saturation."""
    from cadre_b200.encoder import Encoder
    torch.set_num_threads(8)
    sd = R.danet_fixture_state(0, init="xavier") if tag == "xavier" else R.danet_wide_fixture_state(0)
    if tag == "wide":
        v = torch.cat([t.flatten() for k, t in sd.items() if k.endswith("running_var")])
        assert v.min().item() < 1e-3 and v.max().item() > 1e3
    enc = Encoder(sd, "cuda:0", max_batch=16)
    x = torch.from_numpy(np.random.RandomState(17).rand(12, 4, 144, 256).astype(np.float32))
    lat = enc.forward_f32(x.cuda()).cpu()
    with torch.no_grad():
        ref = R.encoder_latent(x, sd)
    assert torch.isfinite(lat).all()
    assert rel_l2(lat, ref) < REL_FEATURE, rel_l2(lat, ref)
    assert enc.activation_absmax(12) < 0.25 * 65504.0


def test_intertask_stage_matches_oracle(encoders):
    """a7 (intertask_att.py:39-80, 123-176) as its own stage: the six Linear(20480,512)+LeakyReLU hidden vectors that
    the library computes as ONE folded [5120 -> 3072] GEMM (conv8 and the two 1x1 task convs folded in) against the
    oracle's unfolded conv8 -> visual_conv / bc_conv -> flatten -> Linear chain."""
    import torch.nn.functional as F
    enc = encoders["base"]
    sd = R.danet_fixture_state(0)
    B = 6
    x = torch.from_numpy(np.random.RandomState(23).rand(B, 4, 144, 256).astype(np.float32))
    lat = enc.forward_f32(x.cuda()).cpu()
    with torch.no_grad():
        da = R.da_head(R.backbone(x, sd), sd)
        hid = []
        for task, conv in (("visual", "visual_conv"), ("bc", "bc_conv")):
            t = F.conv2d(da, sd[conv + ".weight"], sd[conv + ".bias"]).reshape(B, -1)
            for role in ("query", "key", "value"):
                p = f"inter_task_att.{task}_{role}_layer"
                hid.append(F.leaky_relu(F.linear(t, sd[p + ".1.weight"], sd[p + ".1.bias"]), 0.01))
        hid = torch.cat(hid, 1)                                           # [B, 6*512] in the library's order
        ref = R.encoder_latent(x, sd)
    got = enc.debug_buffer(5, B).view(B, 3072).float().cpu()
    assert rel_l2(got, hid) < 5e-3, rel_l2(got, hid)
    assert rel_l2(lat, ref) < REL_FEATURE


# ----------------------------------------------------------------------------------------------------------------------
# layer2 on zero-bordered activations: halo-reuse 128 -> 128 kernel (csrc/tc_halo128.cuh) and bordered conv outputs
def _conv_ops():
    from cadre_b200 import _lib
    return _lib, _lib.lib(), _lib.enc_dtype()


@pytest.mark.parametrize("B,res,act", [(1, False, 1), (3, True, 1), (37, True, 1), (640, False, 1), (3, True, 0),
                                       (37, False, 0)])
def test_halo128_conv_matches_fp32_conv_and_implicit_gemm_kernel(B, res, act):
    """cadre_conv3x3_flat128 (BasicBlock conv of ResNet layer2, resnet.py:39-55: conv3x3 + folded BN bias (+ residual)
    (+ ReLU) on [B][20][34][128] bordered activations) against the float64 convolution of the same fp16 operands,
    element by element (the bound of test_encoder_kernels_gpu.py), and against the implicit-GEMM kernel
    (cadre_conv2d_nhwc) it replaces; the zero border must come back exactly zero and nothing outside the output may
    change. B = 37 gives an odd number of 128-pixel tiles (the last group's second tile is empty), B = 640 is the
    benchmarked chunk."""
    import torch.nn.functional as F
    from test_encoder_kernels_gpu import C_ACC, Guarded, _border_is, _check_bound
    _lib, L, dt = _conv_ops()
    H, W, C = 18, 32, 128
    g = torch.Generator(device="cuda").manual_seed(100 + B)
    x = torch.randn(B, C, H, W, device="cuda", generator=g).to(dt)
    w = (torch.randn(C, C, 3, 3, device="cuda", generator=g) / (C * 9) ** 0.5).to(dt)
    bias = torch.randn(C, device="cuda", generator=g)
    xp = torch.zeros(B, H + 2, W + 2, C, device="cuda", dtype=dt)
    xp[:, 1:-1, 1:-1] = x.permute(0, 2, 3, 1)
    w_k = w.permute(0, 2, 3, 1).contiguous().view(C, -1)
    r = rp = None
    if res:
        r = torch.randn(B, H, W, C, device="cuda", generator=g).to(dt)
        rp = torch.zeros_like(xp)
        rp[:, 1:-1, 1:-1] = r
    guarded = Guarded((B, H + 2, W + 2, C), 7.0, dtype=dt)
    out = guarded.t
    _lib.check(L.cadre_conv3x3_flat128(_lib.ptr(xp), B, H, W, _lib.ptr(w_k), _lib.ptr(bias), _lib.ptr(rp), act,
                                       _lib.ptr(out), _lib.stream_ptr()))
    old = torch.full((B, H, W, C), 7.0, device="cuda", dtype=dt)
    _lib.check(L.cadre_conv2d_nhwc(_lib.ptr(xp), B, H, W, C, _lib.ptr(w_k), C, 3, 3, 1, 1, _lib.ptr(bias), _lib.ptr(r), 0,
                                   act, _lib.ptr(old), 1, _lib.stream_ptr()))
    torch.cuda.synchronize()
    guarded.check()
    ref = F.conv2d(x.double(), w.double(), bias.double(), stride=1, padding=1)
    S = F.conv2d(x.double().abs(), w.double().abs(), bias.double().abs(), stride=1, padding=1)
    if res:
        ref = ref + r.double().permute(0, 3, 1, 2)
        S = S + r.double().abs().permute(0, 3, 1, 2)
    if act:
        ref = ref.relu()
    ref, S = ref.permute(0, 2, 3, 1), S.permute(0, 2, 3, 1)
    got = out[:, 1:-1, 1:-1].float()
    assert _border_is(out, 0.0)
    _check_bound("halo128", got, ref, S, C_ACC["halo128"])
    assert rel_l2(got, ref) < 1e-3                       # fp16 output rounding only (2^-11 relative per element)
    assert rel_l2(got, old.float()) < 1e-3
    assert float((got - ref).abs().max()) < 2e-2 * float(ref.abs().max())


def test_conv_with_bordered_output_equals_plain_output():
    """cadre_conv2d_nhwc_bordered_out (layer2.0.conv1: 3x3 / stride 2, 64 -> 128, bordered input) writes exactly the
    values of cadre_conv2d_nhwc into the interior of a [B][20][34][128] tensor and never touches the border."""
    _lib, L, dt = _conv_ops()
    B, H, W, Cin, Cout = 5, 36, 64, 64, 128
    g = torch.Generator(device="cuda").manual_seed(7)
    xp = torch.zeros(B, H + 2, W + 2, Cin, device="cuda", dtype=dt)
    xp[:, 1:-1, 1:-1] = torch.randn(B, H, W, Cin, device="cuda", generator=g).to(dt)
    w_k = (torch.randn(Cout, 9 * Cin, device="cuda", generator=g) / 24.0).to(dt)
    bias = torch.randn(Cout, device="cuda", generator=g)
    plain = torch.zeros(B, 18, 32, Cout, device="cuda", dtype=dt)
    _lib.check(L.cadre_conv2d_nhwc(_lib.ptr(xp), B, H, W, Cin, _lib.ptr(w_k), Cout, 3, 3, 2, 1, _lib.ptr(bias), None, 0, 1,
                                   _lib.ptr(plain), 1, _lib.stream_ptr()))
    bord = torch.full((B, 20, 34, Cout), -3.0, device="cuda", dtype=dt)
    _lib.check(L.cadre_conv2d_nhwc_bordered_out(_lib.ptr(xp), B, H, W, Cin, _lib.ptr(w_k), Cout, 3, 3, 2, 1, _lib.ptr(bias),
                                                1, _lib.ptr(bord), 1, _lib.stream_ptr()))
    torch.cuda.synchronize()
    assert torch.equal(bord[:, 1:-1, 1:-1], plain) and float(plain.float().abs().max()) > 0
    edge = bord.clone()
    edge[:, 1:-1, 1:-1] = -3.0
    assert bool((edge == -3.0).all())


def test_layer2_halo_path_matches_default_path_and_oracle():
    """The encoder with layer2 on zero-bordered activations (CADRE_LAYER2_HALO, read when the encoder is created) against
    the implicit-GEMM layer2 and the oracle, at a ragged batch and at the benchmarked chunk size."""
    from cadre_b200.encoder import Encoder
    sd = R.danet_fixture_state(0)
    keep = os.environ.get("CADRE_LAYER2_HALO")
    try:
        os.environ["CADRE_LAYER2_HALO"] = "1"
        halo = Encoder(sd, "cuda:0", max_batch=640)
        os.environ["CADRE_LAYER2_HALO"] = "0"
        plain = Encoder(sd, "cuda:0", max_batch=640)
    finally:
        if keep is None:
            os.environ.pop("CADRE_LAYER2_HALO", None)
        else:
            os.environ["CADRE_LAYER2_HALO"] = keep
    x = torch.from_numpy(np.random.RandomState(11).rand(7, 4, 144, 256).astype(np.float32)).cuda()
    a, b = halo.forward_f32(x).cpu(), plain.forward_f32(x).cpu()
    assert halo.launches_per_forward == plain.launches_per_forward
    with torch.no_grad():
        ref = R.encoder_latent(x.cpu(), sd)
    assert rel_l2(a, b) < 2e-3 and rel_l2(a, ref) < REL_FEATURE
    rgb, route, meas = _u8_frames(640, seed=91)
    d = [t.cuda() for t in (rgb, route, meas)]
    fa, fb = halo.forward_u8(*d).clone(), plain.forward_u8(*d).clone()
    torch.cuda.synchronize()
    assert rel_l2(fa[:, :512], fb[:, :512]) < 2e-3 and torch.equal(fa[:, 512:], fb[:, 512:])
    fa2 = halo.forward_u8(*d)                   # the bordered buffers keep their zero border across forwards
    torch.cuda.synchronize()
    assert torch.equal(fa, fa2)
