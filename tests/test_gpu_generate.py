"""Sampling-path parity on the GPU: the persistent kernel (through the C ABI / WaveNetModel.generate_fast) vs the
golden streams of the unmodified reference.  Bar: bit-exact mu-law indices on the argmax path (a divergence is
accepted only at a step where the reference's own top-1/top-2 margin is < 1e-4), per-step logits within 1e-4."""
import numpy as np
import pytest
import torch

from oracle import wavenet_oracle as O
from helpers import build_model, snapshot_model, one_hot_cuda, rel_err, assert_stream_parity, params_from_golden

pytestmark = pytest.mark.gpu
TOL = 1e-4


def audio_of(idx, classes=256):
    return O.mu_law_expansion((np.asarray(idx) / classes) * 2.0 - 1.0, classes)


@pytest.mark.parametrize("name", ["cfg1", "odd_bias", "k3", "deep"])
def test_generate_matches_reference_golden(golden, name):
    g = golden(f"net_{name}.npz")
    m = build_model(g)
    first = g["first"]
    # argmax path through the reference-facing API
    audio = m.generate_fast(24, first_samples=torch.from_numpy(first), temperature=0.0)
    assert audio.dtype == np.float64 and audio.shape == (24,) and m.training
    n_ok = assert_stream_parity(np.rint((O.mu_law_encoding(audio, 256) + 1) * 128).astype(np.int64),
                                g["gen_argmax_idx"], g["gen_argmax_logits"])
    assert np.array_equal(audio[:n_ok], g["gen_argmax_audio"][:n_ok])
    # teacher-forced per-step logits
    idx, logits = m.generate_fast_batch(24, first[None, :], temperature=0.0, forced=g["gen_argmax_idx"][None, :],
                                        return_logits=True)
    assert rel_err(logits[0], g["gen_argmax_logits"]) < TOL
    # sampled path: numpy global RNG seeded like the reference run
    np.random.seed(7)
    audio = m.generate_fast(24, first_samples=first, temperature=0.8, regularize=1e-4)
    np.random.seed(7)
    assert np.array_equal(np.random.random_sample(24), g["gen_sample_uniforms"])
    got = np.rint((O.mu_law_encoding(audio, 256) + 1) * 128).astype(np.int64)
    if not np.array_equal(got, g["gen_sample_idx"]):
        # a draw may land on the other side of a CDF edge only if u is within float noise of that edge
        i = int(np.nonzero(got != g["gen_sample_idx"])[0][0])
        lg = g["gen_sample_logits"][i].astype(np.float64)
        reg = 1e-4 * (np.arange(256) - 128.0) ** 2
        p = np.exp((lg - reg) / 0.8 - ((lg - reg) / 0.8).max()); p /= p.sum()
        cdf = np.cumsum(p)
        assert np.abs(cdf - g["gen_sample_uniforms"][i]).min() < 1e-5, f"sampled stream diverges at step {i}"
    else:
        assert np.array_equal(audio, g["gen_sample_audio"])


def test_generate_snapshot_real_audio(golden):
    gs, gio = golden("snapshot_chaconne_state.npz"), golden("snapshot_chaconne_io.npz")
    m = snapshot_model(gs)
    rf = int(gs["receptive_field"])
    clip = gio["clip"].astype(np.int64)
    idx = m.generate_fast_batch(200, clip[None, :rf], temperature=0.0)
    n_ok = assert_stream_parity(idx[0], gio["gen_argmax_idx"], gio["gen_argmax_logits"])
    assert n_ok >= 8 and idx[0][:8].tolist() == [177, 177, 177, 174, 174, 177, 181, 188]
    _, logits = m.generate_fast_batch(200, clip[None, :rf], temperature=0.0, forced=gio["gen_argmax_idx"][None, :],
                                      return_logits=True)
    assert rel_err(logits[0], gio["gen_argmax_logits"]) < TOL
    # forward() == generate_fast() teacher-forced on the real continuation (SURVEY.md section 3.2)
    _, tf = m.generate_fast_batch(64, clip[None, :rf], temperature=0.0, forced=clip[None, rf:rf + 64], return_logits=True)
    with torch.no_grad():
        fwd = m(one_hot_cuda(clip[None, :rf + 63]))
    assert rel_err(tf[0], fwd.cpu().numpy()) < TOL


def test_generate_cfg2_net(golden):
    g = golden("net_cfg2.npz")
    m = build_model(g)
    idx, logits = m.generate_fast_batch(48, np.array([[128]]), temperature=0.0, return_logits=True)
    assert_stream_parity(idx[0], g["gen_argmax_idx"], g["gen_argmax_logits"])
    _, logits = m.generate_fast_batch(48, np.array([[128]]), temperature=0.0, forced=g["gen_argmax_idx"][None, :],
                                      return_logits=True)
    assert rel_err(logits[0], g["gen_argmax_logits"]) < TOL
    np.random.seed(0)
    audio = m.generate_fast(48, first_samples=g["gen_sample_first"], temperature=1.0)
    got = np.rint((O.mu_law_encoding(audio, 256) + 1) * 128).astype(np.int64)
    _, lg = m.generate_fast_batch(48, g["gen_sample_first"][None, :], temperature=1.0,
                                  uniforms=g["gen_sample_uniforms"][None, :], forced=g["gen_sample_idx"][None, :],
                                  return_logits=True)
    assert rel_err(lg[0], g["gen_sample_logits"]) < TOL
    # the free-running sampled stream: identical, or it parts ways at a draw whose uniform lies within float noise of
    # a CDF edge of the reference's own distribution (the classification used for the small nets above)
    if not np.array_equal(got, g["gen_sample_idx"]):
        i = int(np.nonzero(got != g["gen_sample_idx"])[0][0])
        lg64 = g["gen_sample_logits"][i].astype(np.float64)
        pr = np.exp(lg64 - lg64.max()); pr /= pr.sum()
        edge = np.abs(np.cumsum(pr) - g["gen_sample_uniforms"][i]).min()
        assert edge < 1e-5, f"sampled stream diverges at step {i}, {edge:.3e} away from the nearest CDF edge"


def test_streams_are_independent_and_bitwise_reproducible(golden):
    g = golden("net_deep.npz")
    m = build_model(g)
    rng = np.random.RandomState(5)
    firsts = rng.randint(0, 256, size=(5, 40))
    uni = rng.random_sample((5, 30))
    multi, mlog = m.generate_fast_batch(30, firsts, temperature=0.9, uniforms=uni, return_logits=True)
    for s in range(5):
        single, slog = m.generate_fast_batch(30, firsts[s:s + 1], temperature=0.9, uniforms=uni[s:s + 1], return_logits=True)
        assert np.array_equal(single[0], multi[s]) and np.array_equal(slog[0], mlog[s])
    # 64 streams of the cfg-4 shape run in one launch
    idx = m.generate_fast_batch(8, rng.randint(0, 256, size=(64, 3)), temperature=0.0)
    assert idx.shape == (64, 8) and idx.min() >= 0 and idx.max() < 256


def test_progress_callback_schedule_and_queue_export(golden):
    g = golden("net_odd_bias.npz")
    m = build_model(g)
    first = g["first"]                                   # 18 given samples
    calls = []
    m.generate_fast(24, first_samples=first, temperature=0.0, progress_callback=lambda i, n: calls.append((i, n)),
                    progress_interval=5)
    total = len(first) + 24
    want = [(i, total) for i in range(len(first) - 1) if i % 5 == 0]
    want += [(i + len(first), total) for i in range(24) if (i + len(first)) % 5 == 0]
    assert calls == want                                 # reference wavenet_model.py:266-269, :309-311
    # the exported queues hold what the oracle's queues hold after the same run
    p, spec = params_from_golden(g), None
    from helpers import spec_from_golden
    spec = spec_from_golden(g)
    evals = len(first) - 1 + 24
    for i, q in enumerate(m.dilated_queues):
        assert q.data.shape == (spec.residual_channels, q.max_length) and q.in_pos == evals % q.max_length
    # layer 0's queue holds start_conv columns of the last inputs: check against the weights directly
    q0 = m.dilated_queues[0]
    w = m.start_conv.weight.detach()[:, :, 0]
    b = m.start_conv.bias.detach()
    last_in = int(g["gen_argmax_idx"][22])               # input of the last evaluation = sample chosen before it
    col = q0.data[:, (evals - 1) % q0.max_length]
    assert torch.allclose(col, w[:, last_in] + b, atol=1e-6)


@pytest.mark.parametrize("name", ["odd_bias", "deep", "k3"])
def test_exchange_modes_agree(golden, name):
    """The flag-in-data kernel (default) and the grid-barrier kernel implement the same schedule."""
    g = golden(f"net_{name}.npz")
    m = build_model(g)
    rng = np.random.RandomState(11)
    firsts = rng.randint(0, 256, size=(3, 25))
    uni = rng.random_sample((3, 40))
    res = {}
    for mode in (0, 1, 2):
        m._runtime().gen_mode = mode
        res[mode] = m.generate_fast_batch(40, firsts, temperature=0.7, uniforms=uni, forced=None, return_logits=True)
        _, lg = m.generate_fast_batch(24, g["first"][None, :], temperature=0.0, forced=g["gen_argmax_idx"][None, :],
                                      return_logits=True)
        assert rel_err(lg[0], g["gen_argmax_logits"]) < TOL
    m._runtime().gen_mode = None
    (i0, l0), (i1, l1) = res[0], res[1]
    same = (i0 == i1).all(axis=1)
    for s in range(3):                      # streams may only part ways after a step where the logits differ by rounding
        n = 40 if same[s] else int(np.nonzero(i0[s] != i1[s])[0][0])
        assert n >= 1 and rel_err(l0[s, :n + 1], l1[s, :n + 1]) < 1e-5


def test_fast_kernel_equals_generic_kernel_bitwise(golden):
    """cfg 2 net, single stream: the register-polling kernel (mode 0) and the generic flag-exchange kernel (mode 2)
    share the K split and summation order, so logits and indices are identical bit for bit; a 3-stream run (generic
    kernel) reproduces the single-stream run of each stream."""
    g = golden("net_cfg2.npz")
    m = build_model(g)
    rt = m._runtime()
    rng = np.random.RandomState(3)
    first = rng.randint(0, 256, size=(3, 7))
    uni = rng.random_sample((3, 40))
    out = {}
    for mode in (3, 2):
        rt.gen_mode = mode
        out[mode] = [m.generate_fast_batch(40, first[s:s + 1], temperature=1.0, uniforms=uni[s:s + 1], return_logits=True)
                     for s in range(3)]
    for s in range(3):
        assert np.array_equal(out[3][s][0], out[2][s][0]) and np.array_equal(out[3][s][1], out[2][s][1])
    rt.gen_mode = 2
    multi_idx, multi_lg = m.generate_fast_batch(40, first, temperature=1.0, uniforms=uni, return_logits=True)
    rt.gen_mode = None
    for s in range(3):
        assert np.array_equal(multi_idx[s], out[3][s][0][0]) and np.array_equal(multi_lg[s], out[3][s][1][0])
    # argmax + warm-up + chunked launches (progress callback) through the fast kernel
    calls = []
    a = m.generate_fast(30, first_samples=first[0], temperature=0.0, progress_callback=lambda i, n: calls.append(i),
                        progress_interval=7)
    b = m.generate_fast(30, first_samples=first[0], temperature=0.0)
    assert np.array_equal(a, b) and len(calls) > 3


def test_two_level_exchange_kernel_bitwise_and_golden(golden):
    """cfg 2 net, single stream: the two-level exchange kernel (mode 5: DSMEM inside a cluster, one L2 poller per remote
    producer) keeps kernel 3's row split and summation order -- logits and indices identical bit for bit, over warm-up
    samples, sampling with temperature, chunked launches that continue a session, and the golden teacher-forced stream."""
    g = golden("net_cfg2.npz")
    m = build_model(g)
    rt = m._runtime()
    rng = np.random.RandomState(5)
    first = rng.randint(0, 256, size=(2, 11))
    uni = rng.random_sample((2, 300))
    out = {}
    for mode in (5, 3):
        rt.gen_mode = mode
        out[mode] = [m.generate_fast_batch(300, first[s:s + 1], temperature=1.0, uniforms=uni[s:s + 1], return_logits=True)
                     for s in range(2)]
        _, lg = m.generate_fast_batch(48, np.array([[128]]), temperature=0.0, forced=g["gen_argmax_idx"][None, :],
                                      return_logits=True)
        assert rel_err(lg[0], g["gen_argmax_logits"]) < TOL
    for s in range(2):
        assert np.array_equal(out[5][s][0], out[3][s][0]) and np.array_equal(out[5][s][1], out[3][s][1])
    rt.gen_mode = 5
    calls = []
    a = m.generate_fast(700, first_samples=first[0], temperature=0.0, progress_callback=lambda i, n: calls.append(i),
                        progress_interval=64)
    b = m.generate_fast(700, first_samples=first[0], temperature=0.0)
    rt.gen_mode = 3
    c = m.generate_fast(700, first_samples=first[0], temperature=0.0)
    rt.gen_mode = None
    assert np.array_equal(a, b) and np.array_equal(b, c) and len(calls) > 3


def test_cluster_kernel_cfg2(golden):
    """The cluster (distributed shared memory) kernel is what a 256-channel net runs by default: golden parity,
    agreement with the L2 kernels, and multi-stream == single-stream bit for bit (one cluster per stream)."""
    g = golden("net_cfg2.npz")
    m = build_model(g)
    rt = m._runtime()
    rng = np.random.RandomState(8)
    first = rng.randint(0, 256, size=(5, 9))
    uni = rng.random_sample((5, 60))
    rt.gen_mode = 4
    idx4, lg4 = m.generate_fast_batch(60, first, temperature=1.0, uniforms=uni, return_logits=True)
    singles = [m.generate_fast_batch(60, first[s:s + 1], temperature=1.0, uniforms=uni[s:s + 1], return_logits=True)
               for s in range(5)]
    for s in range(5):
        assert np.array_equal(singles[s][0][0], idx4[s]) and np.array_equal(singles[s][1][0], lg4[s])
    # teacher-forced logits against the reference's golden stream
    _, lg = m.generate_fast_batch(48, np.array([[128]]), temperature=0.0, forced=g["gen_argmax_idx"][None, :],
                                  return_logits=True)
    assert rel_err(lg[0], g["gen_argmax_logits"]) < TOL
    idx, _ = m.generate_fast_batch(48, np.array([[128]]), temperature=0.0, return_logits=True)
    assert_stream_parity(idx[0], g["gen_argmax_idx"], g["gen_argmax_logits"])
    # against the generic L2 kernel on the same inputs (teacher forced so rounding cannot fork the streams)
    rt.gen_mode = 2
    _, lg2 = m.generate_fast_batch(60, first[:2], temperature=1.0, uniforms=uni[:2], forced=idx4[:2], return_logits=True)
    rt.gen_mode = 4
    _, lg4f = m.generate_fast_batch(60, first[:2], temperature=1.0, uniforms=uni[:2], forced=idx4[:2], return_logits=True)
    rt.gen_mode = None
    assert rel_err(lg4f, lg2) < 1e-5
    # chunked launches (progress callback) continue the cluster kernel's state correctly
    calls = []
    a = m.generate_fast(40, first_samples=first[0], temperature=0.0, progress_callback=lambda i, n: calls.append(i),
                        progress_interval=9)
    b = m.generate_fast(40, first_samples=first[0], temperature=0.0)
    assert np.array_equal(a, b) and len(calls) > 3


def test_batched_cluster_kernel_cfg2(golden):
    """The batched tensor-core cluster kernel (mode 6: 8 streams per 16-CTA cluster, bf16 hi/lo pair MMAs, bulk-copy
    exchange) is what several streams of a 256-channel net run by default.  A stream's result does not depend on its
    slot, its cluster or its company (bitwise); logits follow the reference's golden stream and the fp32 L2 kernel;
    launches that continue a session reproduce the single launch."""
    g = golden("net_cfg2.npz")
    m = build_model(g)
    rt = m._runtime()
    rng = np.random.RandomState(21)
    first = rng.randint(0, 256, size=(11, 9))             # 11 streams: one full cluster and a partial one
    uni = rng.random_sample((11, 60))
    rt.gen_mode = 6
    idx6, lg6 = m.generate_fast_batch(60, first, temperature=1.0, uniforms=uni, return_logits=True)
    for sub in ([0, 9], [3, 10], [8, 1, 5]):
        i2, l2 = m.generate_fast_batch(60, first[sub], temperature=1.0, uniforms=uni[sub], return_logits=True)
        for j, s in enumerate(sub):
            assert np.array_equal(i2[j], idx6[s]) and np.array_equal(l2[j], lg6[s])
    # teacher-forced logits against the reference's golden stream; both slots identical
    two = np.array([[128], [128]])
    _, lg = m.generate_fast_batch(48, two, temperature=0.0, forced=np.stack([g["gen_argmax_idx"]] * 2), return_logits=True)
    assert rel_err(lg[0], g["gen_argmax_logits"]) < TOL and np.array_equal(lg[0], lg[1])
    idx, _ = m.generate_fast_batch(48, two, temperature=0.0, return_logits=True)
    assert_stream_parity(idx[0], g["gen_argmax_idx"], g["gen_argmax_logits"])
    # against the generic fp32 L2 kernel on the same inputs (teacher forced so rounding cannot fork the streams)
    rt.gen_mode = 2
    _, lg2 = m.generate_fast_batch(60, first[:3], temperature=1.0, uniforms=uni[:3], forced=idx6[:3], return_logits=True)
    rt.gen_mode = 6
    _, lg6f = m.generate_fast_batch(60, first[:3], temperature=1.0, uniforms=uni[:3], forced=idx6[:3], return_logits=True)
    assert rel_err(lg6f, lg2) < 2e-5
    # chunked launches continue the rings, indices and barrier phases of the previous launch
    calls = []
    with torch.cuda.device(rt.device()):
        a, la, _ = rt.generate(700, first[:3].astype(np.int32), 0.0, 0.0, want_logits=True,
                               callbacks=[(e, lambda: calls.append(1)) for e in (5, 8, 100, 513, 600)])
        b, lb, _ = rt.generate(700, first[:3].astype(np.int32), 0.0, 0.0, want_logits=True)
    rt.gen_mode = None
    assert np.array_equal(a, b) and np.array_equal(la, lb) and len(calls) == 5
    # the default for several streams of this net is this kernel
    d, ld = m.generate_fast_batch(60, first, temperature=1.0, uniforms=uni, return_logits=True)
    assert np.array_equal(d, idx6) and np.array_equal(ld, lg6)
    # 64 streams (8 clusters: more than the 7 sixteen-CTA clusters a B200 holds, so the 8-CTA-cluster variant runs) equal
    # the same streams run 11 at a time
    first64 = np.concatenate([first] * 6)[:64]
    uni64 = np.concatenate([uni] * 6)[:64]
    i64, l64 = m.generate_fast_batch(60, first64, temperature=1.0, uniforms=uni64, return_logits=True)
    for s in range(64):
        assert np.array_equal(i64[s], idx6[s % 11]) and np.array_equal(l64[s], lg6[s % 11])
    # in-place weight updates reach the pre-split weight images (wn_gen_weights_changed)
    with torch.no_grad():
        m.end_conv_2.weight.mul_(0.5)
        m.filter_convs[3].weight.add_(0.01)
        m.skip_convs[7].weight.mul_(1.5)
    _, la = m.generate_fast_batch(60, first[:3], temperature=1.0, uniforms=uni[:3], forced=idx6[:3], return_logits=True)
    rt.gen_mode = 2
    _, lb = m.generate_fast_batch(60, first[:3], temperature=1.0, uniforms=uni[:3], forced=idx6[:3], return_logits=True)
    rt.gen_mode = None
    assert rel_err(la, lb) < 2e-5 and rel_err(la, lg6f) > 1e-2


def test_cfg4_64_streams_vs_oracle(golden):
    """cfg 4: 64 independent streams of the cfg-2 net in one launch.  The reference has no batch dimension in its queues
    (wavenet_model.py:179), so the oracle is 64 single-stream runs: teacher-forced per-step logits of EVERY stream within
    1e-4, and the free-running argmax streams bit-exact up to a reference near-tie."""
    g = golden("net_cfg2.npz")
    m = build_model(g)
    from helpers import spec_from_golden
    spec, p = spec_from_golden(g), params_from_golden(g)
    if not p:
        p = O.init_params(spec, seed=0)
    NS, n = 64, 32
    rng = np.random.RandomState(21)
    firsts = rng.randint(0, 256, size=(NS, 2))
    torch.set_num_threads(min(8, torch.get_num_threads()))
    refs = [O.generate_fast(p, spec, n, first_samples=firsts[s], temperature=0.0, keep_logits=True) for s in range(NS)]
    ref_idx = np.stack([r.indices for r in refs])
    ref_lg = np.stack([r.logits for r in refs])
    _, lg = m.generate_fast_batch(n, firsts, temperature=0.0, forced=ref_idx, return_logits=True)
    errs = [rel_err(lg[s], ref_lg[s]) for s in range(NS)]
    assert max(errs) < TOL, f"worst stream {int(np.argmax(errs))}: {max(errs):.3e}"
    idx = m.generate_fast_batch(n, firsts, temperature=0.0)
    for s in range(NS):
        assert_stream_parity(idx[s], ref_idx[s], ref_lg[s])
    assert len({tuple(r) for r in idx.tolist()}) > 1


def test_wavenet_queue_dilate_single_steps(golden):
    """``model.wavenet(x, model.queue_dilate)`` (reference wavenet_model.py:177-184, :262, :277): one evaluation per one-hot
    column on the device-resident queues; the sequence of returned logits equals the teacher-forced generate_fast run."""
    g = golden("net_odd_bias.npz")
    m = build_model(g)
    first = g["first"]
    seq = np.concatenate([first, g["gen_argmax_idx"][:-1]])             # inputs of all evaluations of the golden run
    for q in m.dilated_queues:
        q.reset()
    outs = []
    for i, s in enumerate(seq):
        x = torch.zeros(1, 256, 1, device="cuda")
        x[0, int(s), 0] = 1.0
        y = m.wavenet(x, dilation_func=m.queue_dilate)
        assert y.shape == (1, 256, 1)
        if i >= len(first) - 1:
            outs.append(y[0, :, 0].cpu().numpy())
    assert rel_err(np.stack(outs), g["gen_argmax_logits"]) < TOL
    assert m.dilated_queues[0].in_pos == len(seq) % m.dilated_queues[0].max_length
    # several columns in one call, after a reset: same state as column by column
    for q in m.dilated_queues:
        q.reset()
    x = torch.zeros(1, 256, len(first), device="cuda")
    x[0, torch.from_numpy(first).long().cuda(), torch.arange(len(first)).cuda()] = 1.0
    y = m.wavenet(x, dilation_func=m.queue_dilate)
    assert rel_err(y[0, :, 0].cpu().numpy(), g["gen_argmax_logits"][0]) < TOL
    with pytest.raises(NotImplementedError):
        m.wavenet(torch.rand(1, 256, 1, device="cuda"), dilation_func=m.queue_dilate)


def test_generate_fast_from_cpu_model(golden):
    """The reference's training script samples from a CPU copy of the model (train_script.py:48): that call must work and
    give the same stream as the CUDA model (it runs the same sampler on a CUDA shadow of the weights)."""
    g = golden("net_cfg1.npz")
    m_cpu = build_model(g, device="cpu")
    a = m_cpu.generate_fast(24, first_samples=g["first"], temperature=0.0)
    b = build_model(g).generate_fast(24, first_samples=g["first"], temperature=0.0)
    assert np.array_equal(a, b) and m_cpu.start_conv.weight.device.type == "cpu"
    assert m_cpu.dilated_queues[0].data.shape[0] == m_cpu.residual_channels


def test_slow_generate_equals_generate_fast(golden):
    """generate() (the repaired slow path, reference wavenet_model.py:198-235) and generate_fast() are two evaluations of the
    same network: with a full receptive field of given samples their argmax continuations coincide (up to a near-tie)."""
    g = golden("net_odd_bias.npz")
    m = build_model(g)
    rf = m.receptive_field
    first = g["first"][:rf]
    slow = m.generate(12, first_samples=first, temperature=0.0)
    assert slow.dtype == np.float64 and slow.shape == (rf + 12,) and m.training
    fast = m.generate_fast(12, first_samples=first, temperature=0.0)
    idx_slow = np.rint((O.mu_law_encoding(slow[rf:], 256) + 1) * 128).astype(np.int64)
    idx_fast = np.rint((O.mu_law_encoding(fast, 256) + 1) * 128).astype(np.int64)
    _, lg = m.generate_fast_batch(12, first[None, :], temperature=0.0, forced=idx_fast[None, :], return_logits=True)
    assert_stream_parity(idx_slow, idx_fast, lg[0])
    # fewer given samples than the receptive field: zero (class 0) padding on the left, as the reference intends
    short = m.generate(3, first_samples=first[:4], temperature=0.0)
    assert short.shape == (rf + 3,) and np.array_equal(short[:rf - 4], np.full(rf - 4, audio_of([0])[0]))
