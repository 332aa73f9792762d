"""Pin the CPU oracle against the reference: known answers of the reference's own tests and the outputs of
the unmodified reference run by tests/golden/make_golden.py (same torch => bit-for-bit)."""
import numpy as np
import pytest
import torch

from oracle import wavenet_oracle as O
from helpers import spec_from_golden, params_from_golden, weight_checksum, rel_err

NETS_WITH_WEIGHTS = ["odd_bias", "k3", "deep"]


# ---------------------------------------------------------------- reference tests/test_modules.py:8-29
def test_fold_known_answers():
    x = torch.linspace(0, 12, steps=13).view(1, 1, 13)
    d = O.fold_time(x, 1)
    assert d.shape == (1, 1, 13) and d[0, 0, 4] == 4
    d = O.fold_time(x, 2)
    assert d.shape == (2, 1, 7) and d[1, 0, 2] == 4
    d = O.fold_time(d, 4, init_dilation=2)
    assert d.shape == (4, 1, 4) and d[3, 0, 1] == 4
    d = O.fold_time(d, 1, init_dilation=4)
    assert d.shape == (1, 1, 16) and d[0, 0, 7] == 4


def test_fold_matches_reference_arrays(golden):
    g = golden("modules.npz")
    x = torch.from_numpy(g["x13"])
    d2 = O.fold_time(x, 2)
    d4 = O.fold_time(d2, 4, init_dilation=2)
    d1 = O.fold_time(d4, 1, init_dilation=4)
    for got, key in ((d2, "d2"), (d4, "d4"), (d1, "d1")):
        assert np.array_equal(got.numpy(), g[key])
    xm = torch.from_numpy(g["xm"])
    assert np.array_equal(O.fold_time(xm, 2).numpy(), g["xm2"])     # tests/test_modules.py:31-36 shapes
    assert np.array_equal(O.fold_time(xm, 4).numpy(), g["xm4"])
    assert np.array_equal(O.pad_to(torch.arange(6.).view(2, 3), 5, dim=1, value=7.0).numpy(), g["pad_end"])
    assert np.array_equal(O.pad_to(torch.arange(6.).view(2, 3), 5, dim=1, at_start=True).numpy(), g["pad_start"])
    with pytest.raises(AssertionError):
        O.pad_to(torch.zeros(4), 3)


# ---------------------------------------------------------------- reference tests/test_tensor_queue.py:13-50
def test_queue_enqueue_wraps():
    q = O.RingQueue(8, 3)
    e = torch.zeros(3)
    for _ in range(11):
        e = e + 1
        q.enqueue(e)
    row = q.data[0]
    assert row[0] == 9 and row[2] == 11 and row[7] == 8


def test_queue_dequeue_strided():
    q = O.RingQueue(8, 1)
    e = torch.zeros(1)
    for _ in range(11):
        e = e + 1
        q.enqueue(e)
    for _ in range(9):
        d = q.dequeue(num_deq=3, dilation=2)
    assert d[0].tolist() == [5, 7, 9]


def test_queue_combined(golden):
    q = O.RingQueue(12, 1)
    e = torch.zeros(1)
    for i in range(30):
        e = e + 1
        q.enqueue(e)
        d = q.dequeue(num_deq=3, dilation=4)
        assert d[0][0] == max(i - 7, 0)
    g = golden("queue.npz")
    q = O.RingQueue(12, 2)
    e = torch.zeros(2)
    for i in range(30):
        e = e + 1
        q.enqueue(e * torch.tensor([1.0, -1.0]))
        assert np.array_equal(q.dequeue(3, 4).numpy(), g["combined"][i])
    assert np.array_equal(q.data.numpy(), g["final"])
    assert q.in_pos == g["in_pos"] and q.out_pos == g["out_pos"]


# ---------------------------------------------------------------- model level: bit-for-bit with the reference
@pytest.mark.parametrize("name", NETS_WITH_WEIGHTS)
def test_forward_bitwise_vs_reference(golden, name):
    g = golden(f"net_{name}.npz")
    spec, p = spec_from_golden(g), params_from_golden(g)
    assert spec.receptive_field == g["receptive_field"]
    x = O.one_hot(torch.from_numpy(g["idx"]), spec.classes)
    with torch.no_grad():
        full = O.stack_folded(p, spec, x, lambda h, d, i0, i: O.fold_time(h, d, i0))
        fwd = O.forward(p, spec, x)
        direct = O.stack_direct(p, spec, x)
    assert np.array_equal(full.numpy(), g["full"])
    assert np.array_equal(fwd.numpy(), g["fwd"])
    assert full.shape[2] == O.valid_lengths(spec, x.shape[2])[-1]
    assert rel_err(direct.numpy(), g["full"]) < 2e-6        # the two statements agree at ALL columns


def test_seeded_init_reproduces_reference_weights(golden):
    g = golden("net_cfg1.npz")
    spec = spec_from_golden(g)
    p = O.init_params(spec, seed=0)
    assert weight_checksum(p) == pytest.approx(float(g["w_checksum"]), rel=0, abs=0)
    x = O.one_hot(torch.from_numpy(g["idx"]), spec.classes)
    with torch.no_grad():
        assert np.array_equal(O.forward(p, spec, x).numpy(), g["fwd"])
    for name in NETS_WITH_WEIGHTS:                          # ctor order == state_dict of the reference
        gg = golden(f"net_{name}.npz")
        pp, ref = O.init_params(spec_from_golden(gg), 0), params_from_golden(gg)
        assert set(pp) == set(ref)
        assert all(torch.equal(pp[k], ref[k]) for k in ref)


@pytest.mark.parametrize("name", NETS_WITH_WEIGHTS)
def test_generate_bitwise_vs_reference(golden, name):
    g = golden(f"net_{name}.npz")
    spec, p = spec_from_golden(g), params_from_golden(g)
    tr = O.generate_fast(p, spec, 24, first_samples=g["first"], temperature=0.0, keep_logits=True)
    assert np.array_equal(tr.indices, g["gen_argmax_idx"])
    assert np.array_equal(tr.audio, g["gen_argmax_audio"])
    assert np.array_equal(tr.logits, g["gen_argmax_logits"])
    # sampled path, numpy global RNG exactly as the reference uses it
    np.random.seed(7)
    tr = O.generate_fast(p, spec, 24, first_samples=g["first"], temperature=0.8, regularize=1e-4)
    assert np.array_equal(tr.indices, g["gen_sample_idx"])
    assert np.array_equal(tr.audio, g["gen_sample_audio"])
    # ... and with the uniforms handed in (one per draw): same stream
    tr = O.generate_fast(p, spec, 24, first_samples=g["first"], temperature=0.8, regularize=1e-4,
                         uniforms=g["gen_sample_uniforms"])
    assert np.array_equal(tr.indices, g["gen_sample_idx"])


def test_snapshot_stream_and_consistency(golden):
    """Trained snapshot on real audio: argmax stream, and forward() == generate_fast() teacher-forced."""
    gs, gio = golden("snapshot_chaconne_state.npz"), golden("snapshot_chaconne_io.npz")
    p = params_from_golden(gs)
    spec = O.spec_from_params(p, int(gs["layers"]), int(gs["blocks"]), output_length=64)
    rf = int(gs["receptive_field"])
    assert spec.receptive_field == rf == 3070
    clip = gio["clip"].astype(np.int64)
    tr = O.generate_fast(p, spec, 40, first_samples=clip[:rf], temperature=0.0, keep_logits=True)
    assert np.array_equal(tr.indices, gio["gen_argmax_idx"][:40])
    assert np.array_equal(tr.logits, gio["gen_argmax_logits"][:40])
    assert tr.indices[:8].tolist() == [177, 177, 177, 174, 174, 177, 181, 188]      # the reference, stored weights
    with torch.no_grad():
        fwd = O.forward(p, spec, O.one_hot(torch.from_numpy(clip[None, :rf + 63]), 256))
    assert np.array_equal(fwd.numpy(), gio["fwd64"])
    # teacher-forced sampling logits equal the training-path logits column for column
    tf = O.generate_fast(p, spec, 12, first_samples=clip[:rf], temperature=0.0, keep_logits=True,
                         forced=clip[rf:rf + 12])
    assert rel_err(tf.logits, gio["fwd64"][:12]) < 1e-5


def test_cfg2_shape_spot_check(golden):
    """cfg 2 net (10x5, 256 ch): seeded init reproduces the reference's weights; first sampling steps match."""
    g = golden("net_cfg2.npz")
    spec = spec_from_golden(g)
    assert spec.receptive_field == g["receptive_field"] == 5116
    p = O.init_params(spec, seed=0)
    assert np.array_equal(p["filter_convs.17.weight"][:4, :4, :].numpy(), g["w_probe"])
    assert weight_checksum(p) == float(g["w_checksum"])
    tr = O.generate_fast(p, spec, 6, temperature=0.0, keep_logits=True)
    assert np.array_equal(tr.indices, g["gen_argmax_idx"][:6])
    assert np.array_equal(tr.logits, g["gen_argmax_logits"][:6])


def test_mu_law_roundtrip():
    x = np.linspace(-1, 1, 41)
    assert np.allclose(O.mu_law_expansion(O.mu_law_encoding(x, 256), 256), x, atol=1e-12)


def test_relu_tie_separation_helper_moves_only_two_biases():
    """helpers.separate_head_relu_ties (used by the GPU backward tests): afterwards no head ReLU input of the case is within
    the margin of zero, and nothing but the last skip bias and the end_conv_1 bias has changed."""
    from helpers import separate_head_relu_ties
    kw = dict(layers=2, blocks=2, dilation_channels=16, residual_channels=16, skip_channels=24, end_channels=20,
              classes=256, output_length=40, kernel_size=2, bias=True)
    spec = O.NetSpec(**kw)
    p = O.init_params(spec, seed=3)
    idx = torch.randint(0, 256, (2, 120), generator=torch.Generator().manual_seed(1))
    x = O.one_hot(idx, 256)
    # plant exact ties: a zero skip channel bias pattern would be luck, so force one pre-activation to ~0 via the bias
    taps = {}
    O.stack_direct(p, spec, x, taps)
    p["end_conv_1.bias"][3] -= taps["pre1"][0, 3, -1]
    taps1 = {}
    O.stack_direct(p, spec, x, taps1)
    assert float(taps1["pre1"][..., -40:].abs().min()) < 1e-6          # the planted tie is there
    sep = separate_head_relu_ties(p, spec, x, 40, margin=2e-5)
    changed = {k for k in p if not torch.equal(p[k], sep[k])}
    assert changed and changed <= {"skip_convs.3.bias", "end_conv_1.bias"}
    taps2 = {}
    O.stack_direct({k: v.double() for k, v in sep.items()}, spec, x.double(), taps2)
    assert float(taps2["skip"][..., -40:].abs().min()) >= 1.9e-5
    assert float(taps2["pre1"][..., -40:].abs().min()) >= 1.9e-5
