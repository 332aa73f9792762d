"""Host-side logic that needs no GPU: constructor / state_dict compatibility, shape planning, the C ABI surface."""
import ctypes
import hashlib
import os
import re
import struct

import numpy as np
import pytest
import torch

import native
import wavenet_model as wmod
from oracle import wavenet_oracle as O
from helpers import spec_from_golden, params_from_golden, weight_checksum
from conftest import ROOT


def test_library_exports_every_declared_symbol():
    """Every function declared in include/wavenet_b200.h is exported and bound (no compute calls here)."""
    header = open(os.path.join(ROOT, "include", "wavenet_b200.h")).read()
    declared = set(re.findall(r"\b(wn_[a-z0-9_]+)\s*\(", header))
    declared -= {"wn_gen_bind"}                      # mentioned in a comment only
    assert declared == set(native.SIGNATURES), declared ^ set(native.SIGNATURES)
    lib = native.lib()
    for name in declared:
        assert getattr(lib, name) is not None
    assert lib.wn_version() == 2
    assert lib.wn_n1p(256) == 512 and lib.wn_n1p(16) == 128 and lib.wn_n2p(32 + 1024) == 1152
    # argument errors are reported through the return code + message, never by crashing
    assert lib.wn_block_fwd(None, None) == -1
    assert b"null" in lib.wn_last_error_string()


def test_ctor_attributes_and_state_dict_layout():
    m = wmod.WaveNetModel(layers=3, blocks=2, dilation_channels=16, residual_channels=8, skip_channels=12,
                          end_channels=10, classes=256, output_length=5, kernel_size=2, bias=True)
    assert m.receptive_field == O.NetSpec(layers=3, blocks=2, kernel_size=2).receptive_field == 15
    assert m.dilations == [(1, 1), (2, 1), (4, 2), (1, 4), (2, 1), (4, 2)]
    assert [q.max_length for q in m.dilated_queues] == [2, 3, 5, 2, 3, 5]
    assert m.dilated_queues[2].data.shape == (8, 5) and m.dilated_queues[2].num_channels == 8
    sd = m.state_dict()
    assert sd["start_conv.weight"].shape == (8, 256, 1) and sd["filter_convs.4.weight"].shape == (16, 8, 2)
    assert sd["gate_convs.0.bias"].shape == (16,) and sd["residual_convs.5.weight"].shape == (8, 16, 1)
    assert sd["skip_convs.1.weight"].shape == (12, 16, 1) and sd["end_conv_1.weight"].shape == (10, 12, 1)
    assert sd["end_conv_2.weight"].shape == (256, 10, 1) and "end_conv_2.bias" in sd
    assert m.parameter_count() == sum(v.numel() for v in sd.values())
    nb = wmod.WaveNetModel(layers=2, blocks=1)
    assert "start_conv.bias" not in nb.state_dict() and "end_conv_1.bias" in nb.state_dict()
    assert m.cpu() is None and m.dtype == torch.FloatTensor          # reference quirk: cpu() returns None
    assert wmod.WaveNetModel(layers=10, blocks=5, kernel_size=2).receptive_field == 5116
    assert wmod.WaveNetModel(layers=10, blocks=3).receptive_field == 3070


@pytest.mark.parametrize("name", ["odd_bias", "k3", "deep", "cfg1"])
def test_seeded_ctor_reproduces_reference_weights(golden, name):
    g = golden(f"net_{name}.npz")
    spec = spec_from_golden(g)
    torch.manual_seed(0)
    m = wmod.WaveNetModel(**{k[3:]: (bool(g[k]) if k == "kw_bias" else int(g[k])) for k in g.files if k.startswith("kw_")})
    sd = m.state_dict()
    assert weight_checksum(sd) == float(g["w_checksum"])
    ref = params_from_golden(g)
    if ref:
        assert set(ref) == set(sd) and all(torch.equal(sd[k], ref[k]) for k in ref)
    assert m.receptive_field == int(g["receptive_field"]) == spec.receptive_field


@pytest.mark.parametrize("L", [15, 16, 61, 77, 400, 1024, 1025, 16000])
@pytest.mark.parametrize("k", [2, 3])
def test_stack_plan_matches_oracle_lengths(L, k):
    spec = O.NetSpec(layers=4, blocks=2, kernel_size=k)
    dil = [d for d, _ in spec.dilation_schedule()]
    try:
        want = O.valid_lengths(spec, L)
    except Exception:
        want = None
    if want is None or min(want) < 1:
        with pytest.raises(RuntimeError):
            wmod.StackPlan(dil, k, L)
        return
    plan = wmod.StackPlan(dil, k, L)
    assert [L - s for s in plan.out_start] == want
    assert plan.in_start == [0] + plan.out_start[:-1]
    assert plan.t_final == want[-1] and plan.skip_start == L - want[-1]
    assert plan.t_final >= L - spec.receptive_field + 1            # SURVEY.md 3.1: extra, padding-contaminated columns


def test_cfg3_plan_numbers():
    dil = [2 ** i for i in range(10)] * 5
    plan = wmod.StackPlan(dil, 2, 16000)
    assert plan.t_final == 13312                                  # SURVEY.md section 3.1
    assert 16000 - 5116 + 1 == 10885


def test_snapshot_state_loads(golden):
    gs = golden("snapshot_chaconne_state.npz")
    p = params_from_golden(gs)
    m = wmod.WaveNetModel(layers=int(gs["layers"]), blocks=int(gs["blocks"]), dilation_channels=32,
                          residual_channels=32, skip_channels=1024, end_channels=512, classes=256,
                          output_length=int(gs["output_length"]), kernel_size=2, bias=True)
    m.load_state_dict(p, strict=True)
    assert m.parameter_count() == 1834592 and m.receptive_field == 3070


def test_reference_pickle_unpickles_into_this_class(golden, tmp_path):
    """The reference snapshots are whole-object pickles of wavenet_model.WaveNetModel; with this package on the
    path they restore into THIS class (wavenet_model.py:330-346 load_latest_model_from / load_to_cpu).  The chaconne
    snapshot is reassembled from its stored pickle header, each storage filled from the stored parameters or with zeros
    (tests/golden/make_golden_pickle.py)."""
    gp = golden("snapshot_chaconne_pickle.npz")
    p = params_from_golden(golden("snapshot_chaconne_state.npz"))
    head = gp["head"].tobytes()
    assert hashlib.sha256(head).hexdigest() == str(gp["head_sha256"])
    path = tmp_path / "chaconne_model"
    with open(path, "wb") as f:
        f.write(head)
        for src, n in zip(gp["sources"], gp["counts"]):
            f.write(struct.pack("<q", int(n)))
            f.write(p[str(src)].numpy().astype("<f4").tobytes() if src else bytes(4 * int(n)))
    m = wmod.load_to_cpu(str(path))
    assert type(m) is wmod.WaveNetModel and m.receptive_field == 3070 and m.dtype == torch.FloatTensor
    assert type(m.dilated_queues[0]).__module__ == "wavenet_modules"
    assert m._runtime() is m._runtime()
    assert set(m.state_dict()) == set(p) and all(torch.equal(v, p[k]) for k, v in m.state_dict().items())


def test_no_cpu_fallback(monkeypatch):
    m = wmod.WaveNetModel(layers=2, blocks=1, dilation_channels=4, residual_channels=4, skip_channels=4, end_channels=4)
    with torch.no_grad(), pytest.raises(RuntimeError, match="CUDA"):
        m(torch.zeros(1, 256, 16))
    # generate_fast of a CPU-resident model samples on a CUDA copy when there is a device (test_gpu_generate covers
    # that); without one it must raise rather than sample on the CPU
    monkeypatch.setattr(torch.cuda, "is_available", lambda: False)
    with pytest.raises(RuntimeError, match="CUDA"):
        m.generate_fast(4)
    with pytest.raises(RuntimeError, match="CUDA"):
        m.generate(4)


def test_shape_predicates_and_workspace_sizes_are_host_side():
    """The capability predicates and the workspace query need no device; argument errors are reported before any launch."""
    import ctypes
    import native
    lib = native.lib()
    assert lib.wn_tc_supported(256, 256, 256, 2) and lib.wn_tc_supported(512, 512, 512, 2)
    assert not lib.wn_tc_supported(32, 32, 256, 2) and not lib.wn_tc_supported(256, 64, 256, 2)
    assert lib.wn_tc_bwd_supported(256, 256, 256, 2) and not lib.wn_tc_bwd_supported(256, 128, 256, 2)
    assert lib.wn_tc_wgrad_supported(512, 256) and lib.wn_tc_wgrad_supported(128, 256)
    assert not lib.wn_tc_wgrad_supported(512, 512) and not lib.wn_tc_wgrad_supported(100, 256)
    # split-frames workspace: ceil(296 / number of 128x128 output tiles) partials of N x C floats
    assert lib.wn_wgrad_workspace_bytes(512, 256) == 37 * 512 * 256 * 4
    assert lib.wn_wgrad_workspace_bytes(256, 256) == 74 * 256 * 256 * 4
    assert lib.wn_wgrad_workspace_bytes(17, 5) == 296 * 17 * 5 * 4
    assert lib.wn_wgrad_workspace_bytes(0, 5) == 0
    a = native.WgradArgs()
    a.N, a.C, a.B, a.rows = 0, 4, 1, 8
    assert lib.wn_wgrad(ctypes.byref(a), None) < 0 and b"bad sizes" in lib.wn_last_error_string()
    a.N, a.C = 512, 128
    assert lib.wn_tc_wgrad(ctypes.byref(a), None) < 0 and b"C == 256" in lib.wn_last_error_string()
    assert lib.wn_tc_block_bwd_data_prec(None, None, None, 0, None) < 0
    assert lib.wn_tc_convert_weights_bf16(None, None, 0, None) < 0


def test_sampler_workspace_and_argument_errors_are_host_side():
    """wn_gen_workspace_bytes needs no device: a 256-wide k = 2 net reserves room for the tensor-core sampler's pre-split
    weight images (16 blocks x (3 x 32 KB per layer + 2 x 16 KB for the head)), other shapes do not; null handles and
    pointers are argument errors."""
    import ctypes
    import native
    lib = native.lib()

    def scratch_bytes(width, n_layers, n_streams):
        dil = (ctypes.c_int * n_layers)(*[2 ** (i % 10) for i in range(n_layers)])
        shape = native.GenShape(n_layers, 2, width, width, width, width, 256, n_streams, dil)
        rb, sb = ctypes.c_size_t(), ctypes.c_size_t()
        assert lib.wn_gen_workspace_bytes(ctypes.byref(shape), ctypes.byref(rb), ctypes.byref(sb)) == 0
        assert rb.value == 8 * sum(d + 1 for d in dil) * n_streams * width        # {value, tag} pairs, ring_len = d + 1
        return sb.value

    images = 16 * (50 * 3 * 32768 + 2 * 16384)
    wide, narrow = scratch_bytes(256, 50, 1), scratch_bytes(128, 50, 1)
    assert wide - images >= 0 and wide - images < 4 * narrow and narrow < images
    assert scratch_bytes(256, 50, 64) > wide
    assert lib.wn_gen_kernel_id(None) == 0
    assert lib.wn_gen_weights_changed(None) < 0 and b"null handle" in lib.wn_last_error_string()
    assert lib.wn_gen_set_mode(None, 6) < 0
    assert lib.wn_scale_by(None, 4, None, None) < 0 and b"bad arguments" in lib.wn_last_error_string()


def test_dataset_matches_reference_items(golden):
    """WavenetDataset (reference audio_data.py:12-131): same lengths, same item -> sample-window map (incl. windows that
    cross array boundaries and the train / test split), and the index mode (one_hot=False, SURVEY.md section 8 row f2)
    returns exactly the indices whose one-hot matrix the reference builds."""
    import os
    from conftest import GOLDEN
    import audio_data
    g = golden("dataset_items.npz")
    tiny = os.path.join(GOLDEN, "tiny_dataset.npz")
    keys = sorted(k[:-4] for k in g.files if k.endswith("_cfg"))
    assert len(keys) == 8
    for key in keys:
        item_length, target_length, stride, train, n = [int(v) for v in g[key + "_cfg"]]
        for one_hot in (True, False):
            ds = audio_data.WavenetDataset(dataset_file=tiny, item_length=item_length, target_length=target_length,
                                           test_stride=stride, train=bool(train), one_hot=one_hot)
            assert len(ds) == n, key
            for j, i in enumerate(g[key + "_picks"]):
                x, t = ds[int(i)]
                assert np.array_equal(t.numpy(), g[key + "_t"][j])
                if one_hot:
                    assert x.shape == (256, item_length) and x.dtype == torch.float32 and float(x.sum()) == item_length
                    assert np.array_equal(x.argmax(0).numpy(), g[key + "_x"][j])
                else:
                    assert x.dtype == torch.uint8 and np.array_equal(x.numpy(), g[key + "_x"][j])


def test_write_wav_roundtrip(tmp_path):
    import wave
    import audio_data
    audio = np.sin(np.linspace(0, 40, 1600)) * 0.5
    path = str(tmp_path / "clip.wav")
    audio_data.write_wav(path, audio, sr=16000)
    with wave.open(path, "rb") as f:
        assert (f.getnchannels(), f.getsampwidth(), f.getframerate(), f.getnframes()) == (1, 2, 16000, 1600)
        pcm = np.frombuffer(f.readframes(1600), dtype="<i2")
    assert np.abs(pcm / 32767.0 - audio).max() < 1e-4
