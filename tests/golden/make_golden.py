#!/usr/bin/env python
"""Generate the golden fixtures in this directory by running the UNMODIFIED reference.

    python tests/golden/make_golden.py <checkout of the original pytorch-wavenet>

The reference sources are imported from where they lie (nothing is copied); five compatibility shims make
the 2017 / torch-0.3 code run on torch 2.x (SURVEY.md section 8c):
  1. a stub ``librosa`` module (audio_data.py:8 imports it at top level),
  2. ``wavenet_modules.constant_pad_1d`` -> ``F.pad`` equivalent (legacy autograd.Function, :80-127),
  3. ``DilatedQueue.enqueue`` reshapes its (R,1) argument to (R,) (torch 0.3 broadcast, wavenet_model.py:179),
  4. ``torch.max(x, 0)`` inside module ``wavenet_model`` returns a (1,1)-shaped index (no 0-dim tensors in 0.3;
     wavenet_model.py:292 does ``[1][0]``),
  5. the snapshot is loaded with ``weights_only=False`` and moved with ``.cpu()`` (wavenet_model.py:343-346).
Everything written is a plain ``.npz`` of arrays, each under 1 MB.  The seeded nets' weights are rebuilt from the seed
by the tests, so only the small nets ship them; ``deep`` ships a SHA-256 per tensor instead.  The trained snapshot
(1.83 M parameters) is re-saved with every tensor but the two head biases quantized to an 8-entry float32 codebook
(``quantize``), and the reference runs on those weights, so its outputs here are exact for the stored weights.
"""
import hashlib
import os
import sys
import types

import numpy as np
import torch
import torch.nn.functional as F

HERE = os.path.dirname(os.path.abspath(__file__))


def import_reference(ref):
    sys.modules.setdefault("librosa", types.ModuleType("librosa"))                    # shim 1
    sys.path.insert(0, ref)
    import wavenet_modules as wm                                                      # noqa: E402
    import wavenet_model as wmod                                                      # noqa: E402

    def pad1d(input, target_size, dimension=0, value=0, pad_start=False):            # shim 2
        n = target_size - input.size(dimension)
        assert n >= 0, "target size has to be greater than input size"
        pads = [0, 0] * input.dim()
        slot = 2 * (input.dim() - 1 - dimension)
        pads[slot + (0 if pad_start else 1)] = n
        return F.pad(input, pads, value=value)

    wm.constant_pad_1d = pad1d
    wmod.constant_pad_1d = pad1d

    _enq = wm.DilatedQueue.enqueue

    def enqueue(self, input):                                                         # shim 3
        return _enq(self, input.reshape(-1))

    wm.DilatedQueue.enqueue = enqueue

    class TorchProxy:                                                                 # shim 4
        def __getattr__(self, name):
            return getattr(torch, name)

        @staticmethod
        def max(x, *a, **k):
            r = torch.max(x, *a, **k)
            if a and isinstance(r, tuple) and r[1].dim() == 0:
                return r[0].view(1), r[1].view(1, 1)
            return r

    wmod.torch = TorchProxy()
    return wm, wmod


def quantize(w, levels=8, iters=25):
    """(codebook, codes): 1-D k-means of the tensor's values, started at evenly spaced quantiles; codebook[codes] is
    the float32 tensor the fixture stands for."""
    x = w.detach().cpu().numpy().astype(np.float64).ravel()
    book = np.quantile(x, (np.arange(levels) + 0.5) / levels)
    for _ in range(iters):
        codes = np.abs(x[:, None] - book[None, :]).argmin(1)
        book = np.array([x[codes == j].mean() if np.any(codes == j) else book[j] for j in range(levels)])
    book = book.astype(np.float32)
    codes = np.abs(x[:, None] - book.astype(np.float64)[None, :]).argmin(1).astype(np.uint8)
    return book, codes.reshape(tuple(w.shape))


def state_arrays(model):
    return {k: v.detach().cpu().numpy() for k, v in model.state_dict().items()}


def indices(b, l, seed=1234, classes=256):
    return torch.randint(0, classes, (b, l), generator=torch.Generator().manual_seed(seed))


def one_hot(idx, classes=256):
    b, l = idx.shape
    return torch.zeros(b, classes, l).scatter_(1, idx.view(b, 1, l), 1.0)


def record_generate(model, num_samples, first_samples, temperature, regularize=0.0, seed=None):
    """Run the reference generate_fast, recording every network output (one per wavenet() call)."""
    outs = []
    orig = model.wavenet

    def spy(input, dilation_func):
        y = orig(input, dilation_func)
        outs.append(y.detach().clone().view(-1).numpy())
        return y

    model.wavenet = spy
    if seed is not None:
        np.random.seed(seed)
    fs = None if first_samples is None else torch.as_tensor(np.asarray(first_samples), dtype=torch.long)
    with torch.no_grad():
        audio = model.generate_fast(num_samples, first_samples=fs, temperature=temperature,
                                    regularize=regularize)
    del model.wavenet                                                                 # restore class method
    logits = np.stack(outs[-num_samples:]).astype(np.float32)                         # raw net outputs
    return np.asarray(audio, dtype=np.float64), logits


def audio_to_indices(audio, classes=256):
    """Invert o=(x/classes)*2-1 followed by mu_law_expansion (exact to rounding)."""
    mu = classes
    o = np.sign(audio) * np.log(1 + mu * np.abs(audio)) / np.log(mu + 1)
    return np.rint((o + 1.0) / 2.0 * classes).astype(np.int64)


def main():
    if len(sys.argv) != 2:
        raise SystemExit(__doc__)
    ref = sys.argv[1]
    wm, wmod = import_reference(ref)
    torch.set_num_threads(8)
    out = {}

    # ---------------- module-level known answers (reference tests/test_modules.py, tests/test_tensor_queue.py)
    x13 = torch.linspace(0, 12, steps=13).view(1, 1, 13)
    d2 = wm.dilate(x13, 2)
    d4 = wm.dilate(d2, 4, init_dilation=2)
    d1 = wm.dilate(d4, 1, init_dilation=4)
    xm = torch.linspace(0, 35, steps=36).view(2, 3, 6)
    np.savez(os.path.join(HERE, "modules.npz"),
             x13=x13.numpy(), d2=d2.numpy(), d4=d4.numpy(), d1=d1.numpy(),
             xm=xm.numpy(), xm2=wm.dilate(xm, 2).numpy(), xm4=wm.dilate(xm, 4).numpy(),
             pad_end=wm.constant_pad_1d(torch.arange(6.).view(2, 3), 5, dimension=1, value=7.0).numpy(),
             pad_start=wm.constant_pad_1d(torch.arange(6.).view(2, 3), 5, dimension=1, pad_start=True).numpy())

    q = wm.DilatedQueue(max_length=12, num_channels=2)
    trace = []
    e = torch.zeros(2)
    for i in range(30):
        e = e + 1
        q.enqueue(e * torch.tensor([1.0, -1.0]))
        trace.append(q.dequeue(num_deq=3, dilation=4).clone().numpy())
    np.savez(os.path.join(HERE, "queue.npz"), combined=np.stack(trace), final=q.data.numpy(),
             in_pos=q.in_pos, out_pos=q.out_pos)

    # ---------------- model-level: seeded random-init nets
    cases = {
        # name: (ctor kwargs, B, L)
        "cfg1": (dict(layers=3, blocks=2, dilation_channels=32, residual_channels=32, skip_channels=32,
                      end_channels=32, classes=256, output_length=32, kernel_size=2, bias=False), 1, 1024),
        "odd_bias": (dict(layers=3, blocks=2, dilation_channels=16, residual_channels=8, skip_channels=12,
                          end_channels=10, classes=256, output_length=5, kernel_size=2, bias=True), 3, 77),
        "k3": (dict(layers=3, blocks=2, dilation_channels=8, residual_channels=8, skip_channels=16,
                    end_channels=8, classes=256, output_length=4, kernel_size=3, bias=True), 2, 61),
        "deep": (dict(layers=6, blocks=2, dilation_channels=64, residual_channels=64, skip_channels=64,
                      end_channels=64, classes=256, output_length=100, kernel_size=2, bias=False), 2, 400),
    }
    for name, (kw, B, L) in cases.items():
        torch.manual_seed(0)
        m = wmod.WaveNetModel(**kw)
        idx = indices(B, L)
        with torch.no_grad():
            full = m.wavenet(one_hot(idx), dilation_func=m.wavenet_dilate)            # all T_final columns
            fwd = m(one_hot(idx))
        first = idx[0, :min(L, m.receptive_field + 3)].numpy()
        a0, lg0 = record_generate(m, 24, first, temperature=0.0)
        a1, lg1 = record_generate(m, 24, first, temperature=0.8, regularize=1e-4, seed=7)
        np.random.seed(7)
        u = np.random.random_sample(24)                       # the uniforms np.random.choice consumed
        w = state_arrays(m)
        arrs = dict(idx=idx.numpy(), full=full.numpy(), fwd=fwd.numpy(),
                    receptive_field=m.receptive_field, first=first,
                    gen_argmax_audio=a0, gen_argmax_idx=audio_to_indices(a0), gen_argmax_logits=lg0,
                    gen_sample_audio=a1, gen_sample_idx=audio_to_indices(a1), gen_sample_logits=lg1,
                    gen_sample_uniforms=u,
                    w_checksum=np.float64(sum(float(np.abs(v).astype(np.float64).sum()) for v in w.values())))
        arrs.update({"kw_" + k: v for k, v in kw.items()})
        if name == "deep":                                    # rebuilt from the seed by the tests, checked per tensor
            arrs.update({"d:" + k: np.array(hashlib.sha256(v.astype("<f4").tobytes()).hexdigest()) for k, v in w.items()})
        elif name != "cfg1":
            arrs.update({"w:" + k: v for k, v in w.items()})  # small nets: ship the weights too
        np.savez_compressed(os.path.join(HERE, f"net_{name}.npz"), **arrs)
        out[name] = (fwd.shape, float(fwd.abs().max()))

    # ---------------- cfg 2 shape (10x5, 256 ch): seeded init is reproduced by ctor order; ship outputs only
    kw = dict(layers=10, blocks=5, dilation_channels=256, residual_channels=256, skip_channels=256,
              end_channels=256, classes=256, output_length=16, kernel_size=2, bias=False)
    torch.manual_seed(0)
    m = wmod.WaveNetModel(**kw)
    w = state_arrays(m)
    a0, lg0 = record_generate(m, 48, None, temperature=0.0)
    a1, lg1 = record_generate(m, 48, [3, 200, 128, 77], temperature=1.0, seed=0)
    np.random.seed(0)
    u = np.random.random_sample(48)
    idx = indices(1, m.receptive_field + 15, seed=99)
    with torch.no_grad():
        fwd = m(one_hot(idx))
    np.savez_compressed(os.path.join(HERE, "net_cfg2.npz"),
                        gen_argmax_audio=a0, gen_argmax_idx=audio_to_indices(a0), gen_argmax_logits=lg0,
                        gen_sample_audio=a1, gen_sample_idx=audio_to_indices(a1), gen_sample_logits=lg1,
                        gen_sample_uniforms=u, gen_sample_first=np.array([3, 200, 128, 77]),
                        idx=idx.numpy(), fwd=fwd.numpy(), receptive_field=m.receptive_field,
                        w_checksum=np.float64(sum(float(np.abs(v).astype(np.float64).sum()) for v in w.values())),
                        w_probe=w["filter_convs.17.weight"][:4, :4, :],
                        **{"kw_" + k: v for k, v in kw.items()})
    out["cfg2"] = (fwd.shape, float(np.abs(fwd.numpy()).max()))

    # ---------------- the shipped trained snapshot on real mu-law audio
    snap = os.path.join(ref, "snapshots", "chaconne_model_2017-12-28_16-44-12")
    m = torch.load(snap, map_location="cpu", weights_only=False)                      # shim 5
    m.cpu()
    packed = {}
    with torch.no_grad():
        for k, v in m.state_dict().items():
            if k in ("end_conv_1.bias", "end_conv_2.bias"):      # exact, so that no two classes' logits tie exactly
                packed["w:" + k] = v.numpy().copy()
                continue
            book, codes = quantize(v)
            v.copy_(torch.from_numpy(book[codes.astype(np.int64)]))
            packed["l:" + k], packed["c:" + k] = book, codes
    np.savez_compressed(os.path.join(HERE, "snapshot_chaconne_state.npz"), layers=m.layers, blocks=m.blocks,
                        kernel_size=m.kernel_size, classes=m.classes, output_length=m.output_length,
                        receptive_field=m.receptive_field, **packed)
    data = np.load(os.path.join(ref, "train_samples", "bach_chaconne", "dataset.npz"))["arr_0"]
    rf = m.receptive_field
    off = 960000
    clip = data[off:off + rf + 260].astype(np.int64)          # rf given samples + 260 for teacher forcing
    first = clip[:rf]
    a0, lg0 = record_generate(m, 200, first, temperature=0.0)
    m.output_length = 64
    with torch.no_grad():
        x = one_hot(torch.from_numpy(clip[None, :rf + 63]))
        fwd = m(x)                                            # (64, 256): teacher-forced logits
    np.savez_compressed(os.path.join(HERE, "snapshot_chaconne_io.npz"), clip=clip.astype(np.uint8),
                        offset=off, gen_argmax_audio=a0, gen_argmax_idx=audio_to_indices(a0),
                        gen_argmax_logits=lg0, fwd64=fwd.numpy())
    out["snapshot"] = (fwd.shape, audio_to_indices(a0)[:8].tolist())
    for k, v in out.items():
        print(k, v)


if __name__ == "__main__":
    main()
