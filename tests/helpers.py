"""Helpers shared by the parity tests (oracle side only; nothing here is product code)."""
import hashlib

import numpy as np
import torch

from oracle import wavenet_oracle as O


def spec_from_golden(g, output_length=None):
    kw = {k[3:]: g[k].item() for k in g.files if k.startswith("kw_")}
    kw["bias"] = bool(kw["bias"])
    if output_length is not None:
        kw["output_length"] = output_length
    return O.NetSpec(**kw)


def params_from_golden(g):
    """The weights a fixture stands for ({} if none): stored ("w:"), stored as a float32 codebook and codes ("l:", "c:";
    the quantized snapshot), or rebuilt from seed 0 and checked against the reference's per-tensor SHA-256 ("d:")."""
    digests = {k[2:]: str(g[k]) for k in g.files if k.startswith("d:")}
    if digests:
        p = O.init_params(spec_from_golden(g), seed=0)
        assert set(p) == set(digests)
        for k, v in p.items():
            assert hashlib.sha256(v.numpy().astype("<f4").tobytes()).hexdigest() == digests[k], k
        return p
    p = {k[2:]: torch.from_numpy(g[k]) for k in g.files if k.startswith("w:")}
    p.update({k[2:]: torch.from_numpy(g["l:" + k[2:]][g[k].astype(np.int64)]) for k in g.files if k.startswith("c:")})
    return p


def weight_checksum(params):
    return sum(float(np.abs(v.detach().cpu().numpy()).astype(np.float64).sum()) for v in params.values())


def rel_err(a, b):
    """max |a-b| / max |b|: the relative measure all fp32 parity gates use (tolerance 1e-4)."""
    a = np.asarray(a, dtype=np.float64)
    b = np.asarray(b, dtype=np.float64)
    return float(np.abs(a - b).max() / max(np.abs(b).max(), 1e-30))


def classify_stream(got_idx, ref_idx, ref_margins, tol=1e-4):
    """Compare two argmax streams.  Returns (n_equal_prefix, first_mismatch_is_near_tie)."""
    got_idx, ref_idx = np.asarray(got_idx), np.asarray(ref_idx)
    neq = np.nonzero(got_idx != ref_idx)[0]
    if len(neq) == 0:
        return len(ref_idx), True
    i = int(neq[0])
    return i, bool(ref_margins[i] < tol)


def separate_head_relu_ties(params, spec, x, out_len, margin=2e-5, step=None):
    """Gradients are discontinuous where a head ReLU input is exactly zero: an fp32-class difference (3xTF32 tensor
    cores vs FFMA, or just another summation order) that flips the sign of a pre-activation of size 1e-7 switches one
    mask element and moves a weight gradient by percent.  The analogue of the argmax near-tie rule for the backward
    tests: nudge the last skip bias and the end_conv_1 bias (per channel, in float64 on the oracle) until no head ReLU
    input of this test case lies within `margin` of zero.  Returns a new fp32 parameter dict."""
    step = 5 * margin if step is None else step
    p = {k: v.detach().clone().double() for k, v in params.items()}
    last = spec.layers * spec.blocks - 1
    taps = {}
    O.stack_direct(p, spec, x.double(), taps)
    sk = taps["skip"][..., -out_len:].clone()                           # (B, S, out_len)
    for name, pre_of in ((f"skip_convs.{last}.bias", lambda: sk),
                         ("end_conv_1.bias", lambda: F_conv1d(torch.relu(sk), p["end_conv_1.weight"], p["end_conv_1.bias"]))):
        if name not in p:              # bias=False nets have no skip bias to nudge: see tie_free_indices
            continue
        pre = pre_of()
        for c in range(pre.shape[1]):
            v, off = pre[:, c, :], 0.0
            while float((v + off).abs().min()) < margin:
                off += step
            p[name][c] += off
            pre[:, c, :] += off
    return {k: v.float() for k, v in p.items()}


def tie_free_indices(params, spec, B, L, out_len, margin=5e-6, seed0=2, tries=30):
    """(B, L) class indices for which no relu(skip) input of the oracle lies within `margin` of zero: the alternative to a
    bias nudge for nets without skip biases.  Feasible only for small B * out_len (the chance of a miss grows with it)."""
    p = {k: v.detach().double() for k, v in params.items()}
    for s in range(seed0, seed0 + tries):
        idx = torch.randint(0, spec.classes, (B, L), generator=torch.Generator().manual_seed(s))
        taps = {}
        O.stack_direct(p, spec, O.one_hot(idx, spec.classes).double(), taps)
        if float(taps["skip"][..., -out_len:].abs().min()) > margin:
            return idx
    raise RuntimeError("no tie-free input found")


def F_conv1d(x, w, b):
    return torch.nn.functional.conv1d(x, w, b)


# ---------------------------------------------------------------- product-side helpers (GPU tests)
def build_model(g, device="cuda", output_length=None):
    """WaveNetModel (product) with the constructor args / weights stored in a golden file."""
    import wavenet_model as wmod
    kw = {k[3:]: (bool(g[k]) if k == "kw_bias" else int(g[k])) for k in g.files if k.startswith("kw_")}
    if output_length is not None:
        kw["output_length"] = output_length
    torch.manual_seed(0)
    m = wmod.WaveNetModel(**kw)
    ref = params_from_golden(g)
    if ref:
        m.load_state_dict(ref, strict=True)
    else:
        assert weight_checksum(m.state_dict()) == float(g["w_checksum"])
    return m.to(device)


def snapshot_model(gs, device="cuda", output_length=64):
    import wavenet_model as wmod
    m = wmod.WaveNetModel(layers=int(gs["layers"]), blocks=int(gs["blocks"]), dilation_channels=32,
                          residual_channels=32, skip_channels=1024, end_channels=512, classes=256,
                          output_length=output_length, kernel_size=2, bias=True)
    m.load_state_dict(params_from_golden(gs), strict=True)
    return m.to(device)


def one_hot_cuda(idx, classes=256):
    idx = torch.as_tensor(np.asarray(idx)).long().cuda()
    b, l = idx.shape
    return torch.zeros(b, classes, l, device="cuda").scatter_(1, idx.view(b, 1, l), 1.0)


def assert_stream_parity(got_idx, ref_idx, ref_logits, tol=1e-4):
    """Bit-exact index stream, except that a first mismatch is accepted only where the reference's own top-1/top-2
    logit gap is below tol (a tie-break divergence, SURVEY.md section 7 hard part 3).  Returns the agreed prefix."""
    got_idx, ref_idx = np.asarray(got_idx), np.asarray(ref_idx)
    neq = np.nonzero(got_idx != ref_idx)[0]
    if len(neq) == 0:
        return len(ref_idx)
    i = int(neq[0])
    top2 = np.sort(ref_logits[i])[-2:]
    assert top2[1] - top2[0] < tol * max(1.0, float(np.abs(ref_logits[i]).max())), (
        f"stream diverges at step {i}: got {got_idx[i]} want {ref_idx[i]}, reference margin {top2[1] - top2[0]:.3e}")
    return i
