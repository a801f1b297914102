"""GPU parity tests proper: everything goes through the C-ABI library (ctypes) and is checked
against the CPU oracle / the committed goldens.  Tolerances are BASELINE.json's:
  MFCC features   |a-b| <= 1e-4 * max(|b|, 1)
  fp32 logits     |a-b| <= 1e-3 * max(|b|_inf per row, 1e-3), identical argmax
"""
import numpy as np
import pytest
import torch

import honk2_b200
from conftest import logit_err, mfcc_err, scaled_err
from honk2_b200 import AudioProcessor, synth
from honk2_b200.zoo import MODEL_ZOO, model_config
from oracle import mfcc_ref, model_ref

pytestmark = pytest.mark.gpu

MFCC_TOL = 1e-4
LOGIT_TOL = 1e-3
ZOO = list(MODEL_ZOO)
RESNETS = [n for n in ZOO if MODEL_ZOO[n]["name"] == "ResNet"]


@pytest.fixture(scope="module")
def dev(native_lib):
    assert torch.cuda.is_available(), "these tests need the B200"
    return torch.device("cuda", 0)


def gpu_model(name, variant, dev, precision="fp32"):
    m = honk2_b200.build_model(name, precision=precision)
    sd = m.state_dict()
    if variant == "hardened":
        synth.harden_(sd)
    return m.to(dev), {k: v.clone() for k, v in sd.items()}


# ---------------------------------------------------------------------------------------------
# front-end

def test_mfcc_matches_golden_and_oracle(dev, golden_waves, mfcc_golden):
    ap = AudioProcessor()
    for name, w in golden_waves.items():
        got = ap.compute_mfccs_batch(torch.from_numpy(w.astype(np.float32)).to(dev)).cpu().numpy()
        ref = mfcc_golden[f"{name}_feat"]
        assert got.shape == ref.shape
        err, n_floor, floor_ok = mfcc_err(got, ref)
        assert err <= MFCC_TOL, (name, err)
        assert floor_ok, f"{name}: numerical-floor bins are not floor bins in the CUDA output"
        if name != "edge":   # only the exactly periodic edge vectors have numerical-floor bins
            assert n_floor == 0, (name, n_floor)
            assert scaled_err(got, ref) <= MFCC_TOL


def test_mfcc_reference_api(dev, golden_waves):
    """compute_mfccs(np 1-D) -> (T, 40, 1) float32 (audio_processor.py:18-30)."""
    ap = AudioProcessor()
    y = golden_waves["broadband"][0]
    f = ap.compute_mfccs(y)
    assert f.shape == (101, 40, 1) and f.dtype == np.float32
    assert scaled_err(f, mfcc_ref.compute_mfccs(y)) <= MFCC_TOL
    f64 = ap.compute_mfccs(y.astype(np.float64))
    assert scaled_err(f64, f) <= MFCC_TOL
    with pytest.raises(ValueError):
        ap.compute_mfccs(np.zeros(16000, dtype=np.int16))
    with pytest.raises(ValueError):
        ap.compute_mfccs(np.full(16000, np.nan, dtype=np.float32))


def test_mfcc_zero_input_is_exact_zero(dev):
    ap = AudioProcessor()
    f = ap.compute_mfccs_batch(torch.zeros(3, 16000, device=dev))
    assert torch.count_nonzero(f).item() == 0


@pytest.mark.parametrize("n", [241, 480, 1000, 15999, 16000, 16001, 144000])
def test_mfcc_clip_lengths(dev, n):
    """T = 1 + N // 160 for any clip length that survives reflect padding (N > 240)."""
    ap = AudioProcessor()
    w = synth.broadband(2, N=n, seed=n)
    got = ap.compute_mfccs_batch(torch.from_numpy(w).to(dev)).cpu().numpy()
    ref = mfcc_ref.compute_mfccs_batch(w)
    assert got.shape == ref.shape == (2, 1 + n // 160, 40)
    assert scaled_err(got, ref) <= MFCC_TOL


def test_mfcc_batch_is_per_utterance(dev):
    """collate semantics: row b of the batch == the single-utterance call."""
    ap = AudioProcessor()
    w = torch.from_numpy(synth.speechlike(5, seed=3)).to(dev)
    full = ap.compute_mfccs_batch(w)
    for b in range(5):
        assert torch.equal(full[b], ap.compute_mfccs_batch(w[b:b + 1])[0])


@pytest.mark.parametrize("window,shift", [(16000, 160), (16000, 320), (16000, 100), (8000, 160), (700, 160),
                                          (16001, 480), (144000, 1600)])
def test_mfcc_stream_windows_equal_materialised_windows(dev, window, shift):
    """Streaming front-end (SURVEY 8f-1; dataset_utils.py:28-31,72 + audio_data_loader.py:26-29): the features of
    window k must be BIT-identical to compute_mfccs_batch on stream[k*shift : k*shift+window], whether frames are
    shared (shift a multiple of the 160-sample hop) or not (shift 100; T < 5), and agree with the CPU oracle."""
    ap = AudioProcessor()
    n_win = 37 if window < 100000 else 5
    L = (n_win + 1) * shift + window - 1          # int((L - window) / shift) == n_win
    stream = torch.from_numpy(synth.speechlike(1, N=L, seed=window + shift)[0]).to(dev)
    assert ap.n_stream_windows(L, window, shift) == n_win
    got = ap.compute_mfccs_stream(stream, window, shift)
    windows = torch.stack([stream[k * shift:k * shift + window] for k in range(n_win)])
    want = ap.compute_mfccs_batch(windows)
    assert got.shape == want.shape == (n_win, 1 + window // 160, 40)
    assert torch.equal(got, want)
    # a sub-range of the windows, into a caller-provided buffer
    out = torch.full((5, 1 + window // 160, 40), float("nan"), device=dev) if n_win >= 9 else None
    if out is not None:
        ap.compute_mfccs_stream(stream, window, shift, first=3, count=5, out=out)
        assert torch.equal(out, want[3:8])
    ks = [0, n_win - 1]
    ref = mfcc_ref.compute_mfccs_batch(windows[ks].cpu().numpy())
    assert scaled_err(got[ks].cpu().numpy(), ref) <= MFCC_TOL


@pytest.mark.parametrize("window,shift", [(16000, 160), (16000, 100), (8000, 320), (144000, 1600)])
def test_mfcc_stream_pcm16_equals_float_stream(dev, window, shift):
    """An int16 PCM stream through the streaming front-end (shared frames, edge frames, row copies, or the unshared path
    for a shift that is not a multiple of the hop): bit-identical to the float32 stream of the same samples, incl. a
    sub-range that starts at an odd sample offset."""
    ap = AudioProcessor()
    n_win = 21 if window < 100000 else 4
    L = (n_win + 1) * shift + window - 1
    pcm = np.random.default_rng(window + shift).integers(-20000, 20000, size=L, dtype=np.int16)
    s16 = torch.from_numpy(pcm).to(dev)
    sf = torch.from_numpy(pcm.astype(np.float32) / 32768.0).to(dev)
    a, b = ap.compute_mfccs_stream(s16, window, shift), ap.compute_mfccs_stream(sf, window, shift)
    assert a.shape == (n_win, 1 + window // 160, 40) and torch.equal(a, b)
    assert torch.equal(ap.compute_mfccs_stream(s16, window, shift, first=1, count=3), b[1:4])


def test_mfcc_stream_at_batch_size_and_argument_errors(dev):
    """8192 windows of 1 s at a 10 ms shift (gsc_dev_config.json:62-63) from a 83 s stream: 4 frames per window are
    computed per window, the other 97 come from the 8293-row stream frame table."""
    ap = AudioProcessor()
    L = 8192 * 160 + 16000 + 159
    stream = torch.from_numpy(synth.broadband(1, N=L, seed=9)[0]).to(dev)
    got = ap.compute_mfccs_stream(stream, 16000, 160)
    assert got.shape == (8192, 101, 40)
    idx = [0, 1, 4095, 8191]
    windows = torch.stack([stream[k * 160:k * 160 + 16000] for k in idx])
    assert torch.equal(got[idx], ap.compute_mfccs_batch(windows))
    # consecutive windows share their interior frames
    assert torch.equal(got[1:, 2:98], got[:-1, 3:99])
    with pytest.raises(ValueError):
        ap.compute_mfccs_stream(stream, 16000, 160, first=8000, count=500)
    with pytest.raises(ValueError):
        ap.compute_mfccs_stream(stream.unsqueeze(0))
    with pytest.raises(honk2_b200.NativeError):
        ap.compute_mfccs_stream(stream, 200, 160)       # reflect padding needs more than 240 samples


def test_evaluate_stream_matches_window_by_window_evaluation(dev):
    """evaluate_stream == slicing the windows like StreamingDataset, collating them and running evaluate's loop."""
    from honk2_b200.streaming import evaluate_stream, stream_window_targets
    ap = AudioProcessor()
    m, _ = gpu_model("res8", "hardened", dev)
    rng = np.random.default_rng(4)
    lens = rng.integers(3000, 20000, 12)
    labs = rng.integers(0, 12, 12)
    stream = torch.from_numpy(synth.speechlike(1, N=int(lens.sum()), seed=8)[0]).to(dev)
    targets = stream_window_targets(lens, labs, 12, 16000, 1600)
    logits, stats = evaluate_stream(m, ap, stream, 16000, 1600, targets=targets, batch_size=32)
    n = len(targets)
    windows = torch.stack([stream[k * 1600:k * 1600 + 16000] for k in range(n)])
    with torch.no_grad():
        want = m(ap.compute_mfccs_batch(windows))
    assert logits.shape == (n, 12)
    assert float((logits - want).abs().max()) <= 1e-4 * float(want.abs().max())
    assert stats["total"] == n
    assert stats["correct"] == int((want.argmax(1).cpu().numpy() == targets).sum())


def test_mfcc_large_batch_statistics(dev):
    """BASELINE size (8192 x 1 s): spot-check 16 random rows against the oracle."""
    ap = AudioProcessor()
    w = synth.broadband(8192, seed=5)
    got = ap.compute_mfccs_batch(torch.from_numpy(w).to(dev))
    idx = np.random.default_rng(0).choice(8192, 16, replace=False)
    ref = mfcc_ref.compute_mfccs_batch(w[idx])
    assert scaled_err(got[torch.from_numpy(idx).to(dev)].cpu().numpy(), ref) <= MFCC_TOL
    assert torch.isfinite(got).all()


# ---------------------------------------------------------------------------------------------
# models, fp32 path

@pytest.mark.parametrize("name", ZOO)
@pytest.mark.parametrize("variant", ["default", "hardened"])
def test_fp32_logits_match_reference_golden(dev, name, variant, model_golden):
    m, _ = gpu_model(name, variant, dev)
    x = torch.from_numpy(model_golden["feats"]).to(dev)
    with torch.no_grad():
        y = m(x).cpu().numpy()
    ref = model_golden[f"{name}/{variant}/logits"]
    assert y.shape == ref.shape
    assert logit_err(y, ref) <= LOGIT_TOL, (name, variant, logit_err(y, ref))
    assert np.array_equal(y.argmax(1), ref.argmax(1))


@pytest.mark.parametrize("name", RESNETS)
def test_fp32_resnet_other_time_lengths(dev, name, model_golden):
    m, _ = gpu_model(name, "hardened", dev)
    with torch.no_grad():
        y = m(torch.from_numpy(model_golden["feats_long"]).to(dev)).cpu().numpy()
    ref = model_golden[f"{name}/hardened/logits_long"]
    assert logit_err(y, ref) <= LOGIT_TOL


@pytest.mark.parametrize("name", ["res8", "res15", "res15_narrow", "res26", "cnn-trad-fpool3", "cnn-one-fstride4"])
def test_fp32_vs_oracle_seeded_batch(dev, name):
    """Same seeded inputs through the CUDA path and the CPU oracle; ragged batch, chunking."""
    kind, cfg = model_config(name)
    m, sd = gpu_model(name, "hardened", dev)
    feats = mfcc_ref.compute_mfccs_batch(synth.noisy_dataset_like(7, seed=9))
    x = torch.from_numpy(feats)
    ref = model_ref.forward(kind, sd, cfg, x).numpy()
    with torch.no_grad():
        y = m(x.to(dev)).cpu().numpy()
        m.chunk = {"fp32": 3, "bf16": 3}          # 7 = 3 + 3 + 1
        y_chunked = m(x.to(dev)).cpu().numpy()
        y1 = m(x[:1].to(dev)).cpu().numpy()
    assert logit_err(y, ref) <= LOGIT_TOL
    assert np.array_equal(y.argmax(1), ref.argmax(1))
    assert np.array_equal(y, y_chunked), "chunking must not change results"
    assert np.array_equal(y[:1], y1), "utterances are independent"


def test_empty_batch(dev):
    m, _ = gpu_model("res8", "default", dev)
    with torch.no_grad():
        assert m(torch.empty(0, 101, 40, device=dev)).shape == (0, 12)


def test_cnn_rejects_wrong_geometry(dev):
    m, _ = gpu_model("cnn-trad-fpool3", "default", dev)
    with pytest.raises(honk2_b200.NativeError):
        m(torch.zeros(2, 100, 40, device=dev))


def test_weights_follow_load_state_dict(dev, model_golden):
    """load_state_dict after the first forward must reach the packed device weights."""
    m, _ = gpu_model("res8", "default", dev)
    x = torch.from_numpy(model_golden["feats"]).to(dev)
    with torch.no_grad():
        m(x)
        sd = {k: v.clone() for k, v in m.state_dict().items()}
        synth.harden_(sd)
        m.load_state_dict(sd)
        y = m(x).cpu().numpy()
    assert logit_err(y, model_golden["res8/hardened/logits"]) <= LOGIT_TOL


def test_wave_to_logits_is_frontend_then_model(dev):
    ap = AudioProcessor()
    m, _ = gpu_model("res8", "hardened", dev)
    w = torch.from_numpy(synth.speechlike(6, seed=4)).to(dev)
    with torch.no_grad():
        a = m.forward_wave(w, ap)
        b = m(ap.compute_mfccs_batch(w))
    assert torch.equal(a, b)


def test_acc_kernel(dev):
    from honk2_b200.metric import Acc
    g = torch.Generator().manual_seed(0)
    logits = torch.randn(1000, 12, generator=g)
    logits[5, 3] = logits[5, 7] = 9.0   # tie -> lowest index, like torch.argmax
    target = torch.randint(0, 12, (1000,), generator=g)
    acc = Acc()
    pred = acc.accumulate(logits.to(dev), target.to(dev), return_pred=True)
    acc.accumulate(logits[:10].to(dev), target[:10].to(dev))
    c1, t1 = model_ref.acc_counts(logits, target)
    c2, t2 = model_ref.acc_counts(logits[:10], target[:10])
    assert acc.counts() == (c1 + c2, t1 + t2)
    assert torch.equal(pred.cpu(), torch.argmax(logits, 1))


@pytest.mark.parametrize("name", ["res15"])
def test_fp32_full_batch_properties(dev, name):
    """BASELINE size (B = 8192 is scaled to 1024 for the fp32 CUDA-core path to keep the suite
    short): batch-split invariance and agreement with the oracle on sampled rows."""
    kind, cfg = model_config(name)
    m, sd = gpu_model(name, "hardened", dev)
    ap = AudioProcessor()
    w = synth.broadband(1024, seed=8)
    wd = torch.from_numpy(w).to(dev)
    with torch.no_grad():
        y = m.forward_wave(wd, ap)
        y2 = torch.cat([m.forward_wave(wd[:300], ap), m.forward_wave(wd[300:], ap)])
    assert torch.equal(y, y2)
    idx = np.random.default_rng(1).choice(1024, 8, replace=False)
    ref = model_ref.forward(kind, sd, cfg, torch.from_numpy(mfcc_ref.compute_mfccs_batch(w[idx]))).numpy()
    got = y[torch.from_numpy(idx).to(dev)].cpu().numpy()
    assert logit_err(got, ref) <= LOGIT_TOL
    assert np.array_equal(got.argmax(1), ref.argmax(1))


# ---------------------------------------------------------------------------------------------
# bf16 tensor-core mode (reported separately, with its own tolerance)

BF16_TOL = 3e-2      # |a-b| <= 3e-2 * max(|b|_inf per row, 1e-3)


@pytest.mark.parametrize("name", RESNETS)
@pytest.mark.parametrize("variant", ["default", "hardened"])
def test_bf16_logits_vs_reference_golden(dev, name, variant, model_golden):
    m, _ = gpu_model(name, variant, dev, precision="bf16")
    x = torch.from_numpy(model_golden["feats"]).to(dev)
    with torch.no_grad():
        y = m(x).cpu().numpy()
    ref = model_golden[f"{name}/{variant}/logits"]
    assert np.isfinite(y).all()
    assert logit_err(y, ref) <= BF16_TOL, (name, variant, logit_err(y, ref))
    # argmax must agree wherever the reference's top-2 margin exceeds twice the bf16 error bound
    bound = BF16_TOL * np.maximum(np.abs(ref).max(axis=1), 1e-3)
    top2 = np.sort(ref, axis=1)[:, -2:]
    decided = (top2[:, 1] - top2[:, 0]) > 2 * bound
    assert np.array_equal(y.argmax(1)[decided], ref.argmax(1)[decided])


def _calibrated(name, dev, n_cal=48, seed=21):
    """Model whose argmax is spread over the classes (output layer calibrated on the oracle)."""
    kind, cfg = model_config(name)
    m = honk2_b200.build_model(name)
    sd = m.state_dict()
    synth.harden_(sd)
    cal = torch.from_numpy(mfcc_ref.compute_mfccs_batch(synth.speechlike(n_cal, seed=seed)))
    _, pooled = model_ref.resnet_forward({k: v.float() for k, v in sd.items() if v.is_floating_point()}, cfg, cal,
                                         return_pooled=True)
    synth.calibrate_output_(sd, pooled)
    return kind, cfg, m, {k: v.clone() for k, v in sd.items()}


# bf16 bound: the calibrated output layer cancels the common part of the pooled features, so the bf16
# rounding of the activations (2^-9 relative per element) is amplified by about the spread/std ratio;
# 0.15 of the row maximum is the stated tolerance for THIS ill-conditioned probe (3e-2 for plain weights).
@pytest.mark.parametrize("name,precision,tol", [("res15", "fp32", LOGIT_TOL), ("res15", "bf16", 0.15),
                                                ("res8", "fp32", LOGIT_TOL), ("res8", "bf16", 0.15)])
def test_argmax_agreement_with_diverse_classes(dev, name, precision, tol):
    """100 % argmax agreement on utterances whose oracle top-2 margin exceeds the error bound,
    with an output layer calibrated so that at least 6 of the 12 classes are hit."""
    kind, cfg, m, sd = _calibrated(name, dev)
    m.precision = precision
    m = m.to(dev)
    w = synth.speechlike(96, seed=77)
    ref = model_ref.forward(kind, sd, cfg, torch.from_numpy(mfcc_ref.compute_mfccs_batch(w))).numpy()
    ap = AudioProcessor()
    with torch.no_grad():
        y = m.forward_wave(torch.from_numpy(w).to(dev), ap).cpu().numpy()
    assert len(set(ref.argmax(1).tolist())) >= 6, "calibration failed to spread the classes"
    err = np.abs(y - ref).max(axis=1)
    bound = tol * np.maximum(np.abs(ref).max(axis=1), 1e-3)
    assert (err <= bound).all(), (err / bound).max()
    top2 = np.sort(ref, axis=1)[:, -2:]
    decided = (top2[:, 1] - top2[:, 0]) > 2 * bound
    assert decided.sum() >= (60 if precision == "fp32" else 10)
    assert np.array_equal(y.argmax(1)[decided], ref.argmax(1)[decided])
    if precision == "fp32":
        assert np.array_equal(y.argmax(1), ref.argmax(1))


def test_bf16_chunking_and_batch_split_invariance(dev):
    m, _ = gpu_model("res15", "hardened", dev, precision="bf16")
    ap = AudioProcessor()
    wd = torch.from_numpy(synth.broadband(300, seed=8)).to(dev)
    with torch.no_grad():
        y = m.forward_wave(wd, ap)
        m.chunk = {"fp32": 0, "bf16": 37}
        y2 = m.forward_wave(wd, ap)
        y3 = torch.cat([m.forward_wave(wd[:123], ap), m.forward_wave(wd[123:], ap)])
    assert torch.allclose(y, y2, rtol=0, atol=2e-3 * float(y.abs().max())), "only the pooled-sum atomics may reorder"
    assert torch.allclose(y, y3, rtol=0, atol=2e-3 * float(y.abs().max()))


CNN_TC = ["cnn-trad-fpool3"]     # the CNN shapes with a tensor-core path (cnn_tc.cu)


@pytest.mark.parametrize("name", CNN_TC)
@pytest.mark.parametrize("variant", ["default", "hardened"])
def test_bf16_cnn_logits_vs_reference_golden(dev, name, variant, model_golden):
    """conv_0 + pool + conv_1 on the tensor cores (cnn_tc_fused_kernel), first Linear as a bf16 split-K GEMM."""
    m, _ = gpu_model(name, variant, dev, precision="bf16")
    x = torch.from_numpy(model_golden["feats"]).to(dev)
    with torch.no_grad():
        y = m(x).cpu().numpy()
    ref = model_golden[f"{name}/{variant}/logits"]
    assert np.isfinite(y).all()
    assert logit_err(y, ref) <= BF16_TOL, (name, variant, logit_err(y, ref))


@pytest.mark.parametrize("B", [1, 149, 700])
def test_bf16_cnn_vs_oracle_seeded_batch(dev, B):
    """Several utterances per persistent CTA (B > 148), a partial last wave, chunking and batch splits."""
    name = "cnn-trad-fpool3"
    kind, cfg = model_config(name)
    m, sd = gpu_model(name, "hardened", dev, precision="bf16")
    feats = torch.from_numpy(mfcc_ref.compute_mfccs_batch(synth.speechlike(min(B, 64), seed=B)))
    feats = feats.repeat((B + feats.shape[0] - 1) // feats.shape[0], 1, 1)[:B].contiguous()
    feats = feats + 0.01 * torch.arange(B, dtype=torch.float32).view(B, 1, 1) / max(B, 1)   # every utterance distinct
    ref = model_ref.forward(kind, sd, cfg, feats).numpy()
    xd = feats.to(dev)
    with torch.no_grad():
        y = m(xd)
        m.chunk = {"fp32": 0, "bf16": 97}
        y2 = m(xd)
        y3 = torch.cat([m(xd[:B // 3]), m(xd[B // 3:])]) if B >= 3 else y
    assert logit_err(y.cpu().numpy(), ref) <= BF16_TOL, logit_err(y.cpu().numpy(), ref)
    assert torch.equal(y, y2), "the CNN tensor-core path is deterministic: chunking must not change a bit"
    assert torch.equal(y, y3)
    top2 = np.sort(ref, axis=1)[:, -2:]
    decided = (top2[:, 1] - top2[:, 0]) > 2 * BF16_TOL * np.maximum(np.abs(ref).max(axis=1), 1e-3)
    assert np.array_equal(y.cpu().numpy().argmax(1)[decided], ref.argmax(1)[decided])


def test_bf16_cnn_wave_to_logits(dev):
    m, _ = gpu_model("cnn-trad-fpool3", "hardened", dev, precision="bf16")
    ap = AudioProcessor()
    wd = torch.from_numpy(synth.broadband(200, seed=3)).to(dev)
    with torch.no_grad():
        y = m.forward_wave(wd, ap)
        y2 = m(ap.compute_mfccs_batch(wd))
    assert torch.equal(y, y2)


def test_tensor_core_modes_not_available_for_other_cnns(dev):
    """Shapes outside the cnn-trad-fpool3 family (and bf16x3 for any CNN) fail loudly: no silent fp32 fallback."""
    m, _ = gpu_model("cnn-one-fstride4", "default", dev, precision="bf16")
    with pytest.raises(honk2_b200.NativeError):
        m(torch.zeros(2, 101, 40, device=dev))
    m, _ = gpu_model("cnn-trad-fpool3", "default", dev, precision="bf16x3")
    with pytest.raises(honk2_b200.NativeError):
        m(torch.zeros(2, 101, 40, device=dev))


# ---------------------------------------------------------------------------------------------
# bf16x3: the split-bf16 tensor-core mode.  Operands are bf16 pairs hi + lo and every product is three MMAs with fp32
# accumulation, so it is held to the FP32 tolerance of the north star (1e-3 of the logit scale, identical argmax).

@pytest.mark.parametrize("name", RESNETS)
@pytest.mark.parametrize("variant", ["default", "hardened"])
def test_bf16x3_logits_match_reference_golden(dev, name, variant, model_golden):
    m, _ = gpu_model(name, variant, dev, precision="bf16x3")
    x = torch.from_numpy(model_golden["feats"]).to(dev)
    with torch.no_grad():
        y = m(x).cpu().numpy()
    ref = model_golden[f"{name}/{variant}/logits"]
    assert np.isfinite(y).all()
    assert logit_err(y, ref) <= LOGIT_TOL, (name, variant, logit_err(y, ref))
    assert np.array_equal(y.argmax(1), ref.argmax(1))


@pytest.mark.parametrize("name", ["res15", "res15_narrow", "res8", "res26"])
def test_bf16x3_other_time_lengths(dev, name, model_golden):
    """T = 301 frames (three strips: the position-major kernel carries the split mode for multi-strip maps)."""
    m, _ = gpu_model(name, "hardened", dev, precision="bf16x3")
    with torch.no_grad():
        y = m(torch.from_numpy(model_golden["feats_long"]).to(dev)).cpu().numpy()
    ref = model_golden[f"{name}/hardened/logits_long"]
    assert logit_err(y, ref) <= LOGIT_TOL, logit_err(y, ref)
    assert np.array_equal(y.argmax(1), ref.argmax(1))


@pytest.mark.parametrize("name", ["res15", "res8"])
def test_bf16x3_argmax_agreement_with_diverse_classes(dev, name):
    """The calibrated, spread-out output layer of test_argmax_agreement_with_diverse_classes at the fp32 tolerance."""
    kind, cfg, m, sd = _calibrated(name, dev)
    m.precision = "bf16x3"
    m = m.to(dev)
    w = synth.speechlike(96, seed=77)
    ref = model_ref.forward(kind, sd, cfg, torch.from_numpy(mfcc_ref.compute_mfccs_batch(w))).numpy()
    with torch.no_grad():
        y = m.forward_wave(torch.from_numpy(w).to(dev), AudioProcessor()).cpu().numpy()
    assert len(set(ref.argmax(1).tolist())) >= 6, "calibration failed to spread the classes"
    assert logit_err(y, ref) <= LOGIT_TOL, logit_err(y, ref)
    assert np.array_equal(y.argmax(1), ref.argmax(1))


def test_bf16x3_full_batch_matches_fp32_path_and_is_reproducible(dev):
    """BASELINE size (8192 x 1 s) through the parity report bench.py prints: bf16x3 against the fp32 CUDA-core path
    on a calibrated model -- max logit error <= 1e-3, 100 % argmax agreement, classes spread -- and bit-identical
    results from repeated launches (all MMAs of an accumulator are issued in a fixed order)."""
    from honk2_b200 import parity
    ap = AudioProcessor()
    w = torch.from_numpy(synth.broadband(8192, seed=5)).to(dev)
    cal = ap.compute_mfccs_batch(torch.from_numpy(synth.speechlike(256, seed=21)).to(dev))
    m = parity.calibrated_model("res15", cal, precision="bf16x3")
    rep = parity.parity_report(m, ap, w, "bf16x3")
    assert rep["n"] == 8192 and rep["max_logit_err"] <= LOGIT_TOL, rep
    assert rep["argmax_agree"] == 1.0, rep
    with torch.no_grad():
        y1 = m.forward_wave(w, ap)
        y2 = m.forward_wave(w, ap)
    assert float((y1 - y2).abs().max()) <= 1e-5 * float(y1.abs().max())


def test_host_pipeline_back_to_back_calls(dev):
    """HostPipeline: pinned host waveforms -> pinned host logits; two calls issued back to back with DIFFERENT inputs
    (no synchronisation in between: staging slots are reused across calls) must both equal forward_wave."""
    from honk2_b200.evaluate import HostPipeline
    ap = AudioProcessor()
    m, _ = gpu_model("res8", "hardened", dev)
    n, sub = 700, 128
    wa = torch.from_numpy(synth.broadband(n, seed=1)).pin_memory()
    wb = torch.from_numpy(synth.speechlike(n, seed=2)).pin_memory()
    oa = torch.empty((n, 12)).pin_memory()
    ob = torch.empty((n, 12)).pin_memory()
    pipe = HostPipeline(m, ap, 16000, sub_batch=sub, device=dev, slots=3)
    ea = pipe(wa, oa, sync=False)
    eb = pipe(wb, ob, sync=False)
    ea.synchronize()
    eb.synchronize()
    with torch.no_grad():
        ra = m.forward_wave(wa.to(dev), ap).cpu()
        rb = m.forward_wave(wb.to(dev), ap).cpu()
    assert torch.allclose(oa, ra, rtol=0, atol=1e-5 * float(ra.abs().max()))
    assert torch.allclose(ob, rb, rtol=0, atol=1e-5 * float(rb.abs().max()))
    oc = torch.empty((n, 12)).pin_memory()
    pipe(wa, oc)                                  # sync=True: the result is complete on return
    assert torch.equal(oc, oa)


@pytest.mark.parametrize("n", [16000, 15999, 8000, 4007, 144000])
def test_pcm16_waveforms_give_bit_identical_features(dev, n):
    """16-bit PCM input (the wav files' own format; librosa hands the reference float32(s / 32768)): the front-end converts
    while staging, so features and logits equal those of the converted floats bit for bit -- odd lengths take the
    unaligned staging path, full-scale samples included."""
    rng = np.random.default_rng(n)
    pcm = rng.integers(-32768, 32768, size=(9, n), dtype=np.int16)
    pcm[0, :8] = [-32768, 32767, 0, 1, -1, 12345, -12345, 7]
    ap = AudioProcessor()
    w16 = torch.from_numpy(pcm).to(dev)
    wf = torch.from_numpy(pcm.astype(np.float32) / 32768.0).to(dev)
    f16, ff = ap.compute_mfccs_batch(w16), ap.compute_mfccs_batch(wf)
    assert f16.dtype == torch.float32 and torch.equal(f16, ff)
    # ... and against the oracle on the converted floats
    ref = mfcc_ref.compute_mfccs_batch(pcm[:2].astype(np.float32) / 32768.0)
    assert mfcc_err(f16[:2].cpu().numpy(), ref)[0] <= MFCC_TOL
    if n == 16000:
        m, _ = gpu_model("res8", "hardened", dev)
        with torch.no_grad():
            assert torch.equal(m.forward_wave(w16, ap), m.forward_wave(wf, ap))


def test_host_pipeline_pcm16(dev):
    from honk2_b200.evaluate import HostPipeline
    ap = AudioProcessor()
    m, _ = gpu_model("res8", "hardened", dev)
    n, sub = 300, 128
    pcm = np.round(synth.broadband(n, seed=4) * 20000).clip(-32768, 32767).astype(np.int16)
    h16 = torch.from_numpy(pcm).pin_memory()
    out = torch.empty((n, 12)).pin_memory()
    pipe = HostPipeline(m, ap, 16000, sub_batch=sub, device=dev, dtype=torch.int16)
    pipe(h16, out)
    with torch.no_grad():
        ref = m.forward_wave(torch.from_numpy(pcm.astype(np.float32) / 32768.0).to(dev), ap).cpu()
    assert torch.equal(out, ref)
    with pytest.raises(ValueError):
        pipe(torch.zeros((4, 16000)).pin_memory(), out[:4])


def test_model_under_data_parallel(dev):
    """run/test.py:69-70 wraps the model in torch.nn.DataParallel whenever the box has more than one GPU, so a drop-in
    class has to survive replicate() (replicas carry their parameters as plain attributes, fresh copies every call) and
    forward() from DataParallel's worker threads, one replica per device."""
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    for name, precision in (("res15", "fp32"), ("res15", "bf16x3"), ("cnn-trad-fpool3", "fp32")):
        m, sd = gpu_model(name, "hardened", dev, precision=precision)
        feats = torch.from_numpy(mfcc_ref.compute_mfccs_batch(synth.noisy_dataset_like(11, seed=5))).to(dev)
        dp = torch.nn.DataParallel(m, device_ids=[0, 1])
        with torch.no_grad():
            y_dp = dp(feats)
            y_dp2 = dp(feats)
            y = m(feats)
        assert y_dp.device == feats.device and y_dp.shape == y.shape
        assert torch.equal(y_dp, y), (name, precision)
        assert torch.equal(y_dp2, y)


def test_audio_data_loader_yields_feature_batches(dev):
    """data_loader.AudioDataLoader (audio_data_loader.py:10-35): (FloatTensor[B, T, 40], LongTensor[B]) batches."""
    from honk2_b200.data_loader import AudioDataLoader
    waves = synth.speechlike(10, seed=3)
    ds = [(waves[i], i % 12) for i in range(10)]
    dl = AudioDataLoader({"audio_preprocessing": "MFCCs", "batch_size": 4, "shuffle": False, "num_workers": 0}, ds)
    got = list(dl)
    assert [tuple(x.shape) for x, _ in got] == [(4, 101, 40), (4, 101, 40), (2, 101, 40)]
    assert torch.equal(torch.cat([t for _, t in got]), torch.arange(10) % 12)
    ref = mfcc_ref.compute_mfccs_batch(waves)
    err, _, ok = mfcc_err(torch.cat([x for x, _ in got]).cpu().numpy(), ref)
    assert err <= MFCC_TOL and ok


@pytest.mark.parametrize("name", ["res15", "res8", "res26_narrow"])
def test_fp32_resident_weight_kernel_matches_tile_kernel(dev, monkeypatch, name, model_golden):
    """The fp32 C -> C layers run on the persistent resident-weight kernel (conv3x3_f32_res_kernel: cp.async double
    buffer, units numbered through the sub-batch); HONK2_F32_RESIDENT=0 selects the older one-tile-per-CTA kernel.  Same
    thread tile and the same order of the fp32 additions, so the logits must be bit-identical -- on a ragged batch that
    leaves the last work item of the persistent kernel half empty."""
    monkeypatch.setenv("HONK2_F32_RESIDENT", "0")
    m_tile, sd = gpu_model(name, "hardened", dev)
    monkeypatch.setenv("HONK2_F32_RESIDENT", "1")
    m_res, _ = gpu_model(name, "hardened", dev)
    feats = mfcc_ref.compute_mfccs_batch(synth.noisy_dataset_like(37, seed=21))
    x = torch.from_numpy(feats).to(dev)
    with torch.no_grad():
        y_tile, y_res = m_tile(x), m_res(x)
        y_long = m_res(torch.from_numpy(model_golden["feats_long"]).to(dev)).cpu().numpy()
    assert torch.equal(y_tile, y_res)
    kind, cfg = model_config(name)
    ref = model_ref.forward(kind, sd, cfg, torch.from_numpy(feats)).numpy()
    assert logit_err(y_res.cpu().numpy(), ref) <= LOGIT_TOL
    assert logit_err(y_long, model_golden[f"{name}/hardened/logits_long"]) <= LOGIT_TOL


@pytest.mark.parametrize("name", [n for n in MODEL_ZOO if n.startswith("cnn")])
def test_fp32_cnn_row_kernel_matches_generic_kernel(dev, monkeypatch, name):
    """The stride-1 convolutions with 4 or 8 kernel columns run on the persistent row-tile kernel (conv_row_f32_kernel);
    HONK2_F32_RESIDENT=0 keeps every convolution on the generic one-tile-per-CTA kernel.  Same order of the fp32
    additions: bit-identical logits for every member of the CNN family (those without such a layer run the generic kernel
    either way), on a ragged batch, and against the oracle."""
    monkeypatch.setenv("HONK2_F32_RESIDENT", "0")
    m_gen, sd = gpu_model(name, "hardened", dev)
    monkeypatch.setenv("HONK2_F32_RESIDENT", "1")
    m_row, _ = gpu_model(name, "hardened", dev)
    feats = mfcc_ref.compute_mfccs_batch(synth.noisy_dataset_like(19, seed=31))
    x = torch.from_numpy(feats).to(dev)
    with torch.no_grad():
        y_gen, y_row = m_gen(x), m_row(x)
    assert torch.equal(y_gen, y_row)
    kind, cfg = model_config(name)
    ref = model_ref.forward(kind, sd, cfg, torch.from_numpy(feats)).numpy()
    assert logit_err(y_row.cpu().numpy(), ref) <= LOGIT_TOL


@pytest.mark.parametrize("C,n_layers,pool,T,F,B", [
    (45, 13, None, 37, 24, 5),      # row kernel, 3 column blocks, ragged last unit (37 = 4 x 8 + 5), dilation up to 16
    (30, 7, None, 64, 48, 3),       # 30 maps (Q = 10, 3 groups), 48 columns, dilation up to 4
    (64, 4, None, 17, 16, 6),       # 64 maps (Q = 11, 6 groups: 165 KB of packed weights per layer)
    (19, 10, None, 101, 8, 9),      # one column block
    (45, 6, [2, 3], 50, 39, 7),     # pooled to 25 x 13: the column-tile resident kernel, no dilation key
    (12, 16, None, 9, 40, 4),       # 12 maps, 9 rows (two units, the second with one row), dilation up to 32 >= H
    (45, 22, None, 20, 40, 2),      # dilation 64 and 128 >= W: only the centre column of taps can touch the map
])
def test_fp32_conv_kernels_on_shapes_outside_the_zoo(dev, C, n_layers, pool, T, F, B):
    """The three fp32 convolution kernels pick their geometry (units per CTA, input maps per chunk, row pitch, register
    window or aligned taps, fallback when the weights do not fit) from the layer shape: shapes the model zoo never
    produces, against the CPU oracle, and resident-weight kernels against the tile kernel bit for bit."""
    from honk2_b200.class_registry import find_cls
    cfg = {"n_layers": n_layers, "n_feature_maps": C, "use_dilation": True, "n_labels": 7}
    if pool is not None:
        cfg["pool"] = pool
        cfg["use_dilation"] = False
    torch.manual_seed(C * 1000 + n_layers)
    m = find_cls("model.ResNet")(dict(cfg))
    m.eval()
    sd = m.state_dict()
    synth.harden_(sd)
    sdc = {k: v.clone() for k, v in sd.items()}
    x = torch.randn(B, T, F, generator=torch.Generator().manual_seed(T * F)) * 3.0
    ref = model_ref.forward("ResNet", sdc, cfg, x).numpy()
    m = m.to(dev)
    with torch.no_grad():
        y = m(x.to(dev))
    assert logit_err(y.cpu().numpy(), ref) <= LOGIT_TOL, logit_err(y.cpu().numpy(), ref)
    import os
    os.environ["HONK2_F32_RESIDENT"] = "0"
    try:
        m2 = find_cls("model.ResNet")(dict(cfg))
        m2.eval()
        m2.load_state_dict(sdc)
        m2 = m2.to(dev)
        with torch.no_grad():
            y2 = m2(x.to(dev))
    finally:
        del os.environ["HONK2_F32_RESIDENT"]
    assert torch.equal(y, y2)


def test_bf16_column_sweep_kernel_matches_position_major_kernel_at_full_batch(dev, monkeypatch):
    """BASELINE size (8192 x 1 s): the two whole-network tensor-core kernels (column sweep, resnet_sweep.cuh;
    position major, resnet_fused.cuh) compute the same network from the same bf16 operands and differ only in the
    order of the fp32 accumulation.  Any stale column (a missed cross-proxy fence between the epilogue's stores and
    the next layer's bulk copies) or lost accumulator update would show up as a gross per-utterance error; repeated
    launches also have to agree with each other."""
    ap = AudioProcessor()
    w = torch.from_numpy(synth.broadband(8192, seed=11)).to(dev)
    with torch.no_grad():
        feats = ap.compute_mfccs_batch(w)
        monkeypatch.setenv("HONK2_TC_SWEEP", "1")
        m_sweep, sd = gpu_model("res15", "hardened", dev, precision="bf16")
        ys = [m_sweep(feats) for _ in range(3)]
        monkeypatch.setenv("HONK2_TC_SWEEP", "0")
        m_pos, _ = gpu_model("res15", "hardened", dev, precision="bf16")
        y_pos = m_pos(feats)
    scale = float(y_pos.abs().max())
    assert torch.isfinite(ys[0]).all()
    for y in ys:
        assert float((y - y_pos).abs().max()) <= 1e-2 * scale
    assert float((ys[0] - ys[1]).abs().max()) <= 2e-3 * scale
    assert float((ys[0] - ys[2]).abs().max()) <= 2e-3 * scale
    # sampled rows against the fp32 CPU oracle
    kind, cfg = model_config("res15")
    idx = np.random.default_rng(2).choice(8192, 8, replace=False)
    ref = model_ref.forward(kind, sd, cfg, feats[torch.from_numpy(idx).to(dev)].cpu()).numpy()
    assert logit_err(ys[0][torch.from_numpy(idx).to(dev)].cpu().numpy(), ref) <= BF16_TOL


@pytest.mark.parametrize("name", ["res15", "res15_narrow"])
def test_bf16_resnet_other_time_lengths(dev, name, model_golden):
    """T = 301 frames: the column-sweep kernel runs three 128-row strips per column (planar layout, one bulk copy per
    8-channel plane, pad rows re-zeroed at the map's top and bottom); checked against the reference golden."""
    m, _ = gpu_model(name, "hardened", dev, precision="bf16")
    with torch.no_grad():
        y = m(torch.from_numpy(model_golden["feats_long"]).to(dev)).cpu().numpy()
    ref = model_golden[f"{name}/hardened/logits_long"]
    assert np.isfinite(y).all()
    assert logit_err(y, ref) <= BF16_TOL, logit_err(y, ref)


def test_bf16_res15_hey_snips_shaped_clips(dev):
    """BASELINE config 5 shape: 9 s clips (144 000 samples -> 901 x 40), res15 with 2 labels, waveform -> logits,
    against the CPU oracle on the same seeded clips."""
    kind, cfg = model_config("res15", n_labels=2)
    m = honk2_b200.build_model("res15", n_labels=2, precision="bf16")
    sd = m.state_dict()
    synth.harden_(sd)
    m.load_state_dict(sd)
    m = m.to(dev)
    w = synth.broadband(3, N=144000, seed=31)
    ref = model_ref.forward(kind, {k: v.clone() for k, v in sd.items()}, cfg,
                            torch.from_numpy(mfcc_ref.compute_mfccs_batch(w))).numpy()
    ap = AudioProcessor()
    with torch.no_grad():
        y = m.forward_wave(torch.from_numpy(w).to(dev), ap).cpu().numpy()
    assert y.shape == (3, 2) and np.isfinite(y).all()
    assert logit_err(y, ref) <= BF16_TOL, logit_err(y, ref)


@pytest.mark.parametrize("n_labels", [1, 35, 100])
def test_bf16_sweep_kernel_label_counts(dev, n_labels, model_golden):
    """The sweep kernel's tail computes one label per epilogue warp (12 warps for 45 maps): fewer labels than warps,
    the 35 words of GSC v2 (three labels per warp), and many more; against the CPU oracle."""
    kind, cfg = model_config("res15", n_labels=n_labels)
    m = honk2_b200.build_model("res15", n_labels=n_labels, precision="bf16")
    sd = m.state_dict()
    synth.harden_(sd)
    m.load_state_dict(sd)
    m = m.to(dev)
    x = torch.from_numpy(model_golden["feats"])
    ref = model_ref.forward(kind, {k: v.clone() for k, v in sd.items()}, cfg, x).numpy()
    with torch.no_grad():
        y = m(x.to(dev)).cpu().numpy()
    assert y.shape == (x.shape[0], n_labels) and np.isfinite(y).all()
    assert logit_err(y, ref) <= BF16_TOL, logit_err(y, ref)


ODD_MAP_PATHS = {100: "resnet_tc_sweep_kernel", 128: "resnet_tc_sweep_kernel", 129: "resnet_tc_fused_kernel",
                 97: "resnet_tc_sweep_kernel"}


@pytest.mark.parametrize("T,F,B", [(100, 8, 5), (128, 3, 2), (129, 17, 3), (97, 1, 4)])
def test_bf16_sweep_kernel_odd_map_shapes(dev, T, F, B):
    """Maps narrower than the dilation (every run is a single column: one-block windows, both stand-in arrivals),
    layers with fewer steps than the weight-prefetch step, a map of exactly one 128-row strip, a single-column map: all
    against the CPU oracle (res15 topology, 13 layers, dilation up to 16).  129 rows fill 50 % of two strips and are too
    tall to stack, so they run on the position-major kernel; test_tc_shapes.py has the sweep's real strip boundaries."""
    kind, cfg = model_config("res15")
    m, sd = gpu_model("res15", "hardened", dev, precision="bf16")
    assert _kernel_path(m, dev, T=T, F=F) == ODD_MAP_PATHS[T]
    g = torch.Generator().manual_seed(T * 100 + F)
    x = torch.randn(B, T, F, generator=g) * 3.0 - 8.0
    ref = model_ref.forward(kind, sd, cfg, x).numpy()
    with torch.no_grad():
        y = m(x.to(dev)).cpu().numpy()
    assert np.isfinite(y).all()
    assert logit_err(y, ref) <= BF16_TOL, logit_err(y, ref)


def test_eval_statistics_on_device(dev):
    """Per-class accuracy and cross entropy counted on the device (metric/per_class_acc.py:14-55,
    loss_function.py:7-9) against the oracle and torch's own CrossEntropyLoss; accumulation over ragged batches."""
    from honk2_b200.metric import PerClassAcc, ce_loss
    g = torch.Generator().manual_seed(3)
    logits = torch.randn(3001, 12, generator=g) * 4.0
    target = torch.randint(0, 11, (3001,), generator=g)          # class 11 never occurs
    pca = PerClassAcc()
    for lo, hi in ((0, 1000), (1000, 1001), (1001, 3001)):
        pca.accumulate(logits[lo:hi].to(dev), target[lo:hi].to(dev))
    ref = model_ref.per_class_counts(logits, target)
    got = pca.get_metric()
    assert set(got) == set(ref) and 11 not in got
    for k, (tot, cor) in ref.items():
        assert got[k] == cor / tot
    loss = ce_loss(logits.to(dev), target.to(dev))
    assert loss.is_cuda and loss.dim() == 0
    want = model_ref.ce_loss(logits, target)
    assert abs(float(loss) - want) <= 1e-5 * max(1.0, abs(want))
    assert abs(float(loss) - float(torch.nn.CrossEntropyLoss()(logits, target))) <= 1e-4
    pca.reset_metric()
    assert pca.get_metric() == {}
    # reference-shaped evaluate(): loss and metrics without a host sync per batch
    from honk2_b200.evaluate import evaluate
    from honk2_b200.metric import Acc

    class Loader(list):
        pass
    m, _ = gpu_model("res8", "hardened", dev)
    feats = torch.from_numpy(mfcc_ref.compute_mfccs_batch(synth.speechlike(6, seed=2)))
    tgt = torch.tensor([0, 1, 2, 3, 4, 5])
    res = evaluate(dev, "test", m, Loader([(feats[:4], tgt[:4]), (feats[4:], tgt[4:])]), ce_loss,
                   {"acc": Acc(), "per_class": PerClassAcc()}, {i: f"label{i}" for i in range(12)})
    assert set(res) == {"loss", "metric_acc", "metric_per_class"} and np.isfinite(res["loss"])
    assert all(k.startswith("label") for k in res["metric_per_class"])


# ---------------------------------------------------------------------------------------------
# packed strips: short maps (res8 / res26 after pooling, short clips) run on the column-sweep kernel with several
# utterances stacked in one 128-row strip; conv_0 + ReLU + AvgPool comes from conv0_pool_pack_kernel

def _kernel_path(m, dev, T=101, F=40):
    import ctypes as C
    lib, st = m._state(dev)
    lib.kws_model_kernel_path.restype = C.c_char_p
    return lib.kws_model_kernel_path(st["handle"], T, F, m._precision_id()).decode()


def _workspace_bytes(m, dev, B, T=101, F=40):
    lib, st = m._state(dev)
    return lib.kws_model_workspace_bytes(st["handle"], B, T, F, m._precision_id())


# The whole-network kernel every zoo ResNet runs in the two tensor-core precisions, on 1 s (101 frames) and 9 s (901
# frames) clips, as measured on a B200.  A change that moves a zoo config to another kernel has to say so here.
ZOO_KERNEL_PATHS = {
    ("dev", "bf16", 101): "resnet_tc_sweep_kernel",
    ("dev", "bf16", 901): "resnet_tc_fused_kernel",
    ("dev", "bf16x3", 101): "resnet_tc_sweep_kernel",
    ("dev", "bf16x3", 901): "resnet_tc_fused_kernel",
    ("hey_snips_res26", "bf16", 101): "resnet_tc_fused_kernel",
    ("hey_snips_res26", "bf16", 901): "resnet_tc_fused_kernel",
    ("hey_snips_res26", "bf16x3", 101): "resnet_tc_fused_kernel",
    ("hey_snips_res26", "bf16x3", 901): "resnet_tc_fused_kernel",
    ("res15", "bf16", 101): "resnet_tc_sweep_kernel",
    ("res15", "bf16", 901): "resnet_tc_sweep_kernel",
    ("res15", "bf16x3", 101): "resnet_tc_sweep_kernel",
    ("res15", "bf16x3", 901): "resnet_tc_fused_kernel",
    ("res15_narrow", "bf16", 101): "resnet_tc_sweep_kernel",
    ("res15_narrow", "bf16", 901): "resnet_tc_sweep_kernel",
    ("res15_narrow", "bf16x3", 101): "resnet_tc_sweep_kernel",
    ("res15_narrow", "bf16x3", 901): "resnet_tc_fused_kernel",
    ("res26", "bf16", 101): "resnet_tc_sweep_kernel",
    ("res26", "bf16", 901): "resnet_tc_fused_kernel",
    ("res26", "bf16x3", 101): "resnet_tc_sweep_kernel",
    ("res26", "bf16x3", 901): "resnet_tc_fused_kernel",
    ("res26_narrow", "bf16", 101): "resnet_tc_sweep_kernel",
    ("res26_narrow", "bf16", 901): "resnet_tc_fused_kernel",
    ("res26_narrow", "bf16x3", 101): "resnet_tc_sweep_kernel",
    ("res26_narrow", "bf16x3", 901): "resnet_tc_fused_kernel",
    ("res8", "bf16", 101): "resnet_tc_sweep_kernel",
    ("res8", "bf16", 901): "resnet_tc_fused_kernel",
    ("res8", "bf16x3", 101): "resnet_tc_sweep_kernel",
    ("res8", "bf16x3", 901): "resnet_tc_fused_kernel",
    ("res8_narrow", "bf16", 101): "resnet_tc_sweep_kernel",
    ("res8_narrow", "bf16", 901): "resnet_tc_fused_kernel",
    ("res8_narrow", "bf16x3", 101): "resnet_tc_sweep_kernel",
    ("res8_narrow", "bf16x3", 901): "resnet_tc_fused_kernel",
}


@pytest.mark.parametrize("name,precision,T", sorted(ZOO_KERNEL_PATHS))
def test_zoo_resnet_kernel_dispatch(dev, name, precision, T):
    assert {n for n, _, _ in ZOO_KERNEL_PATHS} == set(RESNETS)
    m, _ = gpu_model(name, "default", dev, precision=precision)
    assert _kernel_path(m, dev, T=T) == ZOO_KERNEL_PATHS[name, precision, T]


@pytest.mark.parametrize("n_layers", [0, 65])
def test_resnet_depths_without_a_whole_network_kernel(dev, n_layers):
    """No C->C layers, or more than the 64 the whole-network kernels hold: the tensor-core precisions refuse the model
    (no workspace, kernel path "unsupported", NativeError from the forward); the fp32 path still runs it."""
    from honk2_b200.class_registry import find_cls
    cfg = {"n_layers": n_layers, "n_feature_maps": 19, "use_dilation": False, "n_labels": 12}
    torch.manual_seed(n_layers)
    m = find_cls("model.ResNet")(dict(cfg))
    m.eval()
    sd = {k: v.clone() for k, v in m.state_dict().items()}
    x = torch.randn(3, 101, 40, generator=torch.Generator().manual_seed(n_layers)) * 3.0
    ref = model_ref.forward("ResNet", sd, cfg, x).numpy()
    m = m.to(dev)
    with torch.no_grad():
        y = m(x.to(dev)).cpu().numpy()
    assert logit_err(y, ref) <= LOGIT_TOL, logit_err(y, ref)
    for precision in ("bf16", "bf16x3"):
        m.precision = precision
        assert _kernel_path(m, dev) == "unsupported"
        assert _workspace_bytes(m, dev, 3) == 0
        with pytest.raises(honk2_b200.NativeError), torch.no_grad():
            m(x.to(dev))


def test_bf16_workspace_is_what_the_sweep_kernel_uses(dev):
    """res15 at 8192 x 1 s clips in bf16: the workspace is the sweep kernel's two activation buffers per SM slot,
    [n_sms][NP = 6][101][40][16 B] each, rounded up to 1 KB; nothing is reserved for any other path."""
    m, _ = gpu_model("res15", "default", dev, precision="bf16")
    assert _kernel_path(m, dev) == "resnet_tc_sweep_kernel"
    n_sms = torch.cuda.get_device_properties(dev).multi_processor_count
    buf = -(-n_sms * 6 * 101 * 40 * 16 // 1024) * 1024
    assert _workspace_bytes(m, dev, 8192) == 2 * buf


@pytest.mark.parametrize("name", ["res8", "res26", "res8_narrow", "res26_narrow"])
@pytest.mark.parametrize("precision,tol", [("bf16", BF16_TOL), ("bf16x3", LOGIT_TOL)])
def test_packed_strips_ragged_batches_vs_oracle(dev, name, precision, tol):
    """Batch sizes that do not fill the last group of stacked utterances, more groups than SMs, and sub-batching."""
    kind, cfg = model_config(name)
    m, sd = gpu_model(name, "hardened", dev, precision=precision)
    assert _kernel_path(m, dev) == "resnet_tc_sweep_kernel"
    base = torch.from_numpy(mfcc_ref.compute_mfccs_batch(synth.speechlike(48, seed=5)))
    for B in (1, 5, 48, 1301):
        feats = base.repeat((B + 47) // 48, 1, 1)[:B].contiguous()
        feats = feats + 0.02 * torch.arange(B, dtype=torch.float32).view(B, 1, 1) / B   # every utterance distinct
        with torch.no_grad():
            y = m(feats.to(dev)).cpu().numpy()
        idx = np.unique(np.concatenate([np.arange(min(B, 6)), np.arange(max(B - 6, 0), B)]))
        ref = model_ref.forward(kind, sd, cfg, feats[idx]).numpy()
        assert np.isfinite(y).all()
        assert logit_err(y[idx], ref) <= tol, (name, precision, B, logit_err(y[idx], ref))
        if precision == "bf16x3":
            assert np.array_equal(y[idx].argmax(1), ref.argmax(1))
    with torch.no_grad():
        xd = feats.to(dev)
        y_all = m(xd)
        m.chunk = {"fp32": 0, "bf16": 250, "bf16x3": 250}
        y_chunked = m(xd)
    assert torch.equal(y_all, y_chunked), "stacking is per group: sub-batching must not change a bit"


@pytest.mark.parametrize("name", ["res8", "res26"])
def test_packed_strips_match_position_major_reference(dev, monkeypatch, name):
    """Pooled maps run as packed strips on the sweep kernel; HONK2_TC_SWEEP=0 runs them on the position-major kernel,
    which has to agree within 1e-2 of the logit scale."""
    feats = torch.from_numpy(mfcc_ref.compute_mfccs_batch(synth.broadband(300, seed=13))).to(dev)
    with torch.no_grad():
        m_pack, _ = gpu_model(name, "hardened", dev, precision="bf16")
        y_pack = m_pack(feats)
        assert _kernel_path(m_pack, dev) == "resnet_tc_sweep_kernel"
        monkeypatch.setenv("HONK2_TC_SWEEP", "0")
        m_pos, _ = gpu_model(name, "hardened", dev, precision="bf16")
        y_pos = m_pos(feats)
        assert _kernel_path(m_pos, dev) == "resnet_tc_fused_kernel"
    assert float((y_pack - y_pos).abs().max()) <= 1e-2 * float(y_pos.abs().max())


@pytest.mark.parametrize("name", ["res15", "res8"])
def test_retired_tensor_core_variables_change_nothing(dev, monkeypatch, name):
    """The layout, packing, L2 policy, barrier polling and stage count of the tensor-core kernels are decided by their
    plans alone: variables that once overrode them are ignored, so the kernel and every logit bit stay the same."""
    feats = torch.from_numpy(mfcc_ref.compute_mfccs_batch(synth.broadband(300, seed=17))).to(dev)
    with torch.no_grad():
        m, _ = gpu_model(name, "hardened", dev, precision="bf16")
        path, y = _kernel_path(m, dev), m(feats)
        for var, value in (("HONK2_TC_SWEEP_K32", "0"), ("HONK2_TC_SWEEP_PACK", "0"), ("HONK2_TC_L2POLICY", "0"),
                           ("HONK2_TC_WAIT_POLLS", "0"), ("HONK2_TC_SWEEP_STAGES", "3")):
            monkeypatch.setenv(var, value)
        m_env, _ = gpu_model(name, "hardened", dev, precision="bf16")
        assert _kernel_path(m_env, dev) == path == "resnet_tc_sweep_kernel"
        assert torch.equal(m_env(feats), y)


SHORT_CLIP_PATHS = {("res15", 50): "resnet_tc_sweep_kernel", ("res15", 33): "resnet_tc_sweep_kernel",
                    ("res15_narrow", 61): "resnet_tc_fused_kernel", ("res8", 57): "resnet_tc_sweep_kernel"}


@pytest.mark.parametrize("name,T", list(SHORT_CLIP_PATHS))
def test_packed_strips_short_clips(dev, name, T):
    """Short clips: unpooled maps of fewer than 77 rows are stacked with dmax (16 for res15) zero rows between them, as
    many as fit a 128-row strip (two of 50 or 33 rows; eight of res8's pooled 14).  Two maps of 61 rows do not fit, and a
    single map that fills less than 60 % of its strip stays on the position-major kernel."""
    kind, cfg = model_config(name)
    rng = np.random.default_rng(T)
    feats = torch.from_numpy((rng.standard_normal((37, T, 40)) * 4 - 6).astype(np.float32))
    for precision, tol in (("bf16", BF16_TOL), ("bf16x3", LOGIT_TOL)):
        m, sd = gpu_model(name, "hardened", dev, precision=precision)
        assert _kernel_path(m, dev, T=T) == SHORT_CLIP_PATHS[name, T], precision
        with torch.no_grad():
            y = m(feats.to(dev)).cpu().numpy()
        ref = model_ref.forward(kind, sd, cfg, feats).numpy()
        assert logit_err(y, ref) <= tol, (name, T, precision, logit_err(y, ref))


# ---------------------------------------------------------------------------------------------
# size-independent properties at BASELINE's full batch (8192 clips): utterances are independent, so a permutation of the
# batch must permute the logits BIT FOR BIT -- whatever SM, strip position, stacking group or sub-batch an utterance
# lands in -- and repeated launches must agree bit for bit.

@pytest.mark.parametrize("name,precision", [("res15", "bf16"), ("res15", "bf16x3"), ("res8", "bf16"), ("res26", "bf16"),
                                            ("res15_narrow", "bf16"), ("cnn-trad-fpool3", "bf16"), ("res8", "fp32")])
def test_full_batch_permutation_invariance(dev, name, precision):
    B = 8192 if precision != "fp32" else 1024
    ap = AudioProcessor()
    w = torch.from_numpy(synth.broadband(B, seed=31)).to(dev)
    m, _ = gpu_model(name, "hardened", dev, precision=precision)
    g = torch.Generator().manual_seed(5)
    perm = torch.randperm(B, generator=g).to(dev)
    with torch.no_grad():
        feats = ap.compute_mfccs_batch(w)
        y = m(feats)
        y_again = m(feats)
        y_perm = m(feats[perm].contiguous())
        f_perm = ap.compute_mfccs_batch(w[perm].contiguous())
    assert torch.isfinite(y).all()
    assert torch.equal(y, y_again), "repeated launches differ"
    if name in ("res8", "res26") and precision != "fp32":
        # packed strips: the pooled mean of a stacked utterance is reduced over the TMEM lanes it happens to occupy, so its
        # position inside the group of 4 (2) changes the ORDER of that fp32 sum, nothing else: a few ulp of the logit scale
        assert float((y[perm] - y_perm).abs().max()) <= 2e-6 * float(y.abs().max())
    else:
        assert torch.equal(y[perm], y_perm), "an utterance's logits depend on its position in the batch"
    assert torch.equal(feats[perm], f_perm), "a clip's features depend on its position in the batch"


def test_mfcc_gain_shift_property_full_batch(dev):
    """Scaling a clip by 2^k scales every power by 4^k exactly (power-of-two gains commute with fp32 rounding), so the
    features shift by 4 k ln 2 up to the rounding of the logarithm -- checked on the full 8192-clip batch."""
    ap = AudioProcessor()
    w = torch.from_numpy(synth.broadband(8192, seed=17)).to(dev)
    with torch.no_grad():
        f1 = ap.compute_mfccs_batch(w)
        f2 = ap.compute_mfccs_batch(w * 8.0)
    shift = 4.0 * 3 * float(np.log(2.0))
    assert float((f2 - f1 - shift).abs().max()) <= 2e-5 * 40
