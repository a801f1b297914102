"""The MFCC front-end beyond the default filterbank: every n_mels the kernel takes (1..64), f_min 0 / 20 Hz, f_max 4000 Hz
and sr/2 (AudioProcessor(f_max=None), librosa's fmax = sr/2), against the float64 oracle.

Settings other than the default reach code the default never runs: power spectrum bins 120..239 (nb16 up to 15, the
real-FFT split of j >= 8 and its mirror shuffle), one to four passes of the mel loop per lane, filters without an FFT bin
(the reference leaves them at exactly 0), and the scalar row copies of the stream gather and the live paths
(n_mels % 4 != 0).  The band edges follow np.linspace (the last edge exactly at f_max), so a front-end with
f_max = sr/2 never puts weight on the Nyquist bin and every setting the reference takes is built.
"""
import ctypes
import warnings

import numpy as np
import pytest
import torch

from conftest import FLOOR_DB, mfcc_err, scaled_err
from honk2_b200 import AudioProcessor, LiveStreams, NativeError, synth
from oracle import mfcc_ref
from test_live_ragged import check_windows, ragged_lengths, run_ragged
from test_live_streams import make_streams, pushes, run, window_index

gpu = pytest.mark.gpu
SR = 16000
KWS_ERR_INVALID = 1

# (n_mels, f_min, f_max); f_max = 8000 is AudioProcessor(f_max=None)
DEEP = [(13, 20, 4000),    # one mel pass, scalar copies
        (17, 20, 8000),    # the whole spectrum
        (49, 20, 8000),    # four mel passes, scalar copies; refused while the last band edge could round above sr/2
        (64, 20, 1000),    # seven filters without an FFT bin
        (24, 300, 3400)]   # telephone band
DEEP_IDS = [f"{n}-{lo}-{hi}" for n, lo, hi in DEEP]


def processor(n_mels, f_min, f_max):
    return AudioProcessor(n_mels=n_mels, f_min=f_min, f_max=None if f_max == SR // 2 else f_max)


def oracle(waves, n_mels, f_min, f_max):
    return mfcc_ref.compute_mfccs_batch(waves, n_mels=n_mels, fmin=float(f_min), fmax=float(f_max))


def empty_filters(n_mels, f_min, f_max):
    return np.flatnonzero(~mfcc_ref.mel_filterbank(n_mels=n_mels, fmin=float(f_min), fmax=float(f_max)).any(axis=1))


def clips(N, seed):
    """[5, N] float32: broadband noise (energy up to sr/2), speech-like audio, and the edge cases (silence, an
    impulse, a square wave)."""
    return np.concatenate([synth.broadband(1, N, seed=seed), synth.speechlike(1, N, seed=seed),
                           synth.edge_cases(N)]).astype(np.float32)


def feature_err(got, ref):
    """conftest.mfcc_err, where a bin whose mel power the kernel computes as exactly 0 counts as -inf: the features keep
    an exact zero power at 0, as the reference does (audio_processor.py:27).  A float32 FFT can cancel exactly where the
    float64 reference leaves rounding noise (a square wave's missing harmonics under a filter one FFT bin wide): that
    is a floor bin below any floor, and a resolved bin computed as 0 is an infinite error."""
    return mfcc_err(np.where((got == 0) & (ref != 0), -np.inf, got), ref)


def to_pcm16(x):
    return np.clip(np.round(x * 32768.0), -32768, 32767).astype(np.int16)


# ---------------------------------------------------------------------------------------------
# the oracle at these settings, against torchaudio's independent implementation (CPU)

def test_oracle_filterbanks_against_torchaudio():
    """Every (n_mels, f_min, f_max) of the sweep: the same filter weights to float32 rounding, the same empty filters,
    and no weight on the Nyquist bin."""
    torchaudio = pytest.importorskip("torchaudio")
    for f_min in (0, 20):
        for f_max in (4000, 8000):
            for n in range(1, 65):
                W = mfcc_ref.mel_filterbank(n_mels=n, fmin=float(f_min), fmax=float(f_max))
                with warnings.catch_warnings():
                    warnings.simplefilter("ignore")   # torchaudio warns about filters without an FFT bin
                    fb = torchaudio.functional.melscale_fbanks(241, float(f_min), float(f_max), n, SR, norm="slaney",
                                                               mel_scale="slaney").numpy().T
                assert np.abs(fb - W).max() < 1e-6, (n, f_min, f_max)
                assert np.array_equal(fb.any(axis=1), W.any(axis=1)), (n, f_min, f_max)
                assert not W[:, 240].any(), (n, f_min, f_max)
    assert len(empty_filters(64, 20, 1000)) == 7


@pytest.mark.parametrize("n_mels,f_min,f_max", DEEP, ids=DEEP_IDS)
def test_oracle_mel_power_against_torchaudio(n_mels, f_min, f_max):
    """mfcc_ref.mel_power against torchaudio's MelSpectrogram (Slaney scale and norm, reflect pad, periodic Hann) on
    broadband and speech-like clips, as test_oracle_mfcc.test_against_torchaudio does for the default."""
    torchaudio = pytest.importorskip("torchaudio")
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        mel = torchaudio.transforms.MelSpectrogram(sample_rate=SR, n_fft=480, hop_length=160, f_min=float(f_min),
                                                   f_max=float(f_max), n_mels=n_mels, power=2.0, center=True,
                                                   pad_mode="reflect", norm="slaney", mel_scale="slaney")
    for y in clips(16001, seed=n_mels)[:2]:
        ours = mfcc_ref.mel_power(y, n_mels=n_mels, fmin=float(f_min), fmax=float(f_max)).astype(np.float64)
        ta = mel(torch.from_numpy(y)).double().numpy()
        assert ours.shape == ta.shape == (n_mels, 101)
        # Empty filters are exactly 0 here.  torchaudio spaces the band edges in float32: at f_max = 1000 its last edge
        # rounds above 1000 Hz and the last filter keeps a weight of 4e-6 of the largest at that bin.
        empty = empty_filters(n_mels, f_min, f_max)
        assert not ours[empty].any() and (ta[empty] <= 1e-4 * ta.max(axis=0)).all()
        live = ours > 0
        assert live.sum() > n_mels * 30
        assert scaled_err(2.0 * np.log(ta[live]), 2.0 * np.log(ours[live])) < 1e-4


def test_frontend_refusals_without_gpu(native_lib):
    """The C ABI refuses settings outside the kernel or the reference before it touches a device."""
    out = ctypes.c_void_p()
    for n_mels, f_min, f_max in ((0, 20.0, 4000.0), (65, 20.0, 4000.0), (40, 20.0, 8001.0), (40, 4000.0, 4000.0),
                                 (40, 4000.0, 300.0), (40, -1.0, 4000.0)):
        assert native_lib.kws_frontend_create(SR, n_mels, ctypes.c_float(f_min), ctypes.c_float(f_max), 480, 160,
                                              ctypes.byref(out)) == KWS_ERR_INVALID, (n_mels, f_min, f_max)
        assert out.value is None


# ---------------------------------------------------------------------------------------------
# on the device

@pytest.fixture(scope="module")
def dev(native_lib):
    assert torch.cuda.is_available(), "these tests need the B200"
    return torch.device("cuda", 0)


@pytest.fixture(scope="module")
def deep_ap(dev):
    cache = {}

    def get(cfg):
        if cfg not in cache:
            cache[cfg] = processor(*cfg)
        return cache[cfg]
    return get


@gpu
@pytest.mark.parametrize("f_max", [4000, 8000])
@pytest.mark.parametrize("f_min", [0, 20])
def test_every_n_mels_builds_and_matches_float64(dev, f_min, f_max):
    """n_mels = 1..64: the front-end is built, and on two short clips (broadband, speech-like) it matches the float64
    oracle at 1e-4 with the floor bins consistent."""
    waves = clips(4000, seed=f_min + f_max)[:2]
    wd = torch.from_numpy(waves).to(dev)
    refused, wrong, worst = [], [], 0.0
    for n in range(1, 65):
        ap = processor(n, f_min, f_max)
        try:
            got = ap.compute_mfccs_batch(wd).cpu().numpy()
        except NativeError as e:
            refused.append((n, str(e)))
            continue
        err, _, floor_ok = feature_err(got, oracle(waves, n, f_min, f_max))
        worst = max(worst, err)
        if not (err <= 1e-4 and floor_ok):
            wrong.append((n, err, floor_ok))
    print(f"f_min={f_min} f_max={f_max}: worst scaled error {worst:.2e} over n_mels 1..64")
    assert not refused, refused
    assert not wrong, wrong


@gpu
def test_frontend_refusals(dev):
    for kw in (dict(n_mels=0), dict(n_mels=65), dict(f_max=8001), dict(f_min=4000, f_max=4000),
               dict(f_min=5000, f_max=4000)):
        with pytest.raises(NativeError, match="kws_frontend_create"):
            AudioProcessor(**kw).compute_mfccs_batch(torch.zeros(1, 800, device=dev))


@gpu
@pytest.mark.parametrize("cfg", DEEP, ids=DEEP_IDS)
def test_deep_batch_against_float64(dev, deep_ap, cfg):
    """Clips of 241, 16001 and 144000 samples against the float64 oracle; filters without an FFT bin exactly 0."""
    ap = deep_ap(cfg)
    empty = empty_filters(*cfg)
    worst = 0.0
    for N, B in ((241, 5), (16001, 5), (144000, 2)):
        waves = clips(N, seed=N)[:B]
        got = ap.compute_mfccs_batch(torch.from_numpy(waves).to(dev)).cpu().numpy()
        ref = oracle(waves, *cfg)
        assert got.shape == ref.shape == (B, 1 + N // 160, cfg[0])
        err, n_floor, floor_ok = feature_err(got, ref)
        if not floor_ok:
            top = np.broadcast_to(ref.max(axis=-1, keepdims=True), ref.shape)
            bad = (ref < top - FLOOR_DB) & (ref != 0) & (got >= top - 2.0 * np.log(1e8))
            pytest.fail(f"N={N}: floor bins above the floor: got {got[bad][:6]}, ref {ref[bad][:6]}, frame max {top[bad][:6]}")
        assert err <= 1e-4, (N, err)
        assert not got[..., empty].any() and not got[ref == 0].any(), N   # exact zeros where the reference has them
        worst = max(worst, err)
        print(f"{cfg} N={N}: {n_floor} floor bins, {int(((got == 0) & (ref != 0)).sum())} of them exactly 0")
    print(f"{cfg}: worst scaled error {worst:.2e}; {len(empty)} empty filters")
    if cfg == (64, 20, 1000):
        assert len(empty) == 7


@gpu
@pytest.mark.parametrize("cfg", DEEP, ids=DEEP_IDS)
def test_deep_pcm16_and_stream_bit_identical(dev, deep_ap, cfg):
    """int16 PCM == float32 of s / 32768, batch and stream; compute_mfccs_stream == compute_mfccs_batch of the
    materialised windows, at shift 160 (frames shared between windows) and 100 (none shared)."""
    ap = deep_ap(cfg)
    for N in (241, 16001):
        pcm = to_pcm16(clips(N, seed=7)[:3])
        a = ap.compute_mfccs_batch(torch.from_numpy(pcm).to(dev))
        b = ap.compute_mfccs_batch(torch.from_numpy(pcm.astype(np.float32) / 32768.0).to(dev))
        assert torch.equal(a, b), N
    L = 16000 + 37 * 160 + 77
    x = synth.speechlike(1, N=L, seed=3)[0] + synth.broadband(1, N=L, seed=4)[0]
    pcm = torch.from_numpy(to_pcm16(0.5 * x)).to(dev)
    stream = pcm.float() / 32768.0
    for W, H in ((16000, 160), (16000, 100), (16001, 160)):
        got = ap.compute_mfccs_stream(stream, W, H)
        assert got.shape[0] == ap.n_stream_windows(L, W, H) > 30
        assert torch.equal(got, ap.compute_mfccs_batch(stream.unfold(0, W, H)[:got.shape[0]].contiguous())), (W, H)
        assert torch.equal(ap.compute_mfccs_stream(pcm, W, H), got), (W, H)


@gpu
@pytest.mark.parametrize("cfg", DEEP, ids=DEEP_IDS)
def test_deep_live_push_bit_identical(dev, deep_ap, cfg):
    """LiveStreams.push (float and int16) over enough pushes that both rings wrap: every valid slot ==
    compute_mfccs_batch of its window, the warm-up slots 0."""
    ap = deep_ap(cfg)
    S = 3
    for (W, H), kind in (((16000, 160), "varying"), ((16001, 480), "max")):
        max_push = 10 * H
        sizes = pushes(kind, H, max_push, 3 * 16000)
        L = sum(sizes)
        pcm = torch.from_numpy(to_pcm16(make_streams(S, L, seed=W + H))).to(dev)
        streams = pcm.float() / 32768.0
        out = run(LiveStreams(ap, S, W, H, max_push, device=dev), streams, sizes)
        out16 = run(LiveStreams(ap, S, W, H, max_push, device=dev), pcm, sizes)
        seen, n_valid = 0, 0
        for (f, v), (f16, v16), n in zip(out, out16, sizes):
            K = n // H
            assert f.shape == (S, K, 1 + W // 160, cfg[0])
            assert torch.equal(v, v16) and torch.equal(f, f16)
            k = window_index(np.full(S, seen), W, H, K)
            assert np.array_equal(v.numpy(), k >= 0)
            assert torch.count_nonzero(f[~v]).item() == 0
            vs, vj = np.nonzero(v.numpy())
            if len(vs):
                windows = streams.unfold(1, W, H)[torch.from_numpy(vs).to(dev), torch.from_numpy(k[vs, vj]).to(dev)]
                assert torch.equal(f[torch.from_numpy(vs), torch.from_numpy(vj)], ap.compute_mfccs_batch(windows))
            n_valid += len(vs)
            seen += n
        assert n_valid == S * ((L - W) // H + 1)


@gpu
@pytest.mark.parametrize("cfg", DEEP, ids=DEEP_IDS)
def test_deep_live_ragged_bit_identical(dev, deep_ap, cfg):
    """LiveStreams.push_ragged with per-stream lengths (0, 1, 159, 161, ..., max_push): each stream's windows in order,
    == compute_mfccs_batch of the materialised windows and == compute_mfccs_stream."""
    ap = deep_ap(cfg)
    S, W, H, max_push = 6, 16000, 160, 1600
    lengths = ragged_lengths(S, 60, H, max_push, seed=cfg[0])
    totals = lengths.sum(axis=0)
    streams = torch.from_numpy(make_streams(S, int(totals.max()), seed=cfg[0] + 1)).to(dev)
    assert totals.max() > 2 * (W + max_push)                       # the sample ring wraps
    res = run_ragged(LiveStreams(ap, S, W, H, max_push, device=dev), streams, lengths)
    feats = torch.cat([o for o, _, _ in res])
    s_idx = np.concatenate([si.numpy() for _, si, _ in res])
    k_idx = np.concatenate([wi.numpy() for _, _, wi in res])
    assert feats.shape[1:] == (101, cfg[0])
    check_windows(ap, streams, totals, feats, s_idx, k_idx, W, H)


@gpu
def test_a_smaller_front_end_leaves_a_larger_one_working(dev):
    """Each front-end sizes the kernels' shared memory for its own filterbank when it is created.  Creating one with
    fewer filter weights afterwards must not take that memory from the larger one: its batch, stream, live and ragged
    launches keep running and give the same features as before."""
    x = torch.from_numpy(clips(16001, seed=5)[:2]).to(dev)
    stream = x[0, :16000 + 40 * 160].contiguous()
    big = processor(64, 0, 8000)                  # the most filter weights
    want = big.compute_mfccs_batch(x)
    want_stream = big.compute_mfccs_stream(stream, 16000, 160)
    live, ragged = LiveStreams(big, 2, 16000, 160, 1600, device=dev), LiveStreams(big, 2, 16000, 160, 1600, device=dev)
    processor(1, 300, 400).compute_mfccs_batch(x)  # two FFT bins
    assert torch.equal(big.compute_mfccs_batch(x), want)
    assert torch.equal(big.compute_mfccs_stream(stream, 16000, 160), want_stream)
    streams = torch.from_numpy(make_streams(2, 17600, seed=8)).to(dev)
    f, v = run(live, streams, [1600] * 11)[-1]
    assert bool(v.all()) and torch.equal(f[:, -1], big.compute_mfccs_batch(streams[:, -16000:].contiguous()))
    lengths = np.full((11, 2), 1600)
    res = run_ragged(ragged, streams, lengths)
    feats = torch.cat([o for o, _, _ in res])
    s_idx = np.concatenate([si.numpy() for _, si, _ in res])
    k_idx = np.concatenate([wi.numpy() for _, _, wi in res])
    check_windows(big, streams, lengths.sum(axis=0), feats, s_idx, k_idx, 16000, 160)
