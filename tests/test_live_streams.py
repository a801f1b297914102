"""Live multi-stream front-end (LiveStreams / kws_live_*): S streams pushed a chunk at a time give, for every window a
push completes, features bit-identical to the offline paths on the concatenated stream.

Window k of a stream is samples [k*H, k*H + W) since its last reset.  Slot j of a push is window
floor((c - W) / H) + 1 + j for the sample count c before the push.  Note the offline off-by-one:
compute_mfccs_stream (StreamingDataset.num_samples = int((L - W) / H), dataset_utils.py:31) leaves out the last complete
window of an L-sample stream, which the live path emits in the push that completes it.
"""
import ctypes
import pickle

import numpy as np
import pytest
import torch

import honk2_b200
from honk2_b200 import AudioProcessor, LiveStreams, NativeError, synth
from honk2_b200.streaming import evaluate_stream

gpu = pytest.mark.gpu

# (W, H).  (800, 160): T = 6.  (721, 160): T = 5, the smallest shared case.  W = 16001 and 721 are not multiples of the
# hop, so neither is W + max_push: the sample ring (rounded up to 16 samples) wraps inside a frame-table row.
CONFIGS = [(16000, 160), (16000, 480), (8000, 320), (800, 160), (16001, 160), (721, 160)]
SECONDS = 4


@pytest.fixture(scope="module")
def dev(native_lib):
    assert torch.cuda.is_available(), "these tests need the B200"
    return torch.device("cuda", 0)


@pytest.fixture(scope="module")
def ap(dev):
    return AudioProcessor()


def make_streams(S, L, seed):
    """[S, L] float32: speech-like audio, a gain per stream, and stretches of exact zeros in every other stream."""
    rng = np.random.default_rng(seed)
    x = synth.speechlike(S, N=L, seed=seed) * (10.0 ** rng.uniform(-2.0, 0.0, size=(S, 1))).astype(np.float32)
    for s in range(0, S, 2):
        for _ in range(2):
            a = int(rng.integers(0, max(1, L - 6000)))
            x[s, a:a + int(rng.integers(800, 6000))] = 0.0
    return np.ascontiguousarray(x, dtype=np.float32)


def pushes(kind, H, max_push, total):
    if kind == "H":
        seq = [H]
    elif kind == "max":
        seq = [max_push]
    else:
        seq = [H, 7 * H, max_push, 2 * H, 3 * H, 5 * H]
    out, n, i = [], 0, 0
    while n < total:
        out.append(seq[i % len(seq)])
        n += out[-1]
        i += 1
    return out


def run(live, streams, sizes):
    """Push streams [S, L] (CUDA) chunk by chunk; returns [(features, valid)] per push (features cloned)."""
    res, c = [], 0
    for n in sizes:
        f, v = live.push(streams[:, c:c + n])
        res.append((f.clone(), v.clone()))
        c += n
    return res


def window_index(seen, W, H, K):
    return (np.asarray(seen)[:, None] - W) // H + 1 + np.arange(K)[None, :]


# ---------------------------------------------------------------------------------------------

@gpu
@pytest.mark.parametrize("kind", ["H", "max", "varying"])
@pytest.mark.parametrize("W,H", CONFIGS)
@pytest.mark.parametrize("S", [1, 3, 149])
def test_live_windows_bit_identical_to_offline_paths(dev, ap, S, W, H, kind):
    """Every valid slot == compute_mfccs_batch of the materialised window, and the valid windows of each stream, in
    order, == compute_mfccs_stream on the concatenated stream for all the windows that path emits; across several
    wrap-arounds of both rings."""
    max_push = 10 * H
    sizes = pushes(kind, H, max_push, SECONDS * 16000)
    L = sum(sizes)
    streams = torch.from_numpy(make_streams(S, L, seed=S * 7 + W + H)).to(dev)
    live = LiveStreams(ap, S, W, H, max_push, device=dev)
    out = run(live, streams, sizes)
    assert torch.equal(live.samples_seen, torch.full((S,), L, dtype=torch.int64))
    seen = 0
    feats, s_idx, k_idx = [], [], []
    for (f, v), n in zip(out, sizes):
        K = n // H
        assert f.shape == (S, K, 1 + W // 160, 40) and v.shape == (S, K)
        k = window_index(np.full(S, seen), W, H, K)
        assert np.array_equal(v.numpy(), k >= 0)
        assert (k[:, -1] * H + W <= seen + n).all() and ((k[:, -1] + 1) * H + W > seen + n).all()
        vs, vj = np.nonzero(v.numpy())
        feats.append(f[torch.from_numpy(vs), torch.from_numpy(vj)])
        s_idx.append(vs)
        k_idx.append(k[vs, vj])
        assert torch.count_nonzero(f[~v]).item() == 0
        seen += n
    feats = torch.cat(feats)
    s_idx, k_idx = np.concatenate(s_idx), np.concatenate(k_idx)
    n_all = (L - W) // H + 1                    # every complete window of an L-sample stream
    assert len(feats) == S * n_all
    windows = streams.unfold(1, W, H)[torch.from_numpy(s_idx).to(dev), torch.from_numpy(k_idx).to(dev)]
    assert torch.equal(feats, ap.compute_mfccs_batch(windows))
    n_off = ap.n_stream_windows(L, W, H)
    assert n_off == n_all - 1                   # the offline path leaves out the last complete window
    for s in range(S):
        rows = feats[torch.from_numpy(np.nonzero(s_idx == s)[0]).to(dev)]
        assert np.array_equal(k_idx[s_idx == s], np.arange(n_all))
        assert torch.equal(rows[:n_off], ap.compute_mfccs_stream(streams[s], W, H))


@gpu
@pytest.mark.parametrize("W,H", [(16000, 160), (800, 160), (16000, 480)])
def test_live_pcm16_equals_float_push(dev, ap, W, H):
    max_push = 10 * H
    sizes = pushes("varying", H, max_push, 3 * 16000)
    L = sum(sizes)
    pcm = np.random.default_rng(W + H).integers(-20000, 20000, size=(3, L), dtype=np.int16)
    pcm[1, 5000:9000] = 0
    a = run(LiveStreams(ap, 3, W, H, max_push, device=dev), torch.from_numpy(pcm).to(dev), sizes)
    b = run(LiveStreams(ap, 3, W, H, max_push, device=dev),
            torch.from_numpy(pcm.astype(np.float32) / 32768.0).to(dev), sizes)
    for (fa, va), (fb, vb) in zip(a, b):
        assert torch.equal(va, vb) and torch.equal(fa, fb)


@gpu
@pytest.mark.parametrize("W,H", CONFIGS)
def test_live_warm_up_mask(dev, ap, W, H):
    """A fresh stream's first ceil(W/H) - 1 slots have a negative window index: invalid and all zero, also when W is
    not a multiple of H; the mask follows the host arithmetic for every push size."""
    max_push = 10 * H
    for kind in ("H", "max", "varying"):
        sizes = pushes(kind, H, max_push, W + 3 * max_push)
        streams = torch.from_numpy(make_streams(2, sum(sizes), seed=W + H)).to(dev)
        live = LiveStreams(ap, 2, W, H, max_push, device=dev)
        seen, flags = 0, []
        for (f, v), n in zip(run(live, streams, sizes), sizes):
            assert np.array_equal(v.numpy(), window_index(np.full(2, seen), W, H, n // H) >= 0)
            assert torch.count_nonzero(f[~v]).item() == 0
            flags.append(v[0].numpy())
            seen += n
        flags = np.concatenate(flags)
        n_warm = -(-W // H) - 1
        assert not flags[:n_warm].any() and flags[n_warm:].all(), (kind, n_warm)


@gpu
def test_live_reset(dev, ap):
    """Streams 1 and 3 are reset mid-run, twice.  The first push after a reset computes frame-table rows that straddle
    the reset point (they read pre-reset ring contents); no valid window may see them.  Afterwards a reset stream's
    outputs equal a fresh state's fed the same post-reset audio; the other streams' equal a run without the reset."""
    S, W, H, max_push = 5, 16000, 160, 1600
    sizes = pushes("varying", H, max_push, 5 * 16000)
    L = sum(sizes)
    streams = torch.from_numpy(make_streams(S, L, seed=11)).to(dev)
    reset_at = {7: [1, 3], 31: [3]}           # push index -> streams reset before that push
    plain = run(LiveStreams(ap, S, W, H, max_push, device=dev), streams, sizes)
    live = LiveStreams(ap, S, W, H, max_push, device=dev)
    fresh = {}                                # reset stream -> a state created at its reset
    c = 0
    for p, n in enumerate(sizes):
        if p in reset_at:
            live.reset(reset_at[p] + reset_at[p][:1])   # (a repeated id is harmless)
            for s in reset_at[p]:
                fresh[s] = LiveStreams(ap, S, W, H, max_push, device=dev)
            assert all(int(live.samples_seen[s]) == 0 for s in reset_at[p])
        chunk = streams[:, c:c + n]
        f, v = live.push(chunk)
        for s in range(S):
            if s in fresh:
                ff, fv = fresh[s].push(chunk)
                assert torch.equal(v[s], fv[s]) and torch.equal(f[s], ff[s]), (p, s)
            else:
                assert torch.equal(v[s], plain[p][1][s]) and torch.equal(f[s], plain[p][0][s]), (p, s)
        c += n
    assert int(live.samples_seen[0]) == L and int(live.samples_seen[3]) == sum(sizes[31:])
    with pytest.raises(ValueError):
        live.reset([S])
    with pytest.raises(ValueError):
        live.reset([-1])


@gpu
@pytest.mark.parametrize("name,precision", [("res15", "bf16"), ("res15", "bf16x3"), ("res8", "bf16"),
                                            ("cnn-trad-fpool3", "bf16"), ("cnn-trad-fpool3", "fp32")])
def test_live_push_with_model(dev, ap, name, precision):
    """push(chunk, model) == model(features.view(S K, T, F)) bit for bit; valid-slot logits == evaluate_stream on the
    concatenated stream."""
    S, W, H, max_push = 3, 16000, 160, 1600
    m = honk2_b200.build_model(name, precision=precision).to(dev)
    sizes = pushes("varying", H, max_push, 3 * 16000)
    L = sum(sizes)
    streams = torch.from_numpy(make_streams(S, L, seed=5)).to(dev)
    a = LiveStreams(ap, S, W, H, max_push, device=dev)
    b = LiveStreams(ap, S, W, H, max_push, device=dev)
    c, per_stream = 0, [[] for _ in range(S)]
    with torch.no_grad():
        for n in sizes:
            chunk = streams[:, c:c + n]
            y, v = a.push(chunk, m)
            f, v2 = b.push(chunk)
            K = n // H
            assert y.shape == (S, K, 12) and torch.equal(v, v2)
            assert torch.equal(y, m(f.view(S * K, 1 + W // 160, 40)).view(S, K, -1))
            for s in range(S):
                per_stream[s].append(y[s][v[s].to(dev)])
            c += n
        for s in range(S):
            got = torch.cat(per_stream[s])[:ap.n_stream_windows(L, W, H)]
            want = evaluate_stream(m, ap, streams[s], W, H)
            assert got.shape == want.shape
            if name == "res8" and precision != "fp32":
                # packed strips: a stacked utterance's pooled mean is summed in an order set by its place in its group,
                # which differs between the two batchings (test_full_batch_permutation_invariance): a few ulp
                assert float((got - want).abs().max()) <= 2e-6 * float(want.abs().max())
            else:
                assert torch.equal(got, want)


@gpu
def test_live_refusals_and_argument_errors(dev, ap):
    for args in ((3, 16000, 100, 1000),   # shift not a multiple of the hop
                 (3, 600, 160, 1600),     # T = 4: no interior frame
                 (3, 16000, 320, 1000),   # max_push not a multiple of the shift
                 (0, 16000, 160, 1600)):  # no stream
        with pytest.raises(NativeError, match="kws_live_create"):
            LiveStreams(ap, *args, device=dev)
        assert honk2_b200._native.load().kws_live_state_bytes(ap._frontend(dev), *args) == 0
    live = LiveStreams(ap, 3, 16000, 320, 3200, device=dev)
    x = torch.zeros(3, 3200, device=dev)
    with pytest.raises(NativeError, match="multiple of the shift"):
        live.push(x[:, :480])
    with pytest.raises(NativeError, match="multiple of the shift"):
        live.push(torch.zeros(3, 3520, device=dev))   # > max_push
    with pytest.raises(ValueError):
        live.push(torch.zeros(4, 320, device=dev))
    with pytest.raises(NativeError):
        live.push(torch.zeros(3, 320))
    with pytest.raises(ValueError):
        live.reset([3])
    with pytest.raises(ValueError):
        live.reset(torch.tensor([0], device=dev))      # host ids only: the host keeps samples_seen
    assert torch.equal(live.samples_seen, torch.zeros(3, dtype=torch.int64))   # refused pushes change nothing
    # a pickled copy holds no device state: it starts afresh
    live.push(x)
    copy = pickle.loads(pickle.dumps(live))
    assert torch.equal(copy.samples_seen, torch.zeros(3, dtype=torch.int64))
    f, v = copy.push(x)
    assert not v.any() and torch.count_nonzero(f).item() == 0


def test_live_c_abi_argument_errors_without_gpu(native_lib):
    """Null handles and buffers return KWS_ERR_INVALID with a message; the size query returns 0."""
    lib = native_lib
    out = ctypes.c_void_p()
    assert lib.kws_live_state_bytes(None, 4, 16000, 160, 1600) == 0
    assert lib.kws_live_create(None, 4, 16000, 160, 1600, ctypes.byref(out)) == 1
    assert b"frontend is null" in lib.kws_last_error()
    assert lib.kws_live_create(None, 4, 16000, 160, 1600, None) == 1
    assert b"out is null" in lib.kws_last_error()
    assert lib.kws_live_push(None, None, 160, None, None) == 1
    assert b"live state is null" in lib.kws_last_error()
    assert lib.kws_live_push_pcm16(None, None, 160, None, None) == 1
    assert b"live state is null" in lib.kws_last_error()
    assert lib.kws_live_reset(None, None, 1, None) == 1
    assert b"live state is null" in lib.kws_last_error()
    lib.kws_live_destroy(None)


@gpu
def test_live_states_are_independent(dev, ap):
    """Two states on one front-end, pushed alternately, give what each gives alone."""
    sizes_a = pushes("varying", 160, 1600, 2 * 16000)
    sizes_b = pushes("varying", 320, 3200, 4 * 16000)[::-1]
    sizes_a, sizes_b = sizes_a[:len(sizes_b)], sizes_b[:len(sizes_a)]
    sa = torch.from_numpy(make_streams(3, sum(sizes_a), seed=21)).to(dev)
    sb = torch.from_numpy(make_streams(2, sum(sizes_b), seed=22)).to(dev)
    alone_a = run(LiveStreams(ap, 3, 16000, 160, 1600, device=dev), sa, sizes_a)
    alone_b = run(LiveStreams(ap, 2, 8000, 320, 3200, device=dev), sb, sizes_b)
    la = LiveStreams(ap, 3, 16000, 160, 1600, device=dev)
    lb = LiveStreams(ap, 2, 8000, 320, 3200, device=dev)
    ca = cb = 0
    for p, (na, nb) in enumerate(zip(sizes_a, sizes_b)):
        fa, va = la.push(sa[:, ca:ca + na])
        fb, vb = lb.push(sb[:, cb:cb + nb])
        assert torch.equal(fa, alone_a[p][0]) and torch.equal(va, alone_a[p][1])
        assert torch.equal(fb, alone_b[p][0]) and torch.equal(vb, alone_b[p][1])
        ca, cb = ca + na, cb + nb


@gpu
def test_live_state_bytes_match_allocation(dev, ap):
    """kws_live_state_bytes == what create takes from the device (free-memory delta, cudaMalloc rounds to 2 MiB) and
    destroy gives back."""
    fe = ap._frontend(dev)
    torch.cuda.synchronize()
    need = honk2_b200._native.load().kws_live_state_bytes(fe, 4096, 16000, 160, 1600)
    ring = 4096 * (16000 + 1600) * 4
    frames = 4096 * (17600 // 160) * 40 * 4
    assert need == ring + frames + 4096 * (8 + 4)   # + counters, first-window positions
    free0 = torch.cuda.mem_get_info(dev)[0]
    live = LiveStreams(ap, 4096, 16000, 160, 1600, device=dev)
    assert live.state_bytes() == need
    free1 = torch.cuda.mem_get_info(dev)[0]
    assert 0 <= (free0 - free1) - need < 4 << 20, (free0 - free1, need)
    del live
    free2 = torch.cuda.mem_get_info(dev)[0]
    assert abs(free2 - free0) < 4 << 20
