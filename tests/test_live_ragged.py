"""Ragged pushes of the live front-end (LiveStreams.push_ragged / kws_live_push_ragged*): every stream brings its own
number of samples, any number in [0, max_push], and only the windows a push completes come back, compacted, ordered by
stream and then window.  Across any sequence of pushes each stream emits its complete windows 0, 1, 2, ... exactly
once, bit-identical to compute_mfccs_batch on the materialised windows.
"""
import ctypes

import numpy as np
import pytest
import torch

import honk2_b200
from honk2_b200 import AudioProcessor, LiveStreams, NativeError, synth
from honk2_b200.streaming import evaluate_stream, ragged_push_plan

gpu = pytest.mark.gpu

# (W, H), as in the uniform-push tests: W = 16001 and 721 are not multiples of the hop, so the sample ring wraps inside
# a frame-table row.
CONFIGS = [(16000, 160), (16000, 480), (8000, 320), (800, 160), (16001, 160), (721, 160)]


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
        a = int(rng.integers(0, max(1, L - 6000)))
        x[s, a:a + int(rng.integers(800, 6000))] = 0.0
    return np.ascontiguousarray(x, dtype=np.float32)


def ragged_lengths(S, n_pushes, H, max_push, seed):
    """[n_pushes, S] int: per stream a pattern.  s % 4 == 0: the special lengths (0, 1, 159, 160, 161, H +- 1, 1024,
    max_push) at random; 1: idle for the first two thirds, then specials; 2: max_push for the first two thirds, then
    specials; 3: uniform in [0, max_push]."""
    rng = np.random.default_rng(seed)
    special = np.array(sorted({0, 1, 159, 160, 161, H - 1, H, H + 1, 1024, max_push}))
    special = special[special <= max_push]
    out = rng.choice(special, size=(n_pushes, S))
    long_run = (2 * n_pushes) // 3
    kind = np.arange(S) % 4
    out[:long_run, kind == 1] = 0
    out[:long_run, kind == 2] = max_push
    out[:, kind == 3] = rng.integers(0, max_push + 1, size=(n_pushes, int((kind == 3).sum())))
    return out.astype(np.int64)


def gather_samples(flat, L, seen, n):
    """The concatenated new samples of every stream: stream s's [seen[s], seen[s] + n[s]) of a flat [S * L] tensor."""
    idx = np.repeat(np.arange(len(n)) * L + seen - (np.cumsum(n) - n), n) + np.arange(int(n.sum()))
    return flat[torch.from_numpy(idx).to(flat.device)]


def run_ragged(live, streams, lengths, model=None):
    """Push the rows of lengths [P, S] of streams [S, L] (CUDA); returns [(out, stream_ids, window_ids)] per push."""
    S, L = streams.shape
    flat = streams.reshape(-1)
    seen = np.zeros(S, dtype=np.int64)
    res = []
    for n in lengths:
        o, si, wi = live.push_ragged(gather_samples(flat, L, seen, n), n, model)
        res.append((o.clone(), si, wi))
        seen += n
    return res


def check_windows(ap, streams, totals, feats, s_idx, k_idx, W, H):
    """Every row == compute_mfccs_batch of its window; per stream, ids 0 .. n_all - 1 in order; the rows before the last
    complete window == compute_mfccs_stream."""
    dev = streams.device
    n_all = np.where(totals >= W, (totals - W) // H + 1, 0)
    assert len(feats) == n_all.sum()
    if len(feats):
        windows = streams.unfold(1, W, H)[torch.from_numpy(s_idx).to(dev), torch.from_numpy(k_idx).to(dev)]
        assert torch.equal(feats, ap.compute_mfccs_batch(windows))
    for s in range(streams.shape[0]):
        sel = np.flatnonzero(s_idx == s)
        assert np.array_equal(k_idx[sel], np.arange(n_all[s])), s
        n_off = ap.n_stream_windows(int(totals[s]), W, H)
        if n_off > 0:
            rows = feats[torch.from_numpy(sel[:n_off]).to(dev)]
            assert torch.equal(rows, ap.compute_mfccs_stream(streams[s, :int(totals[s])], W, H)), s


# ---------------------------------------------------------------------------------------------

def test_ragged_plan_matches_brute_force():
    """ragged_push_plan against an enumeration of the windows each push completes, and its launch bounds."""
    rng = np.random.default_rng(0)
    for W, H in CONFIGS:
        for trial in range(20):
            S = int(rng.integers(1, 12))
            seen = rng.integers(0, 3 * W, size=S) if trial % 2 else 160 * rng.integers(0, W // 80, size=S)
            n = rng.choice([0, 1, 159, 160, 161, H - 1, H + 1, 1024, 10 * H, int(rng.integers(0, 10 * H))], size=S)
            plan = ragged_push_plan(seen, n, W, H)
            want_s, want_k, rows = [], [], 0
            for s in range(S):
                for k in range(0, (seen[s] + n[s]) // H + 2):
                    if seen[s] < k * H + W <= seen[s] + n[s]:     # complete after the push, not before
                        want_s.append(s)
                        want_k.append(k)
                rows += sum(1 for r in range(-2, (seen[s] + n[s]) // 160 + 2)
                            if seen[s] < 160 * r + 240 <= seen[s] + n[s])
            assert np.array_equal(plan.stream_ids, want_s) and np.array_equal(plan.window_ids, want_k)
            assert plan.stream_ids.dtype == plan.window_ids.dtype == np.int64
            assert len(want_s) <= plan.window_bound == sum(-(-int(x) // H) for x in n)
            assert rows <= plan.row_bound == sum(-(-int(x) // 160) for x in n)
            if trial % 2 == 0 and (n % 160 == 0).all():
                assert rows == plan.row_bound                     # exact for aligned pushes


def test_ragged_c_abi_argument_errors_without_gpu(native_lib):
    lib = native_lib
    assert lib.kws_live_ragged_workspace_bytes(None) == 0
    lengths = (ctypes.c_int32 * 2)(160, 160)
    for fn in (lib.kws_live_push_ragged, lib.kws_live_push_ragged_pcm16):
        assert fn(None, None, lengths, None, None, None, 4, None, None, 0, None) == 1
        assert b"live state is null" in lib.kws_last_error()


@gpu
@pytest.mark.parametrize("W,H", CONFIGS)
@pytest.mark.parametrize("S", [1, 3, 149])
def test_ragged_windows_bit_identical_to_offline_paths(dev, ap, S, W, H):
    max_push = 10 * H
    lengths = ragged_lengths(S, 48, H, max_push, seed=S * 13 + W + H)
    totals = lengths.sum(0)
    streams = torch.from_numpy(make_streams(S, int(totals.max()), seed=S + W + H)).to(dev)
    live = LiveStreams(ap, S, W, H, max_push, device=dev)
    out = run_ragged(live, streams, lengths)
    assert torch.equal(live.samples_seen, torch.from_numpy(totals))
    seen = np.zeros(S, dtype=np.int64)
    for (f, si, wi), n in zip(out, lengths):
        plan = ragged_push_plan(seen, n, W, H)
        assert f.shape == (len(plan.stream_ids), 1 + W // 160, 40)
        assert torch.equal(si, torch.from_numpy(plan.stream_ids)) and torch.equal(wi, torch.from_numpy(plan.window_ids))
        seen += n
    feats = torch.cat([f for f, _, _ in out])
    s_idx = np.concatenate([si.numpy() for _, si, _ in out])
    k_idx = np.concatenate([wi.numpy() for _, _, wi in out])
    check_windows(ap, streams, totals, feats, s_idx, k_idx, W, H)


@gpu
@pytest.mark.parametrize("S,W,H", [(6001, 800, 160), (149, 16001, 160), (3, 16000, 480)])
def test_ragged_device_ids_and_count(dev, ap, S, W, H):
    """Through the C ABI: the device's n_windows, win_stream and win_index equal the host plan, and the features equal
    LiveStreams.push_ragged's on a second state.  S = 6001 spans several CTAs of the plan's scan."""
    lib = honk2_b200._native.load()
    max_push = 10 * H
    lengths = ragged_lengths(S, 12 if S > 1000 else 40, H, max_push, seed=S + W)
    totals = lengths.sum(0)
    streams = torch.from_numpy(make_streams(S, int(totals.max()), seed=S)).to(dev)
    flat = streams.reshape(-1)
    a = LiveStreams(ap, S, W, H, max_push, device=dev)
    b = LiveStreams(ap, S, W, H, max_push, device=dev)
    handle = b._state()
    ws = torch.empty(lib.kws_live_ragged_workspace_bytes(handle), dtype=torch.uint8, device=dev)
    cap = S * (max_push // H)
    feat = torch.empty((cap, 1 + W // 160, 40), device=dev)
    ids = torch.empty((2, cap), dtype=torch.int64, device=dev)
    m = torch.empty((1,), dtype=torch.int64, device=dev)
    seen = np.zeros(S, dtype=np.int64)
    feats, s_idx, k_idx = [], [], []
    for n in lengths:
        x = gather_samples(flat, streams.shape[1], seen, n)
        fa, sa, ka = a.push_ragged(x, n)
        n32 = np.ascontiguousarray(n, dtype=np.int32)
        assert lib.kws_live_push_ragged(handle, ctypes.c_void_p(x.data_ptr()), ctypes.c_void_p(n32.ctypes.data),
                                        ctypes.c_void_p(feat.data_ptr()), ctypes.c_void_p(ids[0].data_ptr()),
                                        ctypes.c_void_p(ids[1].data_ptr()), cap, ctypes.c_void_p(m.data_ptr()),
                                        ctypes.c_void_p(ws.data_ptr()), ws.numel(),
                                        ctypes.c_void_p(torch.cuda.current_stream(dev).cuda_stream)) == 0
        M = len(sa)
        assert int(m.item()) == M
        assert torch.equal(ids[0, :M].cpu(), sa) and torch.equal(ids[1, :M].cpu(), ka)
        assert torch.equal(feat[:M], fa)
        feats.append(fa)
        s_idx.append(sa.numpy())
        k_idx.append(ka.numpy())
        seen += n
    check_windows(ap, streams, totals, torch.cat(feats), np.concatenate(s_idx), np.concatenate(k_idx), W, H)


@gpu
@pytest.mark.parametrize("W,H", [(16000, 160), (8000, 320)])
def test_ragged_equals_uniform_push_and_mixes_with_it(dev, ap, W, H):
    """Equal aligned lengths: ragged output == the valid slots of push, in order, bit for bit.  Aligned ragged pushes
    interleaved with uniform pushes on one state continue correctly; after a misaligned ragged push, push raises
    ValueError and changes nothing."""
    S, max_push = 5, 10 * H
    sizes = [H, 7 * H, max_push, 2 * H, 3 * H, 5 * H] * 6
    L = sum(sizes) + 4 * max_push
    streams = torch.from_numpy(make_streams(S, L, seed=W)).to(dev)
    flat = streams.reshape(-1)
    uni = LiveStreams(ap, S, W, H, max_push, device=dev)
    rag = LiveStreams(ap, S, W, H, max_push, device=dev)
    mix = LiveStreams(ap, S, W, H, max_push, device=dev)
    seen = np.zeros(S, dtype=np.int64)
    rng = np.random.default_rng(1)
    for p, n in enumerate(sizes):
        lengths = np.full(S, n, dtype=np.int64)
        x = gather_samples(flat, L, seen, lengths)
        f, v = uni.push(streams[:, seen[0]:seen[0] + n])
        g, si, wi = rag.push_ragged(x, lengths)
        vs, vj = np.nonzero(v.numpy())
        assert torch.equal(g, f[torch.from_numpy(vs), torch.from_numpy(vj)])
        assert np.array_equal(si.numpy(), vs)
        assert np.array_equal(wi.numpy(), ((seen[:, None] - W) // H + 1 + np.arange(n // H)[None, :])[vs, vj])
        # the mixed state: uniform pushes on odd steps, ragged pushes of the same samples split unevenly (multiples of
        # 160 per stream, so the counts stay aligned) on even steps
        if p % 2:
            fm, vm = mix.push(streams[:, seen[0]:seen[0] + n])
            assert torch.equal(fm, f) and torch.equal(vm, v)
        else:
            cut = 160 * rng.integers(0, n // 160 + 1, size=S)
            first, second = cut, lengths - cut
            g1, s1, w1 = mix.push_ragged(gather_samples(flat, L, seen, first), first)
            g2, s2, w2 = mix.push_ragged(gather_samples(flat, L, seen + first, second), second)
            key = np.concatenate([s1.numpy(), s2.numpy()]) * 10 ** 6 + np.concatenate([w1.numpy(), w2.numpy()])
            order = torch.from_numpy(np.argsort(key, kind="stable")).to(dev)
            assert torch.equal(torch.cat([g1, g2])[order], g)
        seen += n
    # misaligned: push refuses and changes nothing; a realigning ragged push makes it usable again
    odd = np.array([1, 0, 159, 160, 161], dtype=np.int64)
    g, si, wi = mix.push_ragged(gather_samples(flat, L, seen, odd), odd)
    ref = rag.push_ragged(gather_samples(flat, L, seen, odd), odd)
    assert torch.equal(g, ref[0]) and torch.equal(si, ref[1]) and torch.equal(wi, ref[2])
    seen += odd
    before = mix.samples_seen
    with pytest.raises(ValueError, match="stream 0 has seen"):
        mix.push(torch.zeros(S, H, device=dev))
    assert torch.equal(mix.samples_seen, before)
    fix = (-seen) % 160
    for st in (mix, rag):
        st.push_ragged(gather_samples(flat, L, seen, fix), fix)
    seen += fix
    assert (seen % 160 == 0).all()
    lengths = np.full(S, max_push, dtype=np.int64)
    chunk = torch.stack([streams[s, seen[s]:seen[s] + max_push] for s in range(S)])
    fm, vm = mix.push(chunk)
    g, si, wi = rag.push_ragged(chunk.reshape(-1), lengths)
    vs, vj = np.nonzero(vm.numpy())
    assert torch.equal(g, fm[torch.from_numpy(vs), torch.from_numpy(vj)]) and np.array_equal(si.numpy(), vs)


@gpu
@pytest.mark.parametrize("W,H", [(16000, 160), (16001, 160), (16000, 480)])
def test_ragged_pcm16_equals_float_push(dev, ap, W, H):
    S, max_push = 7, 10 * H
    lengths = ragged_lengths(S, 30, H, max_push, seed=W + H)
    L = int(lengths.sum(0).max())
    pcm = np.random.default_rng(W).integers(-20000, 20000, size=(S, L), dtype=np.int16)
    pcm[1, 5000:9000] = 0
    a = run_ragged(LiveStreams(ap, S, W, H, max_push, device=dev), torch.from_numpy(pcm).to(dev), lengths)
    b = run_ragged(LiveStreams(ap, S, W, H, max_push, device=dev),
                   torch.from_numpy(pcm.astype(np.float32) / 32768.0).to(dev), lengths)
    assert sum(len(f) for f, _, _ in a) > 0
    for (fa, sa, ka), (fb, sb, kb) in zip(a, b):
        assert torch.equal(fa, fb) and torch.equal(sa, sb) and torch.equal(ka, kb)


@gpu
def test_ragged_reset(dev, ap):
    """Streams 2 and 3 are reset mid-run: afterwards their windows restart at 0 and equal a fresh state's fed the same
    post-reset audio; the other streams' equal a run without the reset."""
    S, W, H, max_push = 5, 16000, 160, 1600
    lengths = ragged_lengths(S, 70, H, max_push, seed=3)
    L = int(lengths.sum(0).max())
    streams = torch.from_numpy(make_streams(S, L, seed=11)).to(dev)
    flat = streams.reshape(-1)
    plain = run_ragged(LiveStreams(ap, S, W, H, max_push, device=dev), streams, lengths)
    live = LiveStreams(ap, S, W, H, max_push, device=dev)
    reset_at = {20: [2, 3], 41: [3]}
    fresh = {}
    seen = np.zeros(S, dtype=np.int64)
    restarted = set()
    for p, n in enumerate(lengths):
        if p in reset_at:
            live.reset(reset_at[p])
            for s in reset_at[p]:
                fresh[s] = LiveStreams(ap, S, W, H, max_push, device=dev)
            assert all(int(live.samples_seen[s]) == 0 for s in reset_at[p])
        x = gather_samples(flat, L, seen, n)
        f, si, wi = live.push_ragged(x, n)
        for s in range(S):
            mine = torch.from_numpy(np.flatnonzero(si.numpy() == s)).to(dev)
            if s in fresh:
                ff, fs, fw = fresh[s].push_ragged(x, n)
                theirs = np.flatnonzero(fs.numpy() == s)
                want_k = fw.numpy()[theirs]
                ff = ff[torch.from_numpy(theirs).to(dev)]
                if len(want_k) and s not in restarted:
                    assert want_k[0] == 0
                    restarted.add(s)
            else:
                pf, ps, pw = plain[p]
                theirs = np.flatnonzero(ps.numpy() == s)
                want_k = pw.numpy()[theirs]
                ff = pf[torch.from_numpy(theirs).to(dev)]
            assert np.array_equal(wi.numpy()[mine.cpu().numpy()], want_k), (p, s)
            assert torch.equal(f[mine], ff), (p, s)
        seen += n
    assert restarted == {2, 3}


class CountingModel(torch.nn.Module):
    def __init__(self, m):
        super().__init__()
        self.m, self.calls, self.n_labels = m, 0, m.n_labels

    def forward(self, x):
        self.calls += 1
        return self.m(x)


@gpu
@pytest.mark.parametrize("name,precision", [("res15", "bf16"), ("res15", "bf16x3"), ("res8", "bf16"),
                                            ("cnn-trad-fpool3", "bf16"), ("cnn-trad-fpool3", "fp32")])
def test_ragged_push_with_model(dev, ap, name, precision):
    """push_ragged(.., model) == model(features) bit for bit; per-stream logits == evaluate_stream; no model call while
    no window completes."""
    S, W, H, max_push = 4, 16000, 160, 1600
    m = CountingModel(honk2_b200.build_model(name, precision=precision).to(dev))
    lengths = ragged_lengths(S, 70, H, max_push, seed=5)
    lengths[:4] = [[160, 1, 1024, 0], [0, 0, 0, 0], [1600, 159, 0, 1600], [161, 0, 1, 1]]   # no window completes yet
    totals = lengths.sum(0)
    streams = torch.from_numpy(make_streams(S, int(totals.max()), seed=5)).to(dev)
    a = LiveStreams(ap, S, W, H, max_push, device=dev)
    b = LiveStreams(ap, S, W, H, max_push, device=dev)
    flat = streams.reshape(-1)
    seen = np.zeros(S, dtype=np.int64)
    per_stream = [[] for _ in range(S)]
    empty = checked = 0
    with torch.no_grad():
        for p, n in enumerate(lengths):
            x = gather_samples(flat, streams.shape[1], seen, n)
            calls = m.calls
            y, si, wi = a.push_ragged(x, n, m)
            f, si2, wi2 = b.push_ragged(x, n)
            assert torch.equal(si, si2) and torch.equal(wi, wi2) and y.shape == (len(si), 12)
            if len(si) == 0:
                assert m.calls == calls and y.device == dev
                empty += 1
            else:
                assert m.calls == calls + 1
                assert torch.equal(y, m(f))
            for s in range(S):
                per_stream[s].append(y[torch.from_numpy(np.flatnonzero(si.numpy() == s)).to(dev)])
            seen += n
        for s in range(S):
            n_off = ap.n_stream_windows(int(totals[s]), W, H)
            if n_off <= 0:
                continue
            checked += 1
            got = torch.cat(per_stream[s])[:n_off]
            want = evaluate_stream(m.m, ap, streams[s, :int(totals[s])], W, H)
            assert got.shape == want.shape
            if name == "res8" and precision != "fp32":
                # packed strips: the pooled mean's summation order depends on the batching (see test_live_streams)
                assert float((got - want).abs().max()) <= 2e-6 * float(want.abs().max())
            else:
                assert torch.equal(got, want)
    assert empty >= 4 and checked >= 3


@gpu
def test_ragged_refusals(dev, ap):
    """Bad lengths, sums, dtypes, capacity and workspace are refused before anything changes: the state then continues
    exactly like a fresh one fed the same audio."""
    lib = honk2_b200._native.load()
    S, W, H, max_push = 3, 800, 160, 1600
    live = LiveStreams(ap, S, W, H, max_push, device=dev)
    x = torch.zeros(4000, device=dev)
    for lengths in ([-1, 0, 0], [max_push + 1, 0, 0], [0, 0], [0, 0, 0, 0]):
        with pytest.raises(ValueError):
            live.push_ragged(x[:max(0, sum(lengths))], lengths)
    with pytest.raises(ValueError, match="add up to"):
        live.push_ragged(x[:100], [50, 49, 0])
    with pytest.raises(ValueError):
        live.push_ragged(x[:10].double(), [10, 0, 0])
    with pytest.raises(ValueError):
        live.push_ragged(x[:10].view(2, 5), [10, 0, 0])
    with pytest.raises(ValueError):
        live.push_ragged(x[:10], torch.tensor([10, 0, 0], device=dev))
    with pytest.raises(ValueError, match="out must be"):
        live.push_ragged(x[:1000], [1000, 0, 0], out=torch.empty((6, 6, 40), device=dev))   # needs ceil(1000/160) = 7
    with pytest.raises(NativeError):
        live.push_ragged(torch.zeros(10), [10, 0, 0])
    # the C ABI's own checks
    handle = live._state()
    need = lib.kws_live_ragged_workspace_bytes(handle)
    assert need > 0
    ws = torch.empty(need, dtype=torch.uint8, device=dev)
    feat = torch.empty((20, 6, 40), device=dev)

    def c_push(lengths, capacity=20, ws_bytes=need, samples=x):
        n32 = (ctypes.c_int32 * S)(*lengths)
        return lib.kws_live_push_ragged(handle, ctypes.c_void_p(samples.data_ptr()) if samples is not None else None,
                                        n32, ctypes.c_void_p(feat.data_ptr()), None, None, capacity, None,
                                        ctypes.c_void_p(ws.data_ptr()), ws_bytes, None)
    for args, msg in ((([-1, 0, 0],), b"max_push"), (([0, max_push + 1, 0],), b"max_push"),
                      (([1000, 161, 0], 8), b"capacity"), (([10, 0, 0], 20, need - 1), b"workspace"),
                      (([10, 0, 0], 20, need, None), b"samples is null")):
        assert c_push(*args) == 1
        assert msg in lib.kws_last_error(), lib.kws_last_error()
    n32 = (ctypes.c_int32 * S)(0, 0, 0)
    assert lib.kws_live_push_ragged(handle, None, None, None, None, None, 0, None, None, 0, None) == 1
    assert b"lengths is null" in lib.kws_last_error()
    assert lib.kws_live_push_ragged(handle, None, n32, None, None, None, 0, None, None, 0, None) == 1
    assert b"workspace" in lib.kws_last_error()
    assert torch.equal(live.samples_seen, torch.zeros(S, dtype=torch.int64))
    # nothing reached the device: the state continues like a fresh one
    lengths = ragged_lengths(S, 20, H, max_push, seed=9)
    streams = torch.from_numpy(make_streams(S, int(lengths.sum(0).max()), seed=9)).to(dev)
    for (fa, sa, ka), (fb, sb, kb) in zip(run_ragged(live, streams, lengths),
                                          run_ragged(LiveStreams(ap, S, W, H, max_push, device=dev), streams, lengths)):
        assert torch.equal(fa, fb) and torch.equal(sa, sb) and torch.equal(ka, kb)
