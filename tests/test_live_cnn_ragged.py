"""Ragged pushes of live CNN streams (LiveCNN.push_ragged / kws_live_cnn_push_ragged*): every stream brings its own
number of samples, any number in [0, max_push], and only the logits of the windows a push completes come back,
compacted as LiveStreams.push_ragged lists them, while each convolution row of a stream is still computed once.

A push from sample count c to c' computes a stream's convolution rows (top(c), top(c')], top(c) = floor((c - W) / H) m
+ Hc - 3 with the floor not clamped at 0: a function of the counter alone, equal to the uniform push's rows for aligned
counts.  Checked here: the ring capacities for such sequences without a GPU, and on the GPU the logits bit for bit
against LiveStreams.push_ragged(samples, lengths, model), the route that runs the whole CNN per window.
"""
import ctypes

import numpy as np
import pytest
import torch

import honk2_b200
from honk2_b200 import LiveCNN, LiveStreams, NativeError
from honk2_b200.streaming import ragged_push_plan
from oracle import model_ref
from test_live_cnn import SHAPES, ap, ap_for, check_float64, cnn, cnn_for, dev, make_pcm, window_of  # noqa: F401
from test_live_cnn_rows import SHAPES as ROW_SHAPES
from test_live_ragged import gather_samples, ragged_lengths

gpu = pytest.mark.gpu
KWS_ERR_INVALID = 1


# ---- the row rule and the ring capacities, without a GPU ---------------------------------------

def top(c, W, H, Hc):
    """Last stream row of a convolution of Hc rows per window computed once a stream has seen c samples."""
    return (c - W) // H * (H // 160) + Hc - 3


def simulate(T, KH0, KH1, W, H, max_push, pushes):
    """Play a push sequence through the three rings a live CNN stream keeps (frame-table rows, fcap of them; pooled
    conv_0 rows, cap0; conv_1 rows, cap1) as live_cnn.cu schedules its jobs, and assert that every row a push reads is
    in its slot, written by that push or an earlier one and not overwritten since, and computed from rows that were.
    pushes: (n, uniform) pairs; a uniform push (n a multiple of H at a count that is a multiple of 160) takes the rows
    of the uniform push's jobs, which must be the row rule's."""
    P = max_push // 160
    m = H // 160
    H0 = T - KH0 + 1
    H1 = H0 - KH1 + 1
    fcap, cap0, cap1 = -(-(W + max_push) // 160), P + H0, P + H1
    frames, ring0, ring1 = {}, {}, {}

    def ok(ring, cap, r):
        return ring.get(r % cap) == (r, True)

    def store(ring, cap, rows):
        assert len({r % cap for r, _ in rows}) == len(rows), "a push writes two rows to one slot"
        for r, valid in rows:
            ring[r % cap] = (r, valid)

    c, windows = 0, 0
    for n, uniform in pushes:
        c2 = c + n
        new0 = range(top(c, W, H, H0) + 1, top(c2, W, H, H0) + 1)
        new1 = range(top(c, W, H, H1) + 1, top(c2, W, H, H1) + 1)
        if uniform:
            assert c % 160 == 0 and n % H == 0 and 0 < n <= max_push
            k0 = (c - W) // H + 1   # live_cnn.cu's lc_job: (k0 - 1) m + H - 2 + j, j < n / 160
            assert new0 == range((k0 - 1) * m + H0 - 2, (k0 - 1) * m + H0 - 2 + n // 160)
            assert new1 == range((k0 - 1) * m + H1 - 2, (k0 - 1) * m + H1 - 2 + n // 160)
        assert len(new0) == m * ((c2 - W) // H - (c - W) // H) <= m * -(-n // H) <= P
        # the front-end's new frame-table rows (row r covers samples [160 r - 240, +480): valid from row 2 on)
        store(frames, fcap, [(r, r >= 2) for r in range((c - 240) // 160 + 1, (c2 - 240) // 160 + 1)])
        # conv_0 stream rows read frames R .. R + KH0 - 1
        store(ring0, cap0, [(R, all(ok(frames, fcap, R + i) for i in range(KH0))) for R in new0])
        ks = range(max(0, (c - W) // H + 1), (c2 - W) // H + 1)   # the windows the push completes
        for k in ks:   # conv_0 window rows 0, 1, H0-2, H0-1 read the frames that are not the window's edge frames
            for r in (0, 1, H0 - 2, H0 - 1):
                for t in range(r, r + KH0):
                    if 2 <= t <= T - 3:
                        assert ok(frames, fcap, k * m + t), ("frame", c, n, k, t)
        # conv_1 stream rows read pooled rows R .. R + KH1 - 1
        store(ring1, cap1, [(R, all(ok(ring0, cap0, R + i) for i in range(KH1))) for R in new1])
        for k in ks:
            for r in (0, 1, H1 - 2, H1 - 1):   # conv_1 window rows read pooled stream rows 2 .. H0-3 of the window
                for t in range(r, r + KH1):
                    if 2 <= t <= H0 - 3:
                        assert ok(ring0, cap0, k * m + t), ("pooled", c, n, k, t)
            for oh in range(2, H1 - 2):          # the first Linear reads conv_1 stream rows 2 .. H1-3
                assert ok(ring1, cap1, k * m + oh), ("conv_1", c, n, k, oh)
        windows += len(ks)
        c = c2
    return windows


def ragged_sequence(rng, H, max_push, n_pushes, min_samples):
    """(n, uniform) pairs: specials (0, 1, 159, 161, H +- 1, max_push), uniform draws in [0, max_push], idle stretches
    and 1 .. 159-sample trickles followed by max_push bursts, and uniform pushes whenever the count is aligned; at least
    n_pushes of them and min_samples samples."""
    special = [x for x in (0, 1, 159, 161, H - 1, H + 1, max_push) if x <= max_push]
    out, c = [], 0
    while len(out) < n_pushes or c < min_samples:
        kind = rng.integers(0, 5)
        if kind == 0:
            run = [int(rng.choice(special))]
        elif kind == 1:
            run = [int(rng.integers(0, max_push + 1))]
        elif kind == 2:   # idle, then a burst
            run = [0] * int(rng.integers(5, 40)) + [max_push] * int(rng.integers(1, 4))
        elif kind == 3:   # a trickle of pushes that complete no window, then a burst
            run = [int(x) for x in rng.integers(1, 160, size=int(rng.integers(5, 60)))] + [max_push]
        else:
            run = [-1]
        for n in run:
            if n < 0:   # a uniform push, when the count allows it
                if c % 160:
                    continue
                out.append((H * int(rng.integers(1, max_push // H + 1)), True))
            else:
                out.append((n, False))
            c += out[-1][0]
    return out


@pytest.mark.parametrize("H", [160, 320, 480, 800])
@pytest.mark.parametrize("shape", list(ROW_SHAPES))
def test_ragged_ring_capacity_by_brute_force(H, shape):
    """cap0 = P + H0, cap1 = P + H1 and the front-end's fcap = ceil((W + max_push) / 160) hold for counts that are not
    multiples of 160 or of the shift, from a fresh stream (warm-up included) through many ring turns."""
    T, _, k0, k1, _ = ROW_SHAPES[shape]
    rng = np.random.default_rng(H + T + k0[0])
    for W in (160 * (T - 1), 160 * (T - 1) + 1, 160 * (T - 1) + 159):
        for max_push in (H, 4 * H, 10 * H):
            pushes = ragged_sequence(rng, H, max_push, 400, 4 * (W + max_push))   # the frame ring turns 3+ times
            assert simulate(T, k0[0], k1[0], W, H, max_push, pushes) >= 3 * (W + max_push) // H


def test_ragged_row_rule_during_warm_up():
    """A push that completes no window still computes rows: window 0 reads rows 2 .. Hc-3, which a stream fed 1 sample
    at a time computes before its first window completes.  (A row count clamped like the window count would not.)"""
    T, KH0, KH1 = 101, 20, 10
    H0 = T - KH0 + 1
    W, H = 16000, 160
    rows, c = set(), 0
    while c < W:
        rows.update(range(top(c, W, H, H0) + 1, top(c + 1, W, H, H0) + 1))
        c += 1
    assert set(range(2, H0 - 2)) <= rows
    assert simulate(T, KH0, KH1, W, H, 1600, [(1, False)] * (W + 5 * H)) == 6


def test_live_cnn_ragged_c_abi_argument_errors_without_gpu(native_lib):
    """Null state and null lengths return KWS_ERR_INVALID with a message; the workspace query on null returns 0."""
    lib = native_lib
    assert lib.kws_live_cnn_ragged_workspace_bytes(None) == 0
    assert b"live CNN state is null" in lib.kws_last_error()
    lengths = (ctypes.c_int32 * 2)(160, 160)
    for fn in (lib.kws_live_cnn_push_ragged, lib.kws_live_cnn_push_ragged_pcm16):
        for n in (lengths, None):
            assert fn(None, None, n, None, None, None, 4, None, None, 0, None) == KWS_ERR_INVALID
            assert b"live CNN state is null" in lib.kws_last_error()


# ---- on the GPU -----------------------------------------------------------------------------------

def n_pushes_for(H, max_push, seconds):
    """Pushes of ragged_lengths after which a stream of the special-length pattern has seen `seconds` of audio on
    average."""
    special = sorted({0, 1, 159, 160, 161, H - 1, H, H + 1, 1024, max_push})
    return int(np.ceil(seconds * 16000 / np.mean([x for x in special if x <= max_push]))) + 4


def windows_of(wav, s_idx, k_idx, W, H):
    dev = wav.device
    return wav.unfold(1, W, H)[torch.from_numpy(s_idx).to(dev), torch.from_numpy(k_idx).to(dev)]


RUNS = ([pytest.param("zoo", W, S, H, id=f"zoo-w{W}-{S}-{H}")
         for W in (16000, 16001) for S in (1, 3, 149) for H in (160, 480, 800)] +
        [pytest.param(shape, window_of(SHAPES[shape]) + dw, S, H, id=f"{shape}-w{dw}-{S}-{H}")
         for shape in SHAPES if shape != "zoo" for dw in (0, 1) for S in (1, 3, 149) for H in (160, 480, 800)])


@gpu
@pytest.mark.parametrize("shape,W,S,H", RUNS)
def test_ragged_logits_bit_identical_to_live_streams_with_model(dev, ap_for, cnn_for, shape, W, S, H):
    """Logits == LiveStreams.push_ragged(samples, lengths, model) bit for bit, the ids == ragged_push_plan, int16 pushes
    == float pushes of s/32768, and a sample of windows against float64 (oracle.model_ref)."""
    row = SHAPES[shape]
    T, F = row.T, row.F
    cnn, ap = cnn_for(shape), ap_for(F)
    max_push = 10 * H
    lengths = ragged_lengths(S, n_pushes_for(H, max_push, seconds=6.0), H, max_push, seed=S * 7 + W + H + T)
    totals = lengths.sum(0)
    assert totals.max() >= 4 * 16000
    pcm = torch.from_numpy(make_pcm(S, int(totals.max()), seed=S + H + T)).to(dev)
    wav = pcm.float() / 32768.0
    flat, flat16 = wav.reshape(-1), pcm.reshape(-1)
    lc = LiveCNN(cnn, S, W, H, max_push, audio_processor=ap, device=dev)
    lc16 = LiveCNN(cnn, S, W, H, max_push, audio_processor=ap, device=dev)
    ls = LiveStreams(ap, S, W, H, max_push, device=dev)
    sd64 = {k: v.double() for k, v in cnn.state_dict().items() if v.is_floating_point()}
    cfg = dict(cnn.config, n_labels=cnn.n_labels)
    seen = np.zeros(S, dtype=np.int64)
    n_win, n_f64, worst64 = 0, 0, 0.0
    with torch.no_grad():
        for i, n in enumerate(lengths):
            x = gather_samples(flat, wav.shape[1], seen, n)
            y, si, wi = lc.push_ragged(x, n)
            y16, si16, wi16 = lc16.push_ragged(gather_samples(flat16, wav.shape[1], seen, n), n)
            ref, rsi, rwi = ls.push_ragged(x, n, cnn)
            plan = ragged_push_plan(seen, n, W, H)
            assert torch.equal(si, torch.from_numpy(plan.stream_ids)) and torch.equal(wi, torch.from_numpy(plan.window_ids))
            assert torch.equal(si, rsi) and torch.equal(wi, rwi) and torch.equal(si, si16) and torch.equal(wi, wi16)
            assert y.shape == (len(plan.stream_ids), row.labels)
            assert torch.equal(y, ref), f"push {i}: largest difference {float((y - ref).abs().max())}"
            assert torch.equal(y, y16), "int16 pushes equal float pushes of s/32768"
            if i % 5 == 2 and len(si) and n_f64 < (64 if shape == "zoo" else 16):
                sel = np.arange(len(si))[:8]
                feats = ap.compute_mfccs_batch(windows_of(wav, si.numpy()[sel], wi.numpy()[sel], W, H))
                r64 = model_ref.cnn_forward(sd64, cfg, feats.double())
                worst64 = max(worst64, check_float64(y[torch.from_numpy(sel).to(dev)], r64))
                n_f64 += len(sel)
            n_win += len(si)
            seen += n
    assert torch.equal(lc.samples_seen, torch.from_numpy(totals))
    print(f"{shape} W={W} S={S} H={H}: {n_win} windows bit-identical to LiveStreams.push_ragged + model (largest "
          f"difference 0), {n_f64} against float64, worst {worst64:.3e}")
    assert n_f64 > 0


@gpu
@pytest.mark.parametrize("H", [160, 480])
def test_ragged_warm_up_pushes_that_complete_no_window(dev, ap, cnn, H):
    """Fresh streams fed 1 .. 159 samples at a time: most pushes complete no window (M = 0, empty tensors) but still
    compute the rows window 0 reads; the first windows are bit-identical to the route that runs the whole CNN."""
    S, W, max_push = 5, 16000, 10 * H
    rng = np.random.default_rng(H)
    lengths = rng.integers(1, 160, size=(260, S))
    lengths[:, 3] = rng.integers(0, 3, size=260)   # a stream that stays in its warm-up
    totals = lengths.sum(0)
    assert totals[[0, 1, 2, 4]].min() >= W + 4 * H
    pcm = torch.from_numpy(make_pcm(S, int(totals.max()), seed=5)).to(dev)
    wav = pcm.float() / 32768.0
    lc = LiveCNN(cnn, S, W, H, max_push, device=dev)
    ls = LiveStreams(ap, S, W, H, max_push, device=dev)
    seen = np.zeros(S, dtype=np.int64)
    empty, got = 0, 0
    with torch.no_grad():
        for n in lengths:
            x = gather_samples(wav.reshape(-1), wav.shape[1], seen, n)
            y, si, wi = lc.push_ragged(x, n)
            ref, _, _ = ls.push_ragged(x, n, cnn)
            if len(si) == 0:
                empty += 1
                assert y.shape == (0, cnn.n_labels) and si.shape == wi.shape == (0,)
            assert torch.equal(y, ref)
            got += len(si)
            seen += n
    assert empty > 200 and got >= 4 * 4
    assert torch.equal(lc.samples_seen, torch.from_numpy(totals))


@gpu
def test_ragged_window_depends_on_its_audio_only(dev, ap, cnn):
    """Window (s, k)'s logits are bit-identical across two ragged cuts, uniform pushes, and different sets of streams
    pushing alongside it."""
    W, H, max_push = 16000, 160, 1600
    S, L = 5, 3 * 16000
    wav = torch.from_numpy(make_pcm(S, L, seed=21)).to(dev).float() / 32768.0

    def ragged(streams, seed):
        lc = LiveCNN(cnn, streams.shape[0], W, H, max_push, device=dev)
        lengths = np.random.default_rng(seed).integers(0, max_push + 1, size=(200, streams.shape[0]))
        out, seen = {}, np.zeros(streams.shape[0], dtype=np.int64)
        for n in lengths:
            n = np.minimum(n, L - seen)
            y, si, wi = lc.push_ragged(gather_samples(streams.reshape(-1), L, seen, n), n)
            for j, (s, k) in enumerate(zip(si.tolist(), wi.tolist())):
                out[s, k] = y[j]
            seen += n
        assert (seen == L).all()
        return out

    def uniform(streams):
        lc = LiveCNN(cnn, streams.shape[0], W, H, max_push, device=dev)
        out = {}
        for c in range(0, L, max_push):
            y, v = lc.push(streams[:, c:c + max_push])
            for s in range(streams.shape[0]):
                for j in np.flatnonzero(v[s].numpy()):
                    out[s, (c - W) // H + 1 + int(j)] = y[s, j]   # slot j's window
        return out

    with torch.no_grad():
        a, b, u = ragged(wav, 1), ragged(wav, 2), uniform(wav)
        alone = ragged(wav[2:3], 3)
        pair = ragged(wav[[4, 2]], 4)
    n_all = (L - W) // H + 1
    assert set(a) == set(b) == set(u) == {(s, k) for s in range(S) for k in range(n_all)}
    for key in a:
        assert torch.equal(a[key], b[key]) and torch.equal(a[key], u[key]), key
    for k in range(n_all):
        assert torch.equal(alone[0, k], a[2, k]) and torch.equal(pair[1, k], a[2, k]) and torch.equal(pair[0, k], a[4, k])


@gpu
def test_ragged_and_uniform_pushes_mix_and_refusals_change_nothing(dev, ap, cnn):
    """While every count is aligned, uniform and ragged pushes alternate on one state with the logits of a state fed
    ragged pushes only.  Once a count is unaligned, push raises ValueError and changes nothing.  Refused ragged pushes
    change nothing either: the state continues exactly like one that never saw them."""
    S, W, H, max_push = 3, 16000, 320, 3200
    L = 5 * 16000
    wav = torch.from_numpy(make_pcm(S, L, seed=8)).to(dev).float() / 32768.0
    flat = wav.reshape(-1)
    mixed = LiveCNN(cnn, S, W, H, max_push, device=dev)
    ragged = LiveCNN(cnn, S, W, H, max_push, device=dev)
    seen = np.zeros(S, dtype=np.int64)

    def both(n, uniform):
        nonlocal seen
        x = gather_samples(flat, L, seen, n)
        yr, si, wi = ragged.push_ragged(x, n)
        if uniform:
            y, v = mixed.push(x.view(S, -1))
            assert torch.equal(y[v.to(dev)], yr), "uniform push differs from the ragged push of the same audio"
        else:
            y, si2, wi2 = mixed.push_ragged(x, n)
            assert torch.equal(y, yr) and torch.equal(si, si2) and torch.equal(wi, wi2)
        seen += n

    with torch.no_grad():
        for i in range(24):
            both(np.full(S, H * (1 + i % 10)), i % 2 == 0)
        # unalign stream 1: push is refused and changes nothing
        both(np.array([320, 161, 0]), False)
        before = mixed.samples_seen
        with pytest.raises(ValueError, match="multiple of the 160-sample hop"):
            mixed.push(wav[:, :H])
        assert torch.equal(mixed.samples_seen, before)
        # refused ragged pushes
        x = flat[:4000]
        for lengths in ([-1, 0, 0], [max_push + 1, 0, 0], [0, 0], [0, 0, 0, 0]):
            with pytest.raises(ValueError):
                mixed.push_ragged(x[:max(0, sum(lengths))], lengths)
        with pytest.raises(ValueError, match="add up to"):
            mixed.push_ragged(x[:100], [50, 49, 0])
        with pytest.raises(ValueError):
            mixed.push_ragged(x[:10].double(), [10, 0, 0])
        with pytest.raises(ValueError):
            mixed.push_ragged(x[:10], torch.tensor([10, 0, 0], device=dev))
        with pytest.raises(NativeError):
            mixed.push_ragged(x[:10].cpu(), [10, 0, 0])
        with pytest.raises(ValueError, match="out must be"):   # needs ceil(1000 / 320) = 4 rows
            mixed.push_ragged(x[:1000], [1000, 0, 0], out=torch.empty((3, cnn.n_labels), device=dev))
        # the C ABI's own checks: capacity, workspace, null logits
        lib = honk2_b200._native.load()
        handle = mixed._state()
        need = lib.kws_live_cnn_ragged_workspace_bytes(handle)
        ws = torch.empty(need, dtype=torch.uint8, device=dev)
        logits = torch.empty((20, cnn.n_labels), device=dev)

        def c_push(lengths, capacity=20, ws_bytes=need, out=logits):
            n32 = (ctypes.c_int32 * S)(*lengths)
            return lib.kws_live_cnn_push_ragged(handle, ctypes.c_void_p(x.data_ptr()), n32,
                                                ctypes.c_void_p(out.data_ptr()) if out is not None else None, None,
                                                None, capacity, None, ctypes.c_void_p(ws.data_ptr()), ws_bytes, None)
        for args, msg in ((([-1, 0, 0],), b"max_push"), (([1000, 321, 0], 5), b"capacity"),
                          (([10, 0, 0], 20, need - 1), b"workspace"), (([10, 0, 0], 20, need, None), b"logits is null")):
            assert c_push(*args) == KWS_ERR_INVALID
            assert msg in lib.kws_last_error(), lib.kws_last_error()
        assert torch.equal(mixed.samples_seen, before)
        # both states continue alike, ragged pushes realign the counts, and uniform pushes resume
        both(np.array([0, 159, 0]), False)
        for i in range(12):
            both(np.full(S, H * (1 + i % 3)), i % 2 == 1)
    assert seen.max() <= L


@gpu
def test_ragged_reset(dev, ap, cnn):
    """Streams reset mid-run equal fresh streams fed the same audio; the others continue unaffected."""
    S, W, H, max_push = 4, 16000, 160, 1600
    L = 4 * 16000
    wav = torch.from_numpy(make_pcm(S, L, seed=31)).to(dev).float() / 32768.0
    lengths = ragged_lengths(S, 120, H, max_push, seed=31)
    a = LiveCNN(cnn, S, W, H, max_push, device=dev)
    ref = LiveCNN(cnn, S, W, H, max_push, device=dev)
    fresh = LiveCNN(cnn, S, W, H, max_push, device=dev)
    seen, seen_f = np.zeros(S, dtype=np.int64), np.zeros(S, dtype=np.int64)
    reset_at, checked = 40, 0
    with torch.no_grad():
        for i, n in enumerate(lengths):
            n = np.minimum(n, L - np.maximum(seen, seen_f))
            if i == reset_at:
                a.reset([1, 3])
                seen_a = seen.copy()
                seen_a[[1, 3]] = 0
            if i < reset_at:
                x = gather_samples(wav.reshape(-1), L, seen, n)
                a.push_ragged(x, n)
                ref.push_ragged(x, n)
                seen += n
                continue
            # after the reset: a's streams 1 and 3 restart at sample 0, like fresh's
            x_a = gather_samples(wav.reshape(-1), L, seen_a, n)
            y, si, wi = a.push_ragged(x_a, n)
            yr, sr, wr = ref.push_ragged(gather_samples(wav.reshape(-1), L, seen, n), n)
            yf, sf, wf = fresh.push_ragged(gather_samples(wav.reshape(-1), L, seen_f, n), n)
            for s in range(S):
                mine = (si == s).to(dev)
                other, other_s = ((yf, sf), (yr, sr))[s in (0, 2)]
                sel = (other_s == s).to(dev)
                assert torch.equal(y[mine], other[sel]), (i, s)
                checked += int(mine.sum())
            seen_a += n
            seen += n
            seen_f += n
    assert checked > 50


@gpu
@pytest.mark.parametrize("S,H", [(6001, 160), (149, 480), (3, 800)])
def test_ragged_device_ids_and_count(dev, ap, cnn, S, H):
    """Through the C ABI: n_windows, win_stream and win_index equal the host plan and the logits LiveCNN.push_ragged's
    on a second state.  S = 6001 spans several CTAs of both scans."""
    lib = honk2_b200._native.load()
    W, max_push = 16000, 10 * H
    lengths = ragged_lengths(S, 12 if S > 1000 else 48, H, max_push, seed=S + H)
    totals = lengths.sum(0)
    wav = torch.from_numpy(make_pcm(S, int(totals.max()), seed=S)).to(dev).float() / 32768.0
    flat = wav.reshape(-1)
    a = LiveCNN(cnn, S, W, H, max_push, device=dev)
    b = LiveCNN(cnn, S, W, H, max_push, device=dev)
    handle = b._state()
    ws = torch.empty(lib.kws_live_cnn_ragged_workspace_bytes(handle), dtype=torch.uint8, device=dev)
    cap = S * (max_push // H)
    logits = torch.empty((cap, cnn.n_labels), device=dev)
    ids = torch.empty((2, cap), dtype=torch.int64, device=dev)
    m = torch.full((1,), -1, dtype=torch.int64, device=dev)
    seen = np.zeros(S, dtype=np.int64)
    total = 0
    with torch.no_grad():
        for n in lengths:
            x = gather_samples(flat, wav.shape[1], seen, n)
            ya, sa, ka = a.push_ragged(x, n)
            n32 = np.ascontiguousarray(n, dtype=np.int32)
            assert lib.kws_live_cnn_push_ragged(
                handle, ctypes.c_void_p(x.data_ptr()), ctypes.c_void_p(n32.ctypes.data),
                ctypes.c_void_p(logits.data_ptr()), ctypes.c_void_p(ids[0].data_ptr()),
                ctypes.c_void_p(ids[1].data_ptr()), cap, ctypes.c_void_p(m.data_ptr()), ctypes.c_void_p(ws.data_ptr()),
                ws.numel(), ctypes.c_void_p(torch.cuda.current_stream(dev).cuda_stream)) == 0
            M = len(sa)
            assert int(m.item()) == M
            assert torch.equal(ids[0, :M].cpu(), sa) and torch.equal(ids[1, :M].cpu(), ka)
            assert torch.equal(logits[:M], ya)
            total += M
            seen += n
    assert total > 0


@gpu
def test_ragged_sizes_and_no_allocation_after_the_first_push(dev, ap, cnn):
    """The workspace LiveCNN allocates is kws_live_cnn_ragged_workspace_bytes: the front-end's ragged workspace plus two
    i64[S + 1] plans and a scan's scratch.  After the first, ragged pushes given `out` take no device memory."""
    lib = honk2_b200._native.load()
    S, W, H, max_push = 1024, 16000, 160, 1600
    lc = LiveCNN(cnn, S, W, H, max_push, device=dev)
    need = lib.kws_live_cnn_ragged_workspace_bytes(lc._state())
    ls = LiveStreams(ap, S, W, H, max_push, device=dev)   # (kept alive while its handle is used)
    fe = lib.kws_live_ragged_workspace_bytes(ls._state())

    def up(x):
        return -(-x // 256) * 256
    plan = up((S + 1) * 8)
    temp = fe - (up(S * 12) + 2 * plan)   # the front-end's: offsets and lengths, counts, plan, then the scan's scratch
    assert temp > 0 and need == up(fe) + 2 * plan + temp
    out = torch.empty((S * 10, cnn.n_labels), device=dev)
    rng = np.random.default_rng(0)
    wav = torch.zeros(S * max_push, device=dev)
    with torch.no_grad():
        n = rng.integers(0, max_push + 1, size=S)
        lc.push_ragged(wav[:int(n.sum())], n, out=out)
        assert lc._ragged_ws.numel() == need
        torch.cuda.synchronize()
        before = torch.cuda.memory_allocated(dev), torch.cuda.mem_get_info(dev)[0]
        for _ in range(5):
            n = rng.integers(0, max_push + 1, size=S)
            lc.push_ragged(wav[:int(n.sum())], n, out=out)
        torch.cuda.synchronize()
        after = torch.cuda.memory_allocated(dev), torch.cuda.mem_get_info(dev)[0]
    assert after[0] == before[0] and after[1] == before[1]
