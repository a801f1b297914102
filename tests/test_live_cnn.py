"""Live CNN streams (LiveCNN / kws_live_cnn_*): a push returns the logits of the windows it completes, computing each
convolution row of a stream once and per window only the rows next to its reflect-padded edges.

The logits are compared with float64 (oracle.model_ref on the materialised windows' features, at the bf16 tolerance of
test_tc_shapes.py) and with LiveStreams.push(chunk, model), the batch bf16 path on the same windows, bit for bit: the
live row kernels keep cnn_tc_fused_kernel's MMA shape (K = 16 per product) and K order, and the first Linear its
split-K slices.  A window's logits are a function of its audio alone: bit-identical however the audio was cut into
pushes and whichever streams share the push.

Every CNN shape the live row kernels take runs here, each with a front-end of n_mels = frequency and a window of
160 * (time - 1) samples: the accepted shapes of test_tc_shapes.CNN_SHAPES (odd conv_0 height, conv_1 1 to 5 taps wide,
H1 from 32 to the batch plan's 80, zero to two Linear layers after the first) and one at the kernels' limit (pooled
width 16, conv_1 9 taps wide, an odd n_mels).  Shapes the batch path takes but the row kernels do not are refused.
"""
import ctypes
import zlib

import numpy as np
import pytest
import torch

import honk2_b200
from honk2_b200 import AudioProcessor, LiveCNN, LiveStreams, NativeError
from honk2_b200 import synth
from honk2_b200.model import CNN
from oracle import model_ref
from test_tc_shapes import CNN_ROWS, CnnRow, _cnn_cfg, _kernel_path

gpu = pytest.mark.gpu
BF16_TOL = 3e-2
KWS_ERR_INVALID, KWS_ERR_UNSUPPORTED = 1, 3
FUSED = "cnn_tc_fused_kernel"

_STACK = {"lin_0": 32, "dnn_0": 128}
# shape id -> CnnRow; "zoo" is cnn-trad-fpool3 as honk2_b200.build_model makes it
SHAPES = {r.id: r for r in [CNN_ROWS[i] for i in ("zoo", "t60_h1_32", "t108_h1_80", "conv0_h21", "conv0_w5_conv1_w5",
                                                  "f32_conv1_w1", "lin0_dnn0_dnn1", "lin1_only", "dnn0_512")] +
          [CnnRow("t60_f57_conv1_w9", 60, 57, (20, 8), (10, 9), _STACK, 12, True)]}   # WP = 16, KW1 = 9
# the batch path takes these, the live row kernels do not
REFUSED = {r.id: r for r in [CnnRow("f60_conv1_w10", 60, 60, (20, 8), (10, 10), _STACK, 12, True),   # WP = 17
                             CnnRow("t31_h1_3", 31, 40, (20, 8), (10, 4), _STACK, 12, True)]}       # H1 = 3


def window_of(row):
    return 160 * (row.T - 1)


@pytest.fixture(scope="module")
def dev(native_lib):
    assert torch.cuda.is_available(), "these tests need the B200"
    return torch.device("cuda", 0)


@pytest.fixture(scope="module")
def ap_for(dev):
    cache = {}

    def get(n_mels):
        if n_mels not in cache:
            cache[n_mels] = AudioProcessor(n_mels=n_mels)
        return cache[n_mels]
    return get


@pytest.fixture(scope="module")
def ap(ap_for):
    return ap_for(40)


@pytest.fixture(scope="module")
def cnn_for(dev):
    """shape id -> bf16 CNN on the device with seeded, hardened weights (logits spread over the labels)."""
    cache = {}

    def get(shape):
        if shape not in cache:
            if shape == "zoo":
                m = honk2_b200.build_model("cnn-trad-fpool3", precision="bf16").to(dev)
            else:
                torch.manual_seed(zlib.crc32(shape.encode()))
                m = CNN(dict(_cnn_cfg({**SHAPES, **REFUSED}[shape]), precision="bf16")).to(dev)
            m.eval()
            synth.harden_(m.state_dict())   # (in place)
            cache[shape] = m
        return cache[shape]
    return get


@pytest.fixture(scope="module")
def cnn(cnn_for):
    return cnn_for("zoo")


def make_pcm(S, L, seed):
    """[S, L] int16 PCM of speech-like audio with a gain per stream and stretches of zeros in every other stream."""
    rng = np.random.default_rng(seed)
    x = synth.speechlike(S, N=L, seed=seed) * (10.0 ** rng.uniform(-1.5, 0.0, size=(S, 1))).astype(np.float32)
    for s in range(0, S, 2):
        a = int(rng.integers(0, max(1, L - 6000)))
        x[s, a:a + int(rng.integers(800, 6000))] = 0.0
    return np.clip(np.round(x * 32768.0), -32768, 32767).astype(np.int16)


def pushes(kind, H, max_push, total):
    seq = {"H": [H], "max": [max_push], "varying": [H, 7 * H, max_push, 2 * H, 3 * H, 5 * H]}[kind]
    out, n, i = [], 0, 0
    while n < total:
        out.append(seq[i % len(seq)])
        n += out[-1]
        i += 1
    return out


def scale_err(y, ref):
    """max over rows of |y - ref|_inf / max(|ref|_inf of the row, 1e-3)."""
    den = ref.abs().amax(dim=-1, keepdim=True).clamp_min(1e-3)
    return float(((y - ref).abs() / den).max()) if y.numel() else 0.0


def check_float64(y, ref):
    """bf16 logits against float64 at BF16_TOL; the argmax agrees where the reference's top-2 margin exceeds twice the
    bound.  Returns the error."""
    y, ref = y.double().cpu().numpy(), ref.cpu().numpy()
    den = np.maximum(np.abs(ref).max(axis=1, keepdims=True), 1e-3)
    err = float((np.abs(y - ref) / den).max())
    assert err <= BF16_TOL
    bound = BF16_TOL * den[:, 0]
    top2 = np.sort(ref, axis=1)[:, -2:]
    decided = (top2[:, 1] - top2[:, 0]) > 2 * bound
    assert np.array_equal(y.argmax(1)[decided], ref.argmax(1)[decided])
    return err


# (shape, window, S, H, push kind).  cnn-trad-fpool3 at 16000 keeps the ids it always had; 16001 and 16159 are windows
# that are not a multiple of the hop with the same 101 frames.
LOGIT_RUNS = (
    [pytest.param("zoo", 16000, S, H, kind, id=f"{S}-{H}-{kind}")
     for S, H, kind in [(1, 160, "H"), (3, 160, "varying"), (3, 480, "max"), (149, 160, "H"), (149, 160, "max"),
                        (149, 800, "varying")]] +
    [pytest.param("zoo", W, S, H, kind, id=f"zoo_w{W}-{S}-{H}-{kind}")
     for W in (16001, 16159) for S, H, kind in [(3, 160, "varying"), (3, 480, "H")]] +
    [pytest.param(shape, window_of(SHAPES[shape]), S, H, kind, id=f"{shape}-{S}-{H}-{kind}")
     for shape in SHAPES if shape != "zoo"
     for S, H, kind in [(3, 160, "H"), (3, 480, "max"), (3, 800, "varying"), (149, 160, "varying")]])


@gpu
@pytest.mark.parametrize("shape,W,S,H,kind", LOGIT_RUNS)
def test_live_cnn_logits(dev, ap_for, cnn_for, shape, W, S, H, kind):
    """Against float64 on the materialised windows, bit-identical to LiveStreams.push(chunk, model), int16 == float pushes;
    warm-up slots zero and masked.  Four seconds of audio: both rows rings wrap several times."""
    row = SHAPES[shape]
    T, F = row.T, row.F
    assert 1 + W // 160 == T
    cnn, ap = cnn_for(shape), ap_for(F)
    assert _kernel_path(cnn, dev, T, F) == FUSED
    max_push = 10 * H
    sizes = pushes(kind, H, max_push, 4 * 16000 + 7 * H)
    pcm = torch.from_numpy(make_pcm(S, sum(sizes), seed=S + H)).to(dev)
    wav = pcm.float() / 32768.0
    lc = LiveCNN(cnn, S, W, H, max_push, audio_processor=ap, device=dev)
    lc16 = LiveCNN(cnn, S, W, H, max_push, audio_processor=ap, device=dev)
    ls = LiveStreams(ap, S, W, H, max_push, device=dev)
    sd64 = {k: v.double() for k, v in cnn.state_dict().items() if v.is_floating_point()}
    cfg = dict(cnn.config, n_labels=cnn.n_labels)
    f64_cap = None if shape == "zoo" else 48    # (float64 windows per run: the CPU reference is the slow part)
    worst, worst64, c, n_f64 = 0.0, 0.0, 0, 0
    with torch.no_grad():
        for i, n in enumerate(sizes):
            y, v = lc.push(wav[:, c:c + n])
            y16, v16 = lc16.push(pcm[:, c:c + n])
            f, v2 = ls.push(wav[:, c:c + n])
            K = n // H
            assert y.shape == (S, K, row.labels) and torch.equal(v, v2) and torch.equal(v, v16)
            assert torch.equal(y, y16), "int16 pushes equal float pushes of s/32768"
            vd = v.to(dev)
            assert torch.count_nonzero(y[~vd]).item() == 0
            ref = cnn(f.view(S * K, T, F)).view(S, K, -1)
            worst = max(worst, scale_err(y[vd], ref[vd]))
            assert torch.equal(y[vd], ref[vd]), "LiveCNN differs from LiveStreams.push(chunk, model)"
            if i % 7 == 3 and bool(v.any()) and (f64_cap is None or n_f64 < f64_cap):
                sel = torch.nonzero(vd.view(-1)).view(-1)[:64 if f64_cap is None else 16]
                r64 = model_ref.cnn_forward(sd64, cfg, f.view(S * K, T, F)[sel].double())
                worst64 = max(worst64, check_float64(y.view(S * K, -1)[sel], r64))
                n_f64 += sel.numel()
            c += n
    print(f"{shape} W={W} S={S} H={H} {kind}: max |LiveCNN - LiveStreams+model| = {worst:.3e} of the logit scale, "
          f"{n_f64} windows against float64, worst {worst64:.3e}")
    assert n_f64 > 0


@gpu
def test_live_cnn_window_depends_on_its_audio_only(dev, ap, cnn):
    """A window's logits do not depend on how its audio was cut into pushes or on the other streams of the push; two
    identical runs are bit-identical."""
    W, H, max_push = 16000, 160, 1600
    L = 3 * 16000
    pcm = torch.from_numpy(make_pcm(5, L, seed=11)).to(dev)
    wav = pcm.float() / 32768.0

    def run(S, streams, sizes):
        lc = LiveCNN(cnn, S, W, H, max_push, audio_processor=ap, device=dev)
        out, c = [], 0
        for n in sizes:
            y, v = lc.push(streams[:, c:c + n])
            out.append(y[:, v[0].to(dev)])   # (every stream has seen as many samples: one mask row for all)
            c += n
        return torch.cat(out, dim=1)

    a = run(5, wav, pushes("H", H, max_push, L))
    b = run(5, wav, pushes("varying", H, max_push, L))
    n = min(a.shape[1], b.shape[1])
    assert n > 150
    assert torch.equal(a[:, :n], b[:, :n]), "the cut into pushes changed a window's logits"
    alone = run(1, wav[2:3], pushes("H", H, max_push, L))
    assert torch.equal(alone[0], a[2]), "the other streams of a push changed a window's logits"
    assert torch.equal(run(5, wav, pushes("H", H, max_push, L)), a), "two identical runs differ"


@gpu
def test_live_cnn_reset(dev, ap, cnn):
    """A reset stream's windows equal a fresh stream's; the other streams are unaffected."""
    W, H, max_push = 16000, 320, 3200
    pcm = torch.from_numpy(make_pcm(3, 4 * 16000, seed=3)).to(dev)
    wav = pcm.float() / 32768.0
    a = LiveCNN(cnn, 3, W, H, max_push, audio_processor=ap, device=dev)
    ref = LiveCNN(cnn, 3, W, H, max_push, audio_processor=ap, device=dev)
    c = 0
    for n in (3200, 3200, 1600, 3200, 3200, 320):
        a.push(wav[:, c:c + n])
        ref.push(wav[:, c:c + n])
        c += n
    a.reset([1])
    assert a.samples_seen.tolist() == [c, 0, c]
    fresh = LiveCNN(cnn, 3, W, H, max_push, audio_processor=ap, device=dev)
    d = 0
    for n in (3200, 3200, 3200, 3200, 3200, 3200, 960):
        y, v = a.push(torch.stack([wav[0, c:c + n], wav[1, d:d + n], wav[2, c:c + n]]))
        yr, vr = ref.push(wav[:, c:c + n])
        yf, vf = fresh.push(wav[:, d:d + n])
        assert torch.equal(y[0], yr[0]) and torch.equal(y[2], yr[2]) and torch.equal(v[0], vr[0])
        assert torch.equal(y[1], yf[1]) and torch.equal(v[1], vf[1])
        c, d = c + n, d + n
    assert bool(v[1].all())


@gpu
def test_live_cnn_refusals(dev, ap, cnn):
    lib = honk2_b200._native.load()
    fe = ap._frontend(dev)
    with pytest.raises(ValueError, match="CNN"):
        LiveCNN(honk2_b200.build_model("res8", precision="bf16").to(dev), 2, device=dev)
    for prec in ("fp32", "bf16x3"):
        with pytest.raises(ValueError, match="bf16"):
            LiveCNN(honk2_b200.build_model("cnn-trad-fpool3", precision=prec).to(dev), 2, device=dev)
    with pytest.raises(NativeError, match="kws_live_cnn_create"):
        LiveCNN(honk2_b200.build_model("cnn-one-fstride4", precision="bf16").to(dev), 2, audio_processor=ap,
                device=dev)
    with pytest.raises(NativeError, match="frames"):
        LiveCNN(cnn, 2, 8000, 160, audio_processor=ap, device=dev)
    for W, H, mp in ((16000, 100, 1000), (16000, 320, 1000)):
        with pytest.raises(NativeError, match="kws_live_cnn_create"):
            LiveCNN(cnn, 2, W, H, mp, audio_processor=ap, device=dev)
    # the C ABI: a ResNet and an unsupported CNN are KWS_ERR_UNSUPPORTED, a bad shift KWS_ERR_INVALID
    res = honk2_b200.build_model("res8", precision="bf16").to(dev)
    with torch.no_grad():
        res(torch.zeros(1, 101, 40, device=dev))
    out = ctypes.c_void_p()
    handle = res._native_state[dev.index]["handle"]
    assert lib.kws_live_cnn_create(handle, fe, 2, 16000, 160, 1600, ctypes.byref(out)) == KWS_ERR_UNSUPPORTED
    assert lib.kws_live_cnn_state_bytes(handle, fe, 2, 16000, 160, 1600) == 0
    _, st = cnn._state(dev)
    assert lib.kws_live_cnn_create(st["handle"], fe, 2, 16000, 100, 1000, ctypes.byref(out)) == KWS_ERR_INVALID
    assert lib.kws_live_cnn_create(st["handle"], fe, 2, 8000, 160, 1600, ctypes.byref(out)) == KWS_ERR_UNSUPPORTED
    lc = LiveCNN(cnn, 2, 16000, 320, 3200, audio_processor=ap, device=dev)
    with pytest.raises(NativeError, match="multiple of the shift"):
        lc.push(torch.zeros(2, 480, device=dev))
    with pytest.raises(NativeError, match="multiple of the shift"):
        lc.push(torch.zeros(2, 3520, device=dev))
    with pytest.raises(ValueError):
        lc.push(torch.zeros(3, 320, device=dev))
    assert torch.equal(lc.samples_seen, torch.zeros(2, dtype=torch.int64))


@gpu
@pytest.mark.parametrize("shape", list(REFUSED))
def test_live_cnn_refuses_maps_outside_the_row_kernels(dev, ap_for, cnn_for, shape):
    """A pooled width of 17 or H1 = 3: the batch path runs the CNN on the tensor cores, the live state is refused with
    KWS_ERR_UNSUPPORTED and its size query returns 0."""
    row = REFUSED[shape]
    W = window_of(row)
    cnn, ap = cnn_for(shape), ap_for(row.F)
    assert _kernel_path(cnn, dev, row.T, row.F) == FUSED
    with torch.no_grad():
        assert torch.isfinite(cnn(torch.randn(4, row.T, row.F, device=dev) - 8.0)).all()
    with pytest.raises(NativeError, match="live row kernels"):
        LiveCNN(cnn, 2, W, 160, 1600, audio_processor=ap, device=dev)
    lib = honk2_b200._native.load()
    _, st = cnn._state(dev)
    fe = ap._frontend(dev)
    out = ctypes.c_void_p()
    assert lib.kws_live_cnn_create(st["handle"], fe, 2, W, 160, 1600, ctypes.byref(out)) == KWS_ERR_UNSUPPORTED
    assert out.value is None
    assert lib.kws_live_cnn_state_bytes(st["handle"], fe, 2, W, 160, 1600) == 0


@gpu
def test_live_cnn_state_bytes_match_allocation(dev, ap, cnn):
    """state_bytes() == what create takes from the device (free-memory delta; cudaMalloc rounds to 2 MiB per
    allocation, and the state makes three: the live front-end, its copy of the packed weights, its rows) and destroy
    gives back."""
    cnn._state(dev)
    torch.cuda.synchronize()
    free0 = torch.cuda.mem_get_info(dev)[0]
    lc = LiveCNN(cnn, 4096, 16000, 160, 1600, audio_processor=ap, device=dev)
    free1 = torch.cuda.mem_get_info(dev)[0]
    need = lc.state_bytes()
    live = honk2_b200._native.load().kws_live_state_bytes(ap._frontend(dev), 4096, 16000, 160, 1600)
    S, K, P = 4096, 10, 10
    own = S * K * 4 * 40 * 4 + S * (P + 82) * 11 * 128 + S * K * 4 * 11 * 128 + S * (P + 73) * 1024 + \
        S * K * 4 * 1024 + 8 * S * K * 32 * 4
    assert 0 < need - live - own < 4 << 20, (need, live, own)   # the rest: the packed weights (2.8 MB)
    assert 0 <= (free0 - free1) - need < 8 << 20, (free0 - free1, need)
    del lc
    free2 = torch.cuda.mem_get_info(dev)[0]
    assert abs(free2 - free0) < 8 << 20


@gpu
def test_smaller_cnn_plans_and_states_leave_larger_ones_working(dev, ap_for, cnn_for):
    """CNN plans and live states size their kernels' shared memory when they are created.  Creating smaller ones
    afterwards must not take that memory from the larger ones: their launches keep running, with the same logits."""
    def fresh(shape):
        torch.manual_seed(zlib.crc32(shape.encode()))
        m = CNN(dict(_cnn_cfg({**SHAPES, **REFUSED}[shape]), precision="bf16")).to(dev)
        m.eval()
        synth.harden_(m.state_dict())
        return m

    x = torch.randn(8, 101, 40, device=dev) - 8.0
    with torch.no_grad():
        big = fresh("zoo")
        want = big(x).clone()
        big_lc = {s: LiveCNN(cnn_for(s), 2, window_of(SHAPES[s]), 160, 1600, audio_processor=ap_for(SHAPES[s].F),
                             device=dev) for s in ("t60_f57_conv1_w9", "conv0_h21")}   # the widest conv_1, the tallest conv_0
        fresh("t31_h1_3")(torch.randn(2, 31, 40, device=dev))                          # the smallest batch plan
        LiveCNN(cnn_for("f32_conv1_w1"), 2, 16000, 160, 1600, audio_processor=ap_for(32), device=dev)
        assert torch.equal(big(x), want)
        for s, lc in big_lc.items():
            row = SHAPES[s]
            ls = LiveStreams(ap_for(row.F), 2, window_of(row), 160, 1600, device=dev)
            wav = torch.from_numpy(make_pcm(2, 12 * 1600, seed=row.T)).to(dev).float() / 32768.0
            for c in range(0, 12 * 1600, 1600):
                y, v = lc.push(wav[:, c:c + 1600])
                ref, _ = ls.push(wav[:, c:c + 1600], cnn_for(s))
                assert torch.equal(y[v.to(dev)], ref[v.to(dev)]), s
            assert bool(v.all())
