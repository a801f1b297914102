"""The row decomposition behind LiveCNN (kws_live_cnn_*), checked without a GPU.

* A float64 restatement: each window's logits built from stream rows (computed once per stream from its frame table)
  plus the four window-specific rows of each convolution, against oracle.model_ref.cnn_forward on the materialised
  windows, for cnn-trad-fpool3 and the CNN family shapes of test_tc_shapes.py, at shifts of 160, 480 and 800 samples.
* The ring capacities of live_cnn.cu (cap = max_push / 160 + H rows), by brute force over push sequences: no row a
  push reads has been overwritten.
* The C ABI's argument errors.
"""
import ctypes

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from oracle import model_ref

# (T, F, conv_0, conv_1, linear layers): cnn-trad-fpool3 and the accepted CNN rows of test_tc_shapes.py
SHAPES = {
    "cnn-trad-fpool3": (101, 40, (20, 8), (10, 4), {"lin_0": 32, "dnn_0": 128}),
    "t60": (60, 40, (20, 8), (10, 4), {"lin_0": 32, "dnn_0": 128}),
    "t108": (108, 40, (20, 8), (10, 4), {"lin_0": 32, "dnn_0": 128}),
    "conv0_h21": (101, 40, (21, 8), (10, 4), {"lin_0": 32, "dnn_0": 128}),
    "conv0_w5_conv1_w5": (101, 40, (20, 5), (10, 5), {"lin_0": 32, "dnn_0": 128}),
}


def _cfg(T, Fq, k0, k1, lin):
    cfg = {"time": T, "frequency": Fq, "n_labels": 12,
           "conv_0": {"out_channels": 64, "kernel_size": list(k0), "stride": [1, 1]}, "pool_0": {"kernel_size": [1, 3]},
           "conv_1": {"out_channels": 64, "kernel_size": list(k1), "stride": [1, 1]}, "pool_1": {"kernel_size": [1, 1]}}
    for name, n in lin.items():
        cfg[name] = {"out_features": n}
    return cfg


def _weights(cfg, seed):
    g = torch.Generator().manual_seed(seed)
    k0, k1 = cfg["conv_0"]["kernel_size"], cfg["conv_1"]["kernel_size"]
    H1 = cfg["time"] - k0[0] + 1 - k1[0] + 1
    WP = (cfg["frequency"] - k0[1] + 1) // 3
    sd = {"layers.conv_0.weight": torch.randn(64, 1, *k0, generator=g, dtype=torch.float64) * 0.1,
          "layers.conv_0.bias": torch.randn(64, generator=g, dtype=torch.float64) * 0.1,
          "layers.conv_1.weight": torch.randn(64, 64, *k1, generator=g, dtype=torch.float64) * 0.05,
          "layers.conv_1.bias": torch.randn(64, generator=g, dtype=torch.float64) * 0.1}
    width = 64 * H1 * (WP - k1[1] + 1)
    for name in ("lin_0", "dnn_0", "dnn_1"):
        if name in cfg:
            n = cfg[name]["out_features"]
            sd[f"layers.{name}.weight"] = torch.randn(n, width, generator=g, dtype=torch.float64) / width ** 0.5
            sd[f"layers.{name}.bias"] = torch.randn(n, generator=g, dtype=torch.float64) * 0.1
            width = n
    sd["layers.lin_1.weight"] = torch.randn(12, width, generator=g, dtype=torch.float64) / width ** 0.5
    sd["layers.lin_1.bias"] = torch.zeros(12, dtype=torch.float64)
    return sd


def _conv0_rows(sd, x):
    """Pooled conv_0 rows of frames x [R + KH0 - 1, F]: [R, 64, WP]."""
    y = F.relu(F.conv2d(x[None, None], sd["layers.conv_0.weight"], sd["layers.conv_0.bias"]))
    return F.max_pool2d(y, (1, 3))[0].permute(1, 0, 2)


def _conv1_rows(sd, p):
    """conv_1 rows of pooled rows p [R + KH1 - 1, 64, WP]: [R, 64, 8]."""
    y = F.relu(F.conv2d(p.permute(1, 0, 2)[None], sd["layers.conv_1.weight"], sd["layers.conv_1.bias"]))
    return y[0].permute(1, 0, 2)


def live_cnn_ref(sd, cfg, table, edges, m):
    """Logits of windows k = 0 .. len(edges) - 1 of a stream from its rows.  table [R, F]: the stream's frame-table
    rows (window k's frame t = 2 .. T-3 is table row k m + t); edges [n_win, 4, F]: each window's frames 0, 1, T-2,
    T-1.  Stream rows of each convolution are computed once for the whole stream, window-specific rows (0, 1, H-2, H-1)
    once per window."""
    T = cfg["time"]
    KH0, KH1 = cfg["conv_0"]["kernel_size"][0], cfg["conv_1"]["kernel_size"][0]
    H0 = T - KH0 + 1
    H1 = H0 - KH1 + 1
    pooled = _conv0_rows(sd, table)        # stream pooled row r reads table rows r .. r + KH0 - 1
    c1 = _conv1_rows(sd, pooled)           # stream conv_1 row r reads pooled rows r .. r + KH1 - 1
    own = [0, 1, H0 - 2, H0 - 1]
    logits = []
    for k in range(edges.shape[0]):
        def frame(t):
            if t < 2:
                return edges[k, t]
            if t >= T - 2:
                return edges[k, t - T + 4]
            return table[k * m + t]

        def pooled_row(r):
            if r in own:
                return own_p[own.index(r)]
            return pooled[k * m + r]
        own_p = [_conv0_rows(sd, torch.stack([frame(r + i) for i in range(KH0)]))[0] for r in own]
        rows = []
        for r in range(H1):
            if r < 2 or r > H1 - 3:
                rows.append(_conv1_rows(sd, torch.stack([pooled_row(r + i) for i in range(KH1)]))[0])
            else:
                rows.append(c1[k * m + r])
        x = torch.stack(rows).permute(1, 0, 2).reshape(1, -1)   # [64, H1, 8] flattened like x.view(B, -1)
        for name in ("lin_0", "dnn_0", "dnn_1"):
            if f"layers.{name}.weight" in sd:
                x = F.linear(x, sd[f"layers.{name}.weight"], sd[f"layers.{name}.bias"])
        logits.append(F.linear(x, sd["layers.lin_1.weight"], sd["layers.lin_1.bias"])[0])
    return torch.stack(logits)


@pytest.mark.parametrize("shape", list(SHAPES))
@pytest.mark.parametrize("shift", [160, 480, 800])
def test_row_decomposition_matches_model_ref(shape, shift):
    T, Fq, k0, k1, lin = SHAPES[shape]
    cfg = _cfg(T, Fq, k0, k1, lin)
    sd = _weights(cfg, seed=len(shape) + shift)
    m = shift // 160
    n_win = 6
    g = torch.Generator().manual_seed(shift)
    table = torch.randn((n_win - 1) * m + T, Fq, generator=g, dtype=torch.float64) * 3 - 8
    edges = torch.randn(n_win, 4, Fq, generator=g, dtype=torch.float64) * 3 - 8
    wins = torch.stack([torch.cat([edges[k, :2], table[k * m + 2:k * m + T - 2], edges[k, 2:]])
                        for k in range(n_win)])
    with torch.no_grad():
        want = model_ref.cnn_forward(sd, cfg, wins)
        got = live_cnn_ref(sd, cfg, table, edges, m)
    err = float((got - want).abs().max() / want.abs().max())
    assert err <= 1e-12, err


def _rows_read_written(seen, n, W, H, Hc, KHn):
    """Stream rows of one ring a uniform push of n samples writes and reads (live_cnn.cu's jobs).  Hc: rows of this
    convolution's output per window; KHn: the next layer's kernel height (1 for the conv_1 ring, whose reader is the
    first Linear), Hn = Hc - KHn + 1 its output rows per window."""
    m, K = H // 160, n // H
    k0 = (seen - W) // H + 1
    written = range((k0 - 1) * m + Hc - 2, (k0 + K - 1) * m + Hc - 2)
    read = set()
    Hn = Hc - KHn + 1
    for k in range(k0, k0 + K):
        if k < 0:
            continue
        # window-specific rows of the next layer read the stream rows among their inputs; the first Linear reads
        # every stream row of the window
        for r in range(Hn):
            for i in range(KHn):
                t = r + i
                if 2 <= t <= Hc - 3:
                    read.add(k * m + t)
    if KHn > 1:   # the next layer's new stream rows that some window uses read stream rows R .. R + KHn - 1
        for R in range((k0 - 1) * m + Hn - 2, (k0 + K - 1) * m + Hn - 2):
            if any(k * m + 2 <= R <= k * m + Hn - 3 for k in range(max(0, (R - Hn) // m - 1), R // m + 2)):
                read.update(range(R, R + KHn))
    return written, read


@pytest.mark.parametrize("H", [160, 320, 480, 800])
@pytest.mark.parametrize("shape", ["cnn-trad-fpool3", "t60", "conv0_h21"])
def test_ring_capacity_by_brute_force(H, shape):
    """Simulate the pooled and conv_1 rings over push sequences (cap = max_push / 160 + H rows): every stream row a
    push reads is in its slot, written by an earlier or the same push and not overwritten since."""
    T, Fq, k0, k1, lin = SHAPES[shape]
    W = 160 * (T - 1)
    H0 = T - k0[0] + 1
    H1 = H0 - k1[0] + 1
    rng = np.random.default_rng(H)
    for max_push in (H, 4 * H, 10 * H):
        for Hc, KHn in ((H0, k1[0]), (H1, 1)):
            cap = max_push // 160 + Hc
            slot = {}
            seen = 0
            for _ in range(300):
                n = H * int(rng.integers(1, max_push // H + 1))
                written, read = _rows_read_written(seen, n, W, H, Hc, KHn)
                for r in written:
                    slot[r % cap] = r
                for r in read:
                    assert slot.get(r % cap) == r, (max_push, Hc, seen, n, r)
                seen += n


def test_live_cnn_c_abi_argument_errors_without_gpu(native_lib):
    """Null handles and buffers return KWS_ERR_INVALID with a message; the size query returns 0."""
    lib = native_lib
    out = ctypes.c_void_p()
    assert lib.kws_live_cnn_state_bytes(None, None, 4, 16000, 160, 1600) == 0
    assert lib.kws_live_cnn_create(None, None, 4, 16000, 160, 1600, ctypes.byref(out)) == 1
    assert b"model is null" in lib.kws_last_error()
    assert lib.kws_live_cnn_create(None, None, 4, 16000, 160, 1600, None) == 1
    assert b"out is null" in lib.kws_last_error()
    assert lib.kws_live_cnn_push(None, None, 160, None, None) == 1
    assert b"live CNN state is null" in lib.kws_last_error()
    assert lib.kws_live_cnn_push_pcm16(None, None, 160, None, None) == 1
    assert b"live CNN state is null" in lib.kws_last_error()
    assert lib.kws_live_cnn_reset(None, None, 1, None) == 1
    assert b"live CNN state is null" in lib.kws_last_error()
    lib.kws_live_cnn_destroy(None)
