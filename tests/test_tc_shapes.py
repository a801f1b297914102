"""Every tensor-core ResNet kernel variant, and the shapes at the edges of the plans that choose between them, against a
float64 reference.

The bf16 / bf16x3 ResNet path is two whole-network kernels (conv_tc.cu): the column sweep (resnet_sweep.cuh) and the
position-major kernel (resnet_fused.cuh), each templated on NKC = ceil(C / 16) 16-channel K chunks.  The host plans
(tc_sweep_plan, tc_fused_plan, tc_geom) pick one per (model, T, F, precision).  Each row of SHAPES pins the kernel the
plans choose on a B200 in both precisions and names the instantiation it is there to reach; the module asserts at import
that the rows reach all 23 non-debug instantiations.

The reference is oracle.model_ref.resnet_forward / cnn_forward in float64 (they are dtype-agnostic), so the bf16x3
1e-3 bar is not measured against a reference with rounding of its own.
"""
import functools
import zlib
from collections import namedtuple

import numpy as np
import pytest
import torch

import honk2_b200
from conftest import logit_err
from honk2_b200 import synth
from honk2_b200.class_registry import find_cls
from oracle import model_ref

pytestmark = pytest.mark.gpu

LOGIT_TOL = 1e-3     # bf16x3: the fp32 tolerance, identical argmax
BF16_TOL = 3e-2      # bf16: argmax agrees where the reference's top-2 margin exceeds twice the error bound
SWEEP, FUSED, NONE = "resnet_tc_sweep_kernel", "resnet_tc_fused_kernel", "unsupported"


@pytest.fixture(scope="module")
def dev(native_lib):
    assert torch.cuda.is_available(), "these tests need the B200"
    return torch.device("cuda", 0)


def _kernel_path(m, dev, T, F):
    import ctypes as C
    lib, st = m._state(dev)
    lib.kws_model_kernel_path.restype = C.c_char_p
    return lib.kws_model_kernel_path(st["handle"], T, F, m._precision_id()).decode()


def _workspace_bytes(m, dev, B, T, F):
    lib, st = m._state(dev)
    return lib.kws_model_workspace_bytes(st["handle"], B, T, F, m._precision_id())


def _check(y, ref, precision):
    """bf16x3 at the fp32 tolerance with identical argmax; bf16 at its own, argmax where the margin decides it."""
    assert np.isfinite(y).all()
    if precision == "bf16x3":
        assert logit_err(y, ref) <= LOGIT_TOL, logit_err(y, ref)
        assert np.array_equal(y.argmax(1), ref.argmax(1))
    else:
        assert logit_err(y, ref) <= BF16_TOL, logit_err(y, ref)
        if ref.shape[1] < 2:
            return
        bound = BF16_TOL * np.maximum(np.abs(ref).max(axis=1), 1e-3)
        top2 = np.sort(ref, axis=1)[:, -2:]
        decided = (top2[:, 1] - top2[:, 0]) > 2 * bound
        assert np.array_equal(y.argmax(1)[decided], ref.argmax(1)[decided])


# ---------------------------------------------------------------------------------------------
# ResNet shapes

# The 23 kernels conv_tc.cu instantiates outside the debug build: the sweep at NKC 1-3 in five layouts (planar: one
# bulk copy per 8-channel plane, for multi-strip maps; 32B: 16-channel rows, single-strip maps; split: bf16x3 on 32B
# rows; packed: several short maps stacked in one strip; packed+split), and the position-major kernel at NKC 1-4.
VARIANTS = ({f"sweep<{n}>/{lay}" for n in (1, 2, 3) for lay in ("planar", "32B", "split", "packed", "packed+split")}
            | {f"fused<{n}>/{p}" for n in (1, 2, 3, 4) for p in ("bf16", "bf16x3")})

Row = namedtuple("Row", "id C L dil pool labels T F bf16 bf16x3 batches reaches")
S, P, U = SWEEP, FUSED, NONE
SHAPES = [
    # NKC = 1: three epilogue warp groups share two planes
    Row("c16_d13", 16, 13, True, None, 12, 101, 40, S, S, (1, 4, 149), "sweep<1>/32B sweep<1>/split"),
    Row("c16_d13_1label", 16, 13, True, None, 1, 101, 40, S, S, (4,), "sweep<1>/32B sweep<1>/split"),
    Row("c16_d13_13labels", 16, 13, True, None, 13, 101, 40, S, S, (4,), "sweep<1>/32B sweep<1>/split"),  # > 12 epilogue warps
    Row("c1_pool43", 1, 6, False, (4, 3), 12, 101, 40, S, S, (6, 149), "sweep<1>/packed sweep<1>/packed+split"),
    Row("c8_t301", 8, 4, False, None, 12, 301, 40, S, P, (3,), "sweep<1>/planar fused<1>/bf16x3"),
    Row("c12_pool33", 12, 5, True, (3, 3), 12, 101, 40, P, P, (1, 4, 149), "fused<1>/bf16 fused<1>/bf16x3"),
    # NKC = 4: 49-64 maps run on the position-major kernel only
    Row("c64_d13", 64, 13, True, None, 12, 101, 40, P, P, (1, 4, 149), "fused<4>/bf16 fused<4>/bf16x3"),
    Row("c64_d13_100labels", 64, 13, True, None, 100, 101, 40, P, P, (4,), "fused<4>/bf16 fused<4>/bf16x3"),
    Row("c49_pool43", 49, 6, False, (4, 3), 12, 101, 40, P, P, (4,), "fused<4>/bf16 fused<4>/bf16x3"),  # 15 pad channels
    # NKC = 2
    Row("c19_pool43_t901", 19, 6, False, (4, 3), 12, 901, 40, P, P, (3,), "fused<2>/bf16 fused<2>/bf16x3"),
    Row("c32_t257", 32, 7, False, None, 12, 257, 40, S, P, (3,), "sweep<2>/planar fused<2>/bf16x3"),
    Row("c20_pool22", 20, 6, False, (2, 2), 12, 101, 40, S, S, (5,), "sweep<2>/packed sweep<2>/packed+split"),
    # the 6144-byte epilogue-constant table: (1 + layers) * 48 * 4 bytes
    Row("c48_l31", 48, 31, False, None, 12, 101, 40, S, S, (3,), "sweep<3>/32B sweep<3>/split"),
    Row("c48_l32", 48, 32, False, None, 12, 101, 40, P, P, (3,), "fused<3>/bf16 fused<3>/bf16x3"),
    # layers 19-21 have dilation 64, the largest the sweep stages; layer 22 has 128
    Row("c19_l21", 19, 21, True, None, 12, 101, 40, S, S, (3,), "sweep<2>/32B sweep<2>/split"),
    Row("c19_l22", 19, 22, True, None, 12, 101, 40, P, P, (3,), "fused<2>/bf16 fused<2>/bf16x3"),
    # depths: the cap, and 1-3 (layer 1 is the last layer; no skip; one skip)
    Row("c16_l64", 16, 64, False, None, 12, 101, 40, S, S, (3,), "sweep<1>/32B sweep<1>/split"),
    Row("c33_l1", 33, 1, True, None, 12, 101, 40, S, S, (3,), "sweep<3>/32B sweep<3>/split"),
    Row("c17_l2", 17, 2, True, None, 12, 101, 40, S, S, (3,), "sweep<2>/32B sweep<2>/split"),
    Row("c17_l3", 17, 3, True, None, 12, 101, 40, S, S, (3,), "sweep<2>/32B sweep<2>/split"),
    # the column limit is tc_geom's padded width W + d <= 256
    Row("c16_l2_f255", 16, 2, False, None, 12, 101, 255, S, S, (2,), "sweep<1>/32B sweep<1>/split"),
    Row("c16_l2_f256", 16, 2, False, None, 12, 101, 256, U, U, (2,), ""),
    Row("c16_d13_f240", 16, 13, True, None, 12, 101, 240, S, S, (2,), "sweep<1>/32B sweep<1>/split"),
    Row("c16_d13_f241", 16, 13, True, None, 12, 101, 241, U, U, (2,), ""),
    # strips of 128 rows: 154 is the shortest map the sweep runs on two strips, 257 needs three
    Row("c45_t154", 45, 13, True, None, 12, 154, 40, S, P, (1, 3, 149), "sweep<3>/planar fused<3>/bf16x3"),
    Row("c45_t256", 45, 13, True, None, 12, 256, 40, S, P, (3,), "sweep<3>/planar fused<3>/bf16x3"),
    Row("c45_t257", 45, 13, True, None, 12, 257, 40, S, P, (3,), "sweep<3>/planar fused<3>/bf16x3"),
    # a single short map: under 60 % of its strip it gains nothing on the sweep
    Row("c45_t76", 45, 13, True, None, 12, 76, 40, P, P, (3,), "fused<3>/bf16 fused<3>/bf16x3"),
    Row("c45_t77", 45, 13, True, None, 12, 77, 40, S, S, (3,), "sweep<3>/32B sweep<3>/split"),
    # tiny clips, dilation up to 16 >> H: 8, 7 and 4 maps stacked per strip (batches not a multiple of that)
    Row("c45_t2", 45, 13, True, None, 12, 2, 40, S, S, (5, 149), "sweep<3>/packed sweep<3>/packed+split"),
    Row("c45_t3", 45, 13, True, None, 12, 3, 40, S, S, (9,), "sweep<3>/packed sweep<3>/packed+split"),
    Row("c45_t17", 45, 13, True, None, 12, 17, 40, S, S, (6,), "sweep<3>/packed sweep<3>/packed+split"),
    # the label cap of kws_resnet_create (1025 labels are refused in every precision: test_label_cap)
    Row("c16_1024labels", 16, 6, False, None, 1024, 101, 40, S, S, (3,), "sweep<1>/32B sweep<1>/split"),
    # refused by both precisions
    Row("c65", 65, 6, False, None, 12, 101, 40, U, U, (2,), ""),
]
del S, P, U


def _variant(row, precision):
    """The instantiation a row runs, from its pinned path and the plans' layout rules: the sweep packs pooled maps and
    maps under 60 % of their strips, keeps single-strip maps on 32-byte rows, and runs bf16x3 on those two layouts only."""
    path = row.bf16 if precision == "bf16" else row.bf16x3
    nkc = -(-row.C // 16)
    if path == FUSED:
        return f"fused<{nkc}>/{precision}"
    assert path == SWEEP
    ph, pw = row.pool or (1, 1)
    H = row.T // ph
    strips = -(-H // 128)
    packed = row.pool is not None or H * 100 < strips * 128 * 60   # 60: kSwMinStripPct in conv_tc.cu
    layout = "packed" if packed else "32B" if strips == 1 else "planar"
    if precision == "bf16x3":
        assert layout != "planar", row.id
        layout = "packed+split" if packed else "split"
    return f"sweep<{nkc}>/{layout}"


for _r in SHAPES:
    assert set(_r.reaches.split()) == {_variant(_r, p) for p in ("bf16", "bf16x3") if getattr(_r, p) != NONE}, _r.id
assert set().union(*(r.reaches.split() for r in SHAPES)) == VARIANTS, VARIANTS - set().union(*(r.reaches.split() for r in SHAPES))
assert len(VARIANTS) == 23
ROWS = {r.id: r for r in SHAPES}
SUPPORTED = [r.id for r in SHAPES if r.bf16 != NONE]
ON_SWEEP = [(r.id, p) for r in SHAPES for p in ("bf16", "bf16x3") if getattr(r, p) == SWEEP]


def _cfg(row):
    cfg = {"n_layers": row.L, "n_feature_maps": row.C, "use_dilation": row.dil, "n_labels": row.labels}
    if row.pool is not None:
        cfg["pool"] = list(row.pool)
    return cfg


@functools.lru_cache(maxsize=None)
def _weights(row_id):
    """Seeded default initialisation, hardened (synth.harden_): fp32 state dict."""
    row = ROWS[row_id]
    torch.manual_seed(zlib.crc32(row_id.encode()))
    m = find_cls("model.ResNet")(_cfg(row))
    sd = m.state_dict()
    synth.harden_(sd)
    return {k: v.clone() for k, v in sd.items()}


def _model(row, dev, precision):
    m = find_cls("model.ResNet")(_cfg(row))
    m.eval()
    m.load_state_dict(_weights(row.id))
    m.precision = precision
    return m.to(dev)


def _input(row, B):
    """randn * 3 - 8, times a gain in [0.25, 2) per utterance: the pooled features of noise alone barely differ between
    utterances, so without the gain an utterance that got another one's logits would pass."""
    g = torch.Generator().manual_seed(zlib.crc32(f"{row.id}/{B}".encode()))
    x = torch.randn(B, row.T, row.F, generator=g) * 3.0 - 8.0
    return x * (0.25 + 1.75 * torch.rand(B, 1, 1, generator=g))


def _ref_rows(B):
    """The utterances checked against the reference: all of a small batch, the first and last four of a large one."""
    return np.arange(B) if B <= 16 else np.concatenate([np.arange(4), np.arange(B - 4, B)])


@functools.lru_cache(maxsize=None)
def _reference(row_id, B):
    row = ROWS[row_id]
    sd = {k: v.double() for k, v in _weights(row_id).items() if v.is_floating_point()}
    x = _input(row, B)[_ref_rows(B)].double()
    with torch.no_grad():
        return model_ref.resnet_forward(sd, _cfg(row), x).numpy()


@pytest.mark.parametrize("precision", ["bf16", "bf16x3"])
@pytest.mark.parametrize("row_id", list(ROWS))
def test_kernel_path_and_workspace(dev, row_id, precision):
    """The pinned kernel; a workspace of 0 bytes exactly when the model is refused, and then the forward raises."""
    row = ROWS[row_id]
    m = _model(row, dev, precision)
    path = _kernel_path(m, dev, row.T, row.F)
    assert path == getattr(row, precision), (row_id, precision, path)
    ws = _workspace_bytes(m, dev, max(row.batches), row.T, row.F)
    assert (ws == 0) == (path == NONE), ws
    if path == NONE:
        with pytest.raises(honk2_b200.NativeError), torch.no_grad():
            m(_input(row, 2).to(dev))


@pytest.mark.parametrize("row_id", [r.id for r in SHAPES if r.bf16 == NONE])
def test_refused_shapes_still_run_in_fp32(dev, row_id):
    row = ROWS[row_id]
    m = _model(row, dev, "fp32")
    with torch.no_grad():
        y = m(_input(row, 2).to(dev)).cpu().numpy()
    ref = _reference(row_id, 2)
    assert logit_err(y, ref) <= LOGIT_TOL, logit_err(y, ref)
    assert np.array_equal(y.argmax(1), ref.argmax(1))


@pytest.mark.parametrize("precision", ["fp32", "bf16", "bf16x3"])
def test_label_cap(dev, precision):
    """A ResNet with 1025 labels is refused when its native handle is created, in every precision (c16_1024labels
    runs the cap itself)."""
    row = ROWS["c16_1024labels"]._replace(id="c16_1025labels", labels=1025)
    torch.manual_seed(0)
    m = find_cls("model.ResNet")(_cfg(row))
    m.eval()
    m.precision = precision
    m = m.to(dev)
    with pytest.raises(honk2_b200.NativeError, match="n_labels=1025"), torch.no_grad():
        m(_input(row, 2).to(dev))


@pytest.mark.parametrize("precision", ["bf16", "bf16x3"])
@pytest.mark.parametrize("row_id", SUPPORTED)
def test_tc_resnet_vs_float64(dev, row_id, precision):
    """Every batch size of the row against the float64 reference; a repeated launch is bit-identical."""
    row = ROWS[row_id]
    m = _model(row, dev, precision)
    assert _kernel_path(m, dev, row.T, row.F) == getattr(row, precision)
    for B in row.batches:
        xd = _input(row, B).to(dev)
        with torch.no_grad():
            y = m(xd)
            y_again = m(xd)
        assert y.shape == (B, row.labels)
        assert torch.equal(y, y_again), "repeated launches differ"
        _check(y.cpu().numpy()[_ref_rows(B)], _reference(row_id, B), precision)


@pytest.mark.parametrize("row_id,precision", ON_SWEEP)
def test_sweep_rows_on_the_position_major_kernel(dev, monkeypatch, row_id, precision):
    """HONK2_TC_SWEEP=0 (read when the model's native handle is created) moves a sweep row to the position-major
    kernel: it must meet the same reference, and agree with the sweep within 1e-2 of the logit scale."""
    row = ROWS[row_id]
    B = min(row.batches[-1], 16)
    xd = _input(row, B).to(dev)
    m_sweep = _model(row, dev, precision)
    with torch.no_grad():
        y_sweep = m_sweep(xd)
    monkeypatch.setenv("HONK2_TC_SWEEP", "0")
    m_pos = _model(row, dev, precision)
    assert _kernel_path(m_pos, dev, row.T, row.F) == FUSED
    with torch.no_grad():
        y_pos = m_pos(xd)
    _check(y_pos.cpu().numpy()[_ref_rows(B)], _reference(row_id, B), precision)
    assert float((y_sweep - y_pos).abs().max()) <= 1e-2 * float(y_pos.abs().max())


# ---------------------------------------------------------------------------------------------
# CNN: cnn_tc_plan runs conv_0 (64 maps, 1-8 columns) + max pool (1, 3) + conv_1 (64 maps, 8 output columns, at most 80
# output rows) on the tensor cores, the first Linear (<= 32 outputs) as a bf16 GEMM and up to three fp32 Linear layers
# of at most 512.  Each shape sets the fields that differ from cnn-trad-fpool3.

CnnRow = namedtuple("CnnRow", "id T F conv0 conv1 lin labels accepted")
CNN_SHAPES = [
    CnnRow("zoo", 101, 40, (20, 8), (10, 4), {"lin_0": 32, "dnn_0": 128}, 12, True),
    CnnRow("t60_h1_32", 60, 40, (20, 8), (10, 4), {"lin_0": 32, "dnn_0": 128}, 12, True),
    CnnRow("t108_h1_80", 108, 40, (20, 8), (10, 4), {"lin_0": 32, "dnn_0": 128}, 12, True),
    CnnRow("t109_h1_81", 109, 40, (20, 8), (10, 4), {"lin_0": 32, "dnn_0": 128}, 12, False),
    CnnRow("conv0_h21", 101, 40, (21, 8), (10, 4), {"lin_0": 32, "dnn_0": 128}, 12, True),
    CnnRow("conv0_w5_conv1_w5", 101, 40, (20, 5), (10, 5), {"lin_0": 32, "dnn_0": 128}, 12, True),
    CnnRow("f32_conv1_w1", 101, 32, (20, 8), (10, 1), {"lin_0": 32, "dnn_0": 128}, 12, True),
    CnnRow("lin0_dnn0_dnn1", 101, 40, (20, 8), (10, 4), {"lin_0": 32, "dnn_0": 128, "dnn_1": 64}, 12, True),
    CnnRow("lin1_only", 101, 40, (20, 8), (10, 4), {}, 20, True),
    CnnRow("lin1_only_33labels", 101, 40, (20, 8), (10, 4), {}, 33, False),
    CnnRow("lin0_33", 101, 40, (20, 8), (10, 4), {"lin_0": 33, "dnn_0": 128}, 12, False),
    CnnRow("dnn0_512", 101, 40, (20, 8), (10, 4), {"lin_0": 32, "dnn_0": 512}, 12, True),
    CnnRow("dnn0_513", 101, 40, (20, 8), (10, 4), {"lin_0": 32, "dnn_0": 513}, 12, False),
]
CNN_ROWS = {r.id: r for r in CNN_SHAPES}


def _cnn_cfg(row):
    cfg = {"time": row.T, "frequency": row.F, "dropout_prob": 0.5, "n_labels": row.labels,
           "conv_0": {"out_channels": 64, "kernel_size": list(row.conv0), "stride": [1, 1]},
           "pool_0": {"kernel_size": [1, 3]},
           "conv_1": {"out_channels": 64, "kernel_size": list(row.conv1), "stride": [1, 1]},
           "pool_1": {"kernel_size": [1, 1]}}
    for name, n in row.lin.items():
        cfg[name] = {"out_features": n}
    return cfg


@functools.lru_cache(maxsize=None)
def _cnn_weights(row_id):
    torch.manual_seed(zlib.crc32(row_id.encode()))
    sd = find_cls("model.CNN")(_cnn_cfg(CNN_ROWS[row_id])).state_dict()
    synth.harden_(sd)
    return {k: v.clone() for k, v in sd.items()}


@pytest.mark.parametrize("row_id", list(CNN_ROWS))
def test_cnn_tc_shapes_vs_float64(dev, row_id):
    """Accepted shapes: bf16 against float64 at BF16_TOL, bit-identical under chunking and batch splits.  Refused
    shapes: kernel path "unsupported", no workspace, NativeError from the bf16 forward, and the fp32 path still matches."""
    row = CNN_ROWS[row_id]
    cfg = _cnn_cfg(row)
    B = 23
    g = torch.Generator().manual_seed(zlib.crc32(row_id.encode()))
    x = (torch.randn(B, row.T, row.F, generator=g) * 3.0 - 8.0) * (0.25 + 1.75 * torch.rand(B, 1, 1, generator=g))
    sd64 = {k: v.double() for k, v in _cnn_weights(row_id).items() if v.is_floating_point()}
    with torch.no_grad():
        ref = model_ref.cnn_forward(sd64, cfg, x.double()).numpy()
    m = find_cls("model.CNN")(cfg)
    m.eval()
    m.load_state_dict(_cnn_weights(row_id))
    m.precision = "bf16"
    m = m.to(dev)
    xd = x.to(dev)
    path = _kernel_path(m, dev, row.T, row.F)
    assert path == ("cnn_tc_fused_kernel" if row.accepted else NONE), path
    assert (_workspace_bytes(m, dev, B, row.T, row.F) == 0) == (not row.accepted)
    if not row.accepted:
        with pytest.raises(honk2_b200.NativeError), torch.no_grad():
            m(xd)
        m.precision = "fp32"
        with torch.no_grad():
            y = m(xd).cpu().numpy()
        assert logit_err(y, ref) <= LOGIT_TOL, logit_err(y, ref)
        assert np.array_equal(y.argmax(1), ref.argmax(1))
        return
    with torch.no_grad():
        y = m(xd)
        m.chunk = {"fp32": 0, "bf16": 7}
        y2 = m(xd)
        y3 = torch.cat([m(xd[:10]), m(xd[10:])])
    _check(y.cpu().numpy(), ref, "bf16")
    assert torch.equal(y, y2), "the CNN tensor-core path is deterministic: chunking must not change a bit"
    assert torch.equal(y, y3)
