"""The Faster R-CNN proposal layer on a batch of images in one call (od_frcnn_proposal_forward with B > 1).

Expected output: oracle.frcnn_proposals run on each image alone, column 0 set to the image index, the images
concatenated. Rows are compared bit for bit, and so are the zero rows of proposals_padded after the last kept one.
The CPU-only checks at the end (workspace query, argument refusals) run in a child process that sees no GPU."""
import ctypes
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [os.path.dirname(os.path.abspath(__file__)), ROOT]

import oracle  # noqa: E402

torch = pytest.importorskip("torch")
f32 = np.float32
H, W, NA = 38, 63, 9            # 600x1000 at stride 16: 21,546 anchors
IMAGE = (600, 1000, 3)


@pytest.fixture
def need_cuda():
    if not torch.cuda.is_available():
        pytest.fail("GPU tests need a CUDA device (there is no CPU path)")


def cu(a):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def host(t):
    torch.cuda.synchronize()
    return t.detach().cpu().numpy()


def _bits(x):
    return np.ascontiguousarray(x, f32).view(np.uint32)


def _inputs(rs, B, h=H, w=W):
    return rs.random_sample((B, h, w, 2 * NA)), rs.normal(0, 0.5, size=(B, h, w, 4 * NA))


def _expected(probs, bbox, image_h, image_w, pre_n, post_n, thr, **kw):
    """Per-image oracle rows with column 0 = b, and the per-image counts."""
    rows = []
    for b in range(probs.shape[0]):
        r = oracle.frcnn_proposals(probs[b:b + 1], bbox[b:b + 1], image_h, image_w, pre_n, post_n, thr, **kw)
        r[:, 0] = b
        rows.append(r)
    return np.concatenate(rows), np.array([r.shape[0] for r in rows])


def _check(P, want, counts, post_n):
    """get_proposals, num_proposals and proposals_padded (kept rows, then zeros) against the expected rows."""
    B = counts.size
    num = host(P.num_proposals)
    assert num.dtype == np.int32 and np.array_equal(num, counts), (num, counts)
    got = host(P.get_proposals())
    assert got.shape == want.shape, (got.shape, want.shape)
    assert np.array_equal(_bits(got), _bits(want))
    pad = host(P.proposals_padded)
    assert pad.shape == (B * post_n, 5)
    n = int(counts.sum())
    assert np.array_equal(_bits(pad[:n]), _bits(want))
    assert not _bits(pad[n:]).any()


# ------------------------------------------------------------------ parity against the per-image oracle
@pytest.mark.gpu
@pytest.mark.parametrize("mode,thr", [("train", 0.7), ("train", 0.2), ("test", 0.7)])
def test_batch_fp64(need_cuda, mode, thr):
    """B = 4, fp64 inputs (128-bit keys, rank sort per image): 'train' 12000 -> 2000, 'test' 6000 -> 300."""
    from objectdetection_b200 import fasterrcnn
    rs = np.random.RandomState(41)
    probs, bbox = _inputs(rs, 4)
    pre, post = (12000, 2000) if mode == "train" else (6000, 300)
    P = fasterrcnn.Proposals(mode, probs, bbox, image_shape=IMAGE, nms_threshold=thr)
    want, counts = _expected(probs, bbox, 600, 1000, pre, post, thr)
    assert counts.min() > 0
    _check(P, want, counts, post)


@pytest.mark.gpu
@pytest.mark.parametrize("thr,pre", [(0.7, 12000), (0.2, 3000)])
def test_batch_fp32_tied_scores(need_cuda, thr, pre):
    """B = 3, fp32 inputs with scores quantised to 3 decimals: the radix-select top-k over B rows, ties to the lower
    index within each image."""
    from objectdetection_b200 import fasterrcnn
    rs = np.random.RandomState(42)
    probs, bbox = _inputs(rs, 3)
    p32, b32 = np.round(probs, 3).astype(f32), bbox.astype(f32)
    P = fasterrcnn.Proposals('train', cu(p32), cu(b32), image_shape=IMAGE, nms_threshold=thr, pre_nms_top_n=pre)
    want, counts = _expected(p32.astype(np.float64), b32.astype(np.float64), 600, 1000, pre, 2000, thr)
    _check(P, want, counts, 2000)


def _mixed_batch(rs, kinds):
    """One image per kind: 'normal'; 'empty' (every decoded box below the 16 px minimum, so the min-size filter removes
    all); 'few' (only 60 boxes pass the filter, fewer than post_n)."""
    probs, bbox = _inputs(rs, len(kinds))
    for b, k in enumerate(kinds):
        if k == "normal":
            continue
        small = np.ones((H * W * NA,), bool)
        if k == "few":
            small[rs.choice(small.size, 60, replace=False)] = False
        d = bbox[b].reshape(-1, 4)
        d[small, 2:] = -8.0                      # exp(-8) * anchor side + 1 < 16 px
    return probs, bbox


@pytest.mark.gpu
@pytest.mark.parametrize("kinds", [
    ["empty", "normal", "few", "normal"],
    ["normal", "few", "empty", "normal"],
    ["normal", "few", "normal", "empty"],
    ["empty", "empty"],
], ids=["empty-first", "empty-middle", "empty-last", "all-empty"])
@pytest.mark.parametrize("dtype", ["f64", "f32"])
def test_batch_mixed_images(need_cuda, kinds, dtype):
    from objectdetection_b200 import fasterrcnn
    rs = np.random.RandomState(43 + len(kinds))
    probs, bbox = _mixed_batch(rs, kinds)
    if dtype == "f32":
        probs, bbox = probs.astype(f32), bbox.astype(f32)
    P = fasterrcnn.Proposals('test', probs, bbox, image_shape=IMAGE, nms_threshold=0.7)
    want, counts = _expected(probs.astype(np.float64), bbox.astype(np.float64), 600, 1000, 6000, 300, 0.7)
    for b, k in enumerate(kinds):
        assert (counts[b] == 0) == (k == "empty") and (counts[b] < 300) == (k != "normal"), (kinds, counts)
    _check(P, want, counts, 300)


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", ["f64", "f32"])
def test_batch_equals_single_image_calls(need_cuda, dtype):
    """Every image of a batch gives the rows of its own batch-of-one call (with its index in column 0)."""
    from objectdetection_b200 import fasterrcnn
    rs = np.random.RandomState(44)
    probs, bbox = _inputs(rs, 4)
    if dtype == "f32":
        probs, bbox = probs.astype(f32), bbox.astype(f32)
    P = fasterrcnn.Proposals('train', cu(probs), cu(bbox), image_shape=IMAGE, nms_threshold=0.7)
    got, num = host(P.get_proposals()), host(P.num_proposals)
    off = 0
    for b in range(4):
        S = fasterrcnn.Proposals('train', cu(probs[b:b + 1]), cu(bbox[b:b + 1]), image_shape=IMAGE, nms_threshold=0.7)
        one = host(S.get_proposals()).copy()
        assert host(S.num_proposals)[0] == num[b] == one.shape[0]
        assert not one[:, 0].any()
        one[:, 0] = b
        assert np.array_equal(_bits(got[off:off + num[b]]), _bits(one)), b
        off += num[b]
    assert off == got.shape[0]


@pytest.mark.gpu
def test_batch_tall_images_without_fp32_screen(need_cuda):
    """Two 131072 x 48 images (past kFrcnnScreenMaxSide: every pair takes the fp64 path) of near-threshold pairs chosen
    so that the fp32 screen alone would misjudge them."""
    from objectdetection_b200 import fasterrcnn
    from test_gpu_filter_edges import _frcnn_pair_inputs
    image_h = 131072
    pairs = [_frcnn_pair_inputs(np.random.RandomState(s), image_h, 48, 0.7, adversarial=True) for s in (5, 6)]
    assert all(m > 100 for _, _, m in pairs)
    probs = np.concatenate([p for p, _, _ in pairs])
    bbox = np.concatenate([b for _, b, _ in pairs])
    n = probs.shape[1] * probs.shape[2] * NA
    P = fasterrcnn.Proposals('test', probs, bbox, image_shape=(image_h, 48, 3), nms_threshold=0.7, pre_nms_top_n=n,
                             post_nms_top_n=n, min_box_hw=1)
    want, counts = _expected(probs, bbox, image_h, 48, n, n, 0.7, min_hw=1)
    assert np.all((n // 2 < counts) & (counts < n)), counts
    _check(P, want, counts, n)


@pytest.mark.gpu
def test_roi_pool_on_batched_proposals(need_cuda):
    """roi_pool on a [B,38,63,512] map takes the batched rows as they are: each row pools from its own image."""
    from objectdetection_b200 import fasterrcnn
    rs = np.random.RandomState(45)
    B = 3
    probs, bbox = _inputs(rs, B)
    p32, b32 = probs.astype(f32), bbox.astype(f32)
    P = fasterrcnn.Proposals('test', cu(p32), cu(b32), image_shape=IMAGE, nms_threshold=0.7)
    want, counts = _expected(p32.astype(np.float64), b32.astype(np.float64), 600, 1000, 6000, 300, 0.7)
    _check(P, want, counts, 300)
    fmap = rs.random_sample((B, H, W, 512)).astype(f32)
    pooled = host(fasterrcnn.roi_pool(cu(fmap), P.get_proposals(), IMAGE))
    wp = oracle.roi_pool(fmap, want, 600.0, 1000.0)
    assert pooled.shape == (want.shape[0], 7, 7, 512)
    assert np.array_equal(_bits(pooled), _bits(wp))
    # the same rows pooled against each image alone: the batch column selected the image
    first = want[want[:, 0] == 1].copy()
    first[:, 0] = 0
    assert np.array_equal(_bits(pooled[want[:, 0] == 1]), _bits(oracle.roi_pool(fmap[1:2], first, 600.0, 1000.0)))


@pytest.mark.gpu
def test_batch16_realistic_workspace(need_cuda):
    """B = 16 at 600x1000, 12000 -> 2000 (about 18 MB of NMS mask per image), fp32 inputs as the bench feeds them."""
    from objectdetection_b200 import _lib, fasterrcnn
    rs = np.random.RandomState(46)
    B = 16
    probs = rs.random_sample((B, H, W, 2 * NA)).astype(f32)
    bbox = rs.normal(0, 0.5, size=(B, H, W, 4 * NA)).astype(f32)
    P = fasterrcnn.Proposals('train', cu(probs), cu(bbox), image_shape=IMAGE, nms_threshold=0.7)
    want, counts = _expected(probs.astype(np.float64), bbox.astype(np.float64), 600, 1000, 12000, 2000, 0.7)
    _check(P, want, counts, 2000)
    p = _frcnn_params(_lib, 12000, 2000)
    nbytes = _lib.lib().od_frcnn_proposal_workspace_bytes_batch(B, H, W, ctypes.byref(p))
    assert nbytes > B * 12000 * 188 * 8         # one [K, ceil(K/64) rounded to even] u64 mask per image


# ------------------------------------------------------------------ CPU only: workspace query and refusals
def _frcnn_params(lib, pre_n, post_n):
    p = lib.FrcnnParams()
    p.feat_stride, p.image_h, p.image_w, p.min_box_hw = 16, 600, 1000, 16
    p.pre_nms_top_n, p.post_nms_top_n, p.nms_threshold, p.num_anchors = pre_n, post_n, 0.7, NA
    for i, v in enumerate(oracle.FRCNN_BASE_ANCHORS.reshape(-1)):
        p.base_anchors[i] = float(v)
    return p


# (case, probs shape, bbox shape, proposals shape, num_out shape, post_n)
_REFUSALS = [
    ("baseline-B3", (3, 2, 3, 18), (3, 2, 3, 36), (15, 5), (3,), 5),
    ("empty-batch", (0, 2, 3, 18), (0, 2, 3, 36), (0, 5), (0,), 5),
    ("bbox-batch-mismatch", (3, 2, 3, 18), (2, 2, 3, 36), (15, 5), (3,), 5),
    ("proposals-rows-one-image", (3, 2, 3, 18), (3, 2, 3, 36), (5, 5), (3,), 5),
    ("proposals-rows-plus-one", (3, 2, 3, 18), (3, 2, 3, 36), (16, 5), (3,), 5),
    ("num_out-one", (3, 2, 3, 18), (3, 2, 3, 36), (15, 5), (1,), 5),
    ("batch-above-cap", (65536, 2, 3, 18), (65536, 2, 3, 36), (65536 * 5, 5), (65536,), 5),
    ("rows-above-int32", (65535, 2, 3, 18), (65535, 2, 3, 36), (65535 * 40000, 5), (65535,), 40000),
]
_EXPECT = {"baseline-B3": -7, "empty-batch": 0, "bbox-batch-mismatch": -3, "proposals-rows-one-image": -3,
           "proposals-rows-plus-one": -3, "num_out-one": -3, "batch-above-cap": -8, "rows-above-int32": -8}
_NAMES = {"bbox-batch-mismatch": "rpn_bbox", "proposals-rows-one-image": "proposals",
          "proposals-rows-plus-one": "proposals", "num_out-one": "num_out", "batch-above-cap": "batch",
          "rows-above-int32": "post_nms_top_n"}


def _worker():
    """Runs in a child process with CUDA_VISIBLE_DEVICES="": fake DLTensors that are never dereferenced, as in
    test_abi_validation.py (an accepted call fails at its first CUDA call with OD_ERR_CUDA, -7)."""
    if os.environ.get("CUDA_VISIBLE_DEVICES") != "":
        raise SystemExit("refusing to run: CUDA_VISIBLE_DEVICES must be empty")
    from objectdetection_b200 import _lib
    from test_abi_validation import _a, _tensor
    L = _lib.lib()
    out = {"ws": {}, "calls": {}}
    p = _frcnn_params(_lib, 12000, 2000)
    out["ws"]["single"] = L.od_frcnn_proposal_workspace_bytes(H, W, ctypes.byref(p))
    for b in (-1, 0, 1, 2, 4, 16, 65535, 65536):
        out["ws"][str(b)] = L.od_frcnn_proposal_workspace_bytes_batch(b, H, W, ctypes.byref(p))
    for case, ps, bs, prs, ns, post_n in _REFUSALS:
        keep = []
        t = [_tensor(_a(n, dt, sh), "baseline", keep, 0x10000000 * (i + 1))
             for i, (n, dt, sh) in enumerate((("p", "f32", ps), ("b", "f32", bs), ("pr", "f32", prs), ("n", "i32", ns)))]
        before = L.od_launch_count()
        status = L.od_frcnn_proposal_forward(t[0], t[1], ctypes.byref(_frcnn_params(_lib, 10, post_n)), t[2], t[3],
                                             0x7F0000000000, 1 << 40, None)
        out["calls"][case] = [status, L.od_last_error_detail().decode(errors="replace"), L.od_launch_count() != before]
    json.dump(out, sys.stdout)


@pytest.fixture(scope="module")
def cpu_results():
    env = dict(os.environ, CUDA_VISIBLE_DEVICES="")
    flags = ["-s"] if sys.flags.no_user_site else []
    r = subprocess.run([sys.executable, *flags, os.path.abspath(__file__), "--worker"], env=env, cwd=ROOT,
                       capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-4000:]
    return json.loads(r.stdout)


def test_workspace_query_batch(cpu_results):
    ws = cpu_results["ws"]
    assert ws["1"] == ws["single"] > 0
    assert ws["0"] < ws["1"] < ws["2"] < ws["4"] < ws["16"] < ws["65535"]
    # the per-image part grows linearly: 16 images need 15 more image-sized segments than one
    assert ws["16"] - ws["1"] >= 15 * (ws["1"] - ws["0"]) - 16 * 4096
    assert ws["-1"] == 0 and ws["65536"] == 0


@pytest.mark.parametrize("case", [c[0] for c in _REFUSALS])
def test_batch_arguments_refused(cpu_results, case):
    status, detail, launched = cpu_results["calls"][case]
    assert status == _EXPECT[case], (case, status, detail)
    if status not in (-7, 0):
        assert not launched, case
    if case in _NAMES:
        assert _NAMES[case] in detail, (case, detail)


if __name__ == "__main__" and sys.argv[1:] == ["--worker"]:
    _worker()
