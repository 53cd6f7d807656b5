"""Seeded synthetic inputs of the BASELINE.json configurations (SURVEY.md §8d), shared by tests and bench."""
import numpy as np

f32 = np.float32


def rpn_outputs(rs, B, A):
    """fg prob ~ Beta(0.5, 4); bbox ~ N(0,1)."""
    fg = rs.beta(0.5, 4, size=(B, A)).astype(f32)
    probs = np.stack([f32(1) - fg, fg], axis=2).astype(f32)
    bbox = rs.normal(0, 1, size=(B, A, 4)).astype(f32)
    return probs, bbox


def rois_log_uniform(rs, B, N, image=1024, lo=16, hi=512):
    """sqrt(area) log-uniform [lo,hi] px, aspect log-uniform [0.5,2], centre uniform, clipped, normalised."""
    s = np.exp(rs.uniform(np.log(lo), np.log(hi), size=(B, N)))
    r = np.exp(rs.uniform(np.log(0.5), np.log(2.0), size=(B, N)))
    h, w = s / np.sqrt(r), s * np.sqrt(r)
    cy, cx = rs.uniform(0, image, size=(B, N)), rs.uniform(0, image, size=(B, N))
    boxes = np.stack([cy - h / 2, cx - w / 2, cy + h / 2, cx + w / 2], axis=2)
    boxes = np.clip(boxes, 0, image - 1) / (image - 1)
    return boxes.astype(f32)


def rois_with_edge_cases(rs, B, N, lo=4, hi=900):
    """rois_log_uniform boxes with the last 10 of image 1 zero padded and rows 0..12 of image 0 set to the cases where
    ROIAlign kernels go wrong: whole image, zero area, far edge, partly / entirely outside, flipped, NaN, thin,
    sub-pixel and integer-aligned taps."""
    props = rois_log_uniform(rs, B, N, lo=lo, hi=hi)
    props[1, N - 10:] = 0                                                     # zero padded proposals -> level 2
    props[0, 0] = [0, 0, 1, 1]                                                # last tap exactly on the far edge
    props[0, 1] = [0.3, 0.3, 0.3, 0.3]                                        # zero area: every bin on one pixel
    props[0, 2] = [0.25, 0.5, 1.0, 1.0]
    props[0, 3] = [-0.1, -0.2, 0.4, 0.5]                                      # partly outside -> extrapolated bins
    props[0, 4] = [0.5, 0.5, 1.2, 1.3]
    props[0, 5] = [0.9, 0.1, 0.2, 0.8]                                        # flipped in y -> per-bin path
    props[0, 6] = [0.1, 0.9, 0.8, 0.2]                                        # flipped in x
    props[0, 7] = [np.nan, 0.1, 0.5, 0.6]
    props[0, 8] = [0.0, 0.40, 1.0, 0.41]                                      # tall and thin: sparse rows, one column pair
    props[0, 9] = [0.40, 0.0, 0.41, 1.0]                                      # wide and flat: many column runs
    props[0, 10] = [1.5, 1.5, 2.0, 2.0]                                       # entirely outside
    props[0, 11] = [0.5, 0.5, 0.5 + 1e-4, 0.5 + 1e-4]                         # sub-pixel ROI
    props[0, 12] = [0.2, 0.2, 0.2 + 3 / 63.0, 0.2 + 3 / 63.0]                 # integer-aligned taps on P2 (lerp 0)
    return props


def pyramid(rs, B, sizes=(256, 128, 64, 32), D=256):
    return [rs.random_sample((B, s, s, D)).astype(f32) for s in sizes]


def head_outputs(rs, B, N, C, boosted=0.2):
    """probs = softmax(N(0,3) logits) with a fraction of rows boosted on a random fg class; bbox ~ N(0,1)."""
    logits = rs.normal(0, 3, size=(B, N, C))
    rows = rs.random_sample((B, N)) < boosted
    cls = rs.randint(1, C, size=(B, N))
    bi, ni = np.nonzero(rows)
    logits[bi, ni, cls[bi, ni]] += 12
    e = np.exp(logits - logits.max(-1, keepdims=True))
    probs = (e / e.sum(-1, keepdims=True)).astype(f32)
    bbox = rs.normal(0, 1, size=(B, N, C, 4)).astype(f32)
    return probs, bbox


def target_inputs(rs, B, N, G, n_pad=200):
    """proposals with trailing zero pads; GT = jittered copies of random proposals; explicit permutations."""
    props = rois_log_uniform(rs, B, N)
    props[:, N - n_pad:] = 0
    gt = np.zeros((B, G, 4), f32)
    cls = np.zeros((B, G), np.int32)
    for b in range(B):
        nv = int(rs.randint(1, G + 1))
        src = rs.choice(N - n_pad, nv, replace=False)
        gt[b, :nv] = props[b, src] + rs.normal(0, 0.01, size=(nv, 4)).astype(f32)
        cls[b, :nv] = rs.randint(1, 81, nv)
    pp = np.stack([rs.permutation(N) for _ in range(B)]).astype(np.int32)
    pn = np.stack([rs.permutation(N) for _ in range(B)]).astype(np.int32)
    return props, cls, gt, pp, pn


def random_boxes(rs, n, scale=1.0, flip=False):
    yx = rs.random_sample((n, 2)) * 0.8
    hw = rs.random_sample((n, 2)) * 0.3 + 0.01
    b = np.concatenate([yx, yx + hw], axis=1) * scale
    if flip:
        sw = rs.random_sample(n) < 0.3
        b[sw] = b[sw][:, [2, 3, 0, 1]]
    return b.astype(f32)
