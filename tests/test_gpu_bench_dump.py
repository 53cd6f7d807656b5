"""bench.py --dump-outputs against the CPU oracle: the files must hold what the LAST timed step computed, from the
input set that step read (step i reads set i % NSETS), so a change to the step loop that dumps another set's buffers
fails here."""
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
pytestmark = pytest.mark.gpu


def test_dump_outputs_hold_the_last_timed_step(tmp_path):
    torch = pytest.importorskip("torch")
    if not torch.cuda.is_available():
        pytest.fail("GPU tests need a CUDA device (there is no CPU path)")
    steps, lanes = 7, 4                  # 4 lanes -> 4 input sets; the last step (6) reads set 2
    out = tmp_path / "dump"
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--gpus", "1", "--steps", str(steps),
                        "--warmup", "1", "--lanes", str(lanes), "--no-extras", "--no-cpu-baseline",
                        "--dump-outputs", str(out)], cwd=tmp_path, capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stderr[-3000:]
    got = {n: np.load(out / f"{n}.npy") for n in ("proposals", "detections", "pooled_7x7_sample", "pooled_14x14_sample")}
    assert all(a.dtype == np.float32 for a in got.values())
    assert sum(a.nbytes for a in got.values()) <= 64 << 20

    if ROOT not in sys.path:
        sys.path.insert(0, ROOT)
    import bench
    import oracle
    from objectdetection_b200.config import config
    conf = config()
    shapes = oracle.get_resnet_stage_shapes(conf.RESNET_STRIDES, conf.IMAGE_SHAPE)
    B = bench.B_PER_GPU
    anchors = oracle.gen_anchors(conf.IMAGE_SHAPE, B, conf.RPN_ANCHOR_SCALES, conf.RPN_ANCHOR_RATIOS, shapes,
                                 conf.RESNET_STRIDES, conf.RPN_ANCHOR_STRIDE)
    win = oracle.norm_boxes(np.array([bench.WINDOW_PX] * B), (bench.IMAGE, bench.IMAGE))

    def proposals_of(inp):
        return oracle.proposal_forward(inp["probs"], inp["bbox"], anchors, conf.RPN_BBOX_STDDEV, conf.PRE_NMS_ROIS_COUNT,
                                       conf.POST_NMS_ROIS_INFERENCE, conf.RPN_NMS_THRESHOLD)

    inp = bench.synth_inputs(1000 + (steps - 1) % lanes, B, anchors.shape[1])
    p = proposals_of(inp)
    det = oracle.detection_forward(p, inp["hprobs"], inp["hbbox"], win, conf.BBOX_STD_DEV, conf.DETECTION_MIN_THRESHOLD,
                                   conf.DETECTION_NMS_THRESHOLD, conf.DETECTION_POST_NMS_INSTANCES)
    assert np.array_equal(got["proposals"].view(np.uint32), p.view(np.uint32)), "proposals are not the last step's"
    other = proposals_of(bench.synth_rpn_head(1000 + steps % lanes, B, anchors.shape[1]))
    assert not np.array_equal(got["proposals"], other), "the check cannot tell the input sets apart"
    assert np.array_equal(got["detections"].view(np.uint32), det.view(np.uint32)), "detections are not the last step's"
    assert (det[:, :, 4] > 0).any()
    rows = np.sort(np.random.RandomState(0).choice(B * bench.N_ROIS, bench.DUMP_ROIS, replace=False))
    for P in (7, 14):
        want, _ = oracle.pyramid_roi_align(inp["fmaps"], p, bench.IMAGE, bench.IMAGE, P, P)
        want = want.reshape(B * bench.N_ROIS, P, P, bench.DEPTH)[rows]
        sample = got[f"pooled_{P}x{P}_sample"]
        if P == 14:
            assert np.array_equal(sample.view(np.uint32), want.view(np.uint32)), "14x14 sample differs from the oracle"
        else:
            assert np.allclose(sample, want, rtol=1e-4, atol=0), "7x7 sample differs from the oracle"
