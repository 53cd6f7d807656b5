"""Head losses with the reference's interface (MaskRCNN/building_blocks/loss_optimize.py:7-201): forward values.

``Loss`` keeps the four static methods, their argument order and their return tuples; each launches the fused
gather + reduce kernels of ``libodhead.so`` (``csrc/losses.cu``) on the current CUDA stream and returns 0-d CUDA
tensors. Gradients are not produced here — in the reference they come from TensorFlow's autodiff.

The network's outputs (``rpn_class_logits``, ``rpn_pred_box``, ``mrcnn_pred_logits``, ``mrcnn_pred_box``) may each be
float32 or bfloat16: a bfloat16 CUDA tensor aligned to the kernel's load (4 bytes for the RPN logit pairs, 2 for the
mrcnn logits, 8 for a box row) is read as it is, anything else is converted to float32. bfloat16 values are widened
exactly, so the losses, ``rpn_pred_box_pos`` and ``pred_active`` (all float32) are bit for bit those of the call on
``t.float()``. Targets and ``batch_active_class_ids`` are float32 / int32 as before.
"""
from __future__ import annotations

import torch

from . import _lib


def _losses(dev):
    return torch.empty((2,), dtype=torch.float32, device=dev)


class Loss():
    def __init__(self):
        pass

    @staticmethod
    def rpn_losses(rpn_target_class, rpn_class_logits, rpn_target_bbox=None, rpn_pred_box=None, want_pos=False):
        """Both RPN losses in one pass: (rpn_class_loss, rpn_box_loss, rpn_pred_box_pos or None)."""
        logits = _lib.as_cuda(rpn_class_logits, _lib.read_dtype([rpn_class_logits], 4))
        dev = logits.device
        tc = _lib.as_cuda(rpn_target_class, torch.int32, dev)
        tb = None if rpn_target_bbox is None else _lib.as_cuda(rpn_target_bbox, torch.float32, dev)
        pb = None if rpn_pred_box is None else _lib.as_cuda(rpn_pred_box, _lib.read_dtype([rpn_pred_box], 8), dev)
        B, A = logits.shape[0], logits.shape[1]
        L = _lib.lib()
        out = _losses(dev)
        pos = num = None
        if want_pos and pb is not None:
            pos = torch.zeros((min(B * A, B * max(int(tb.shape[1]), 1)), 4), dtype=torch.float32, device=dev)
            num = torch.zeros((1,), dtype=torch.int32, device=dev)
        ws = _lib.workspace(L.od_rpn_loss_workspace_bytes(B, A), dev)
        dl = _lib.DL()
        _lib.check(L.od_rpn_loss_forward(dl(tc), dl(logits), dl(tb), dl(pb), dl(out), dl(pos), dl(num), ws.data_ptr(),
                                         ws.numel(), _lib.stream_ptr(dev)), "od_rpn_loss_forward")
        if pos is not None:
            pos = pos[:min(int(num.item()), pos.shape[0])]
        return out[0], out[1], pos

    @staticmethod
    def rpn_class_loss(rpn_target_class, rpn_class_logits):
        """loss_optimize.py:11-44. rpn_target_class [B,A,1] (+1/-1/0), rpn_class_logits [B,A,2] -> scalar."""
        return Loss.rpn_losses(rpn_target_class, rpn_class_logits)[0]

    @staticmethod
    def rpn_box_loss(rpn_target_bbox, rpn_pred_box, rpn_target_class, batch_size):
        """loss_optimize.py:47-87 -> (rpn_pred_box_pos [P,4], loss)."""
        pb = _lib.as_cuda(rpn_pred_box, _lib.read_dtype([rpn_pred_box], 8))
        if pb.shape[0] != batch_size:
            raise ValueError(f"batch_size={batch_size} but rpn_pred_box has batch {pb.shape[0]}")
        # the class logits are not needed for this loss: a zero tensor keeps the single entry point
        logits = torch.zeros((pb.shape[0], pb.shape[1], 2), dtype=torch.float32, device=pb.device)
        _, loss, pos = Loss.rpn_losses(rpn_target_class, logits, rpn_target_bbox, pb, want_pos=True)
        return pos, loss

    @staticmethod
    def mrcnn_losses(mrcnn_target_class_ids, mrcnn_pred_logits=None, batch_active_class_ids=None, mrcnn_target_box=None,
                     mrcnn_pred_box=None):
        """Both detection-head losses in one launch: (pred_active or None, mrcnn_class_loss, mrcnn_box_loss)."""
        ids = _lib.as_cuda(mrcnn_target_class_ids, torch.int32)
        dev = ids.device
        lg = None if mrcnn_pred_logits is None else _lib.as_cuda(mrcnn_pred_logits, _lib.read_dtype([mrcnn_pred_logits], 2), dev)
        ac = None if batch_active_class_ids is None else _lib.as_cuda(batch_active_class_ids, torch.float32, dev)
        tb = None if mrcnn_target_box is None else _lib.as_cuda(mrcnn_target_box, torch.float32, dev)
        pb = None if mrcnn_pred_box is None else _lib.as_cuda(mrcnn_pred_box, _lib.read_dtype([mrcnn_pred_box], 8), dev)
        out = _losses(dev)
        pa = None if lg is None else torch.empty(tuple(ids.shape), dtype=torch.float32, device=dev)
        dl = _lib.DL()
        _lib.check(_lib.lib().od_mrcnn_loss_forward(dl(ids), dl(lg), dl(ac), dl(tb), dl(pb), dl(out), dl(pa),
                                                    _lib.stream_ptr(dev)), "od_mrcnn_loss_forward")
        return pa, out[0], out[1]

    @staticmethod
    def mrcnn_class_loss(mrcnn_target_class_ids, mrcnn_pred_logits, batch_active_class_ids):
        """loss_optimize.py:89-151 -> (pred_active [B,R], loss)."""
        pa, loss, _ = Loss.mrcnn_losses(mrcnn_target_class_ids, mrcnn_pred_logits, batch_active_class_ids)
        return pa, loss

    @staticmethod
    def mrcnn_box_loss(mrcnn_target_box, mrcnn_pred_box, mrcnn_target_class_ids, batch_size=2):
        """loss_optimize.py:154-201 (K.binary_crossentropy, as the reference has it) -> loss."""
        ids = _lib.as_cuda(mrcnn_target_class_ids, torch.int32)
        if ids.shape[0] != batch_size:
            raise ValueError(f"batch_size={batch_size} but mrcnn_target_class_ids has batch {ids.shape[0]}")
        return Loss.mrcnn_losses(ids, None, None, mrcnn_target_box, mrcnn_pred_box)[2]
