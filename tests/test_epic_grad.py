"""CPU: the float64 restatement that the native gradients are checked against (tests/grad_lib.py) is pinned to the reference's
own heads and losses; the differentiable blob equals the packed one; the loss / gradient call rejects bad arguments."""
import ctypes
import os

import numpy as np
import pytest
import torch

import grad_lib
import oracle_lib as ol
from multimodal_particles_b200 import _native

MBM_CASES = ["mbm_c1", "mbm_odd", "mbm_n128", "mbm_wide", "mbm_ctx", "mbm_ctx_id"]
HEAD_RTOL, HEAD_ATOL = 2e-5, 2e-5   # the oracle's bar against the reference's fp32 heads (test_oracle_golden.py)


@pytest.mark.parametrize("case", MBM_CASES)
def test_restatement_heads_match_reference(case, golden_dir):
    z, cfg, model = ol.load_mbm_golden(os.path.join(golden_dir, case + ".npz"))
    ref = grad_lib.Restatement(model)
    ctx = z["context_continuous"] if "context_continuous" in z.files else None
    with torch.no_grad():
        for i in z["snap_steps"]:
            v, logits = ref.heads(torch.from_numpy(z["temb"][i][None]), z[f"snap{i}/x"], z[f"snap{i}/k"], z["mask"], ctx)
            np.testing.assert_allclose(v.numpy(), z[f"snap{i}/v"], rtol=HEAD_RTOL, atol=HEAD_ATOL)
            np.testing.assert_allclose(logits.numpy(), z[f"snap{i}/logits"], rtol=HEAD_RTOL, atol=HEAD_ATOL)


def test_restatement_losses_match_reference(golden_dir):
    z = np.load(os.path.join(golden_dir, "train_forward.npz"))
    mse, ce = grad_lib.bridge_losses(z["v"], z["logits"], z["x0"], z["x1"], z["k1"], z["mask"])
    np.testing.assert_allclose([float(mse), float(ce)], [z["loss_continuous"], z["loss_discrete"]], rtol=2e-6)


@pytest.mark.parametrize("case", MBM_CASES)
def test_packed_parameters_equal_pack_weights(case, golden_dir):
    _, _, model = ol.load_mbm_golden(os.path.join(golden_dir, case + ".npz"))
    enc = model.encoder
    head = enc.fc_layer if enc.add_discrete_head else None
    blob = enc.epic.packed_parameters(head)
    assert blob.requires_grad and blob.dtype == torch.float32
    assert torch.equal(blob.detach(), enc.epic.pack_weights(head))
    blob.sum().backward()
    assert enc.epic.epic.epic_proj.local_0.weight_g.grad is not None and enc.epic.epic.output_layer.weight_v.grad is not None


def test_loss_grad_argument_errors_are_codes():
    lib = _native.load()
    d = _native.EpicDims(dim_continuous=3, vocab_size=8, dim_time_emb=16, dim_cont_emb=16, dim_disc_emb=16, dim_hidden_local=16,
                         dim_hidden_glob=16, num_blocks=2, skip_connection=1, disc_head_hidden=8, dim_context=0)
    need = lib.mmb_epic_loss_grad_workspace_bytes(ctypes.byref(d), 64, 30)
    assert need > 0
    assert lib.mmb_epic_loss_grad_workspace_bytes(None, 64, 30) == 0
    assert lib.mmb_epic_loss_grad_workspace_bytes(ctypes.byref(d), -1, 30) == 0
    assert lib.mmb_epic_loss_grad_workspace_bytes(ctypes.byref(d), 64, 1025) == 0
    fake = ctypes.c_void_p(256)   # never dereferenced: every call below fails its checks first
    call = lambda dims, B, N, ws_bytes, W=fake, x=fake, out=fake: lib.mmb_epic_loss_grad(
        dims, W, x, fake, fake, fake, 16, fake, fake, fake, B, N, out, fake, None, fake, ws_bytes, None)
    assert call(None, 64, 30, need) == -1
    assert call(ctypes.byref(d), -1, 30, need) == -1 and b"B >= 1" in lib.mmb_last_error()
    assert call(ctypes.byref(d), 64, 1025, need) == -1
    assert call(ctypes.byref(d), 64, 30, need, W=None) == -1 and b"null" in lib.mmb_last_error()
    assert call(ctypes.byref(d), 64, 30, need, x=None) == -1
    assert call(ctypes.byref(d), 64, 30, need, out=None) == -1
    assert call(ctypes.byref(d), 64, 30, need - 1) == -3 and b"workspace" in lib.mmb_last_error()
    bad = _native.EpicDims(**{**d.as_dict(), "vocab_size": 33})
    assert call(ctypes.byref(bad), 64, 30, need) == -1
