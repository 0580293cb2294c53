"""Own bounds check of every kernel family (compute-sanitizer is closed on this GPU pool: profiles/r02_sanitizer.txt).

The C ABI is called directly with EVERY output tensor and the workspace embedded between guard bands filled with a
sentinel pattern; after forward + backward the guard bands must be untouched and every output fully written (no
sentinel left inside, nothing non-finite).  Geometries are ragged on purpose (batch not a multiple of any row tile,
T not a multiple of any chunk) and cover: SIMT recurrences (H = 32/64/128, fp32 and tensor-core GEMMs), the
tensor-core recurrences (recur_tc.cuh, forced), the non-recurrent scans (recur_nr.cuh), the wide weight-stationary
kernels (recur_wide.cuh, H = 256 / 1024: several m-tiles, a partial last tile) and the generic wide kernels, dense
and frame-dedup inputs.
"""
import ctypes

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

from snnimageclassification_b200 import ToSpikes, _cabi  # noqa: E402
from snnimageclassification_b200.modules import functional as F_  # noqa: E402
from _util import Guarded  # noqa: E402

DEV = torch.device("cuda:0")


def _run(B, T, N, H, O, layer, rec, tc, dedup, monkeypatch=None):
	g = torch.Generator().manual_seed(B * 1000 + H)
	theta = 0.03 if layer else 1.0
	consts = F_.LayerConsts(layer, 0, rec, float(np.float32(np.exp(-1 / 20))), float(np.float32(np.exp(-1 / 200))), theta,
		0.3 if layer else 1.0, float(np.float32(np.exp(-1 / 10))), tensor_core=tc)
	if dedup:
		img = (torch.randint(1, 256, (B, N), generator=g).float() / 255.0) * (torch.rand(B, N, generator=g) < 0.3)
		x = ToSpikes(T, use_periods=True).encode_batch(img.to(DEV))
	else:
		x = F_.mark_binary((torch.rand(B, T, N, generator=g) < 0.15).float().to(DEV))
	W_in = (torch.randn(N, H, generator=g) * theta).to(DEV)
	W_rec = (torch.randn(H, H, generator=g) * theta).to(DEV) if rec else None
	mask = (1 - torch.eye(H)).to(DEV) if rec else None
	W_out = torch.randn(H, O, generator=g).to(DEV)
	b_out = (torch.randn(O, generator=g) * 0.1).to(DEV)
	beta = torch.tensor([1.6], device=DEV) if layer else None
	labels = torch.randint(0, O, (B,), generator=g).to(DEV)
	lib = _cabi.lib()
	desc = F_.make_desc(consts, B, T, N, H, O, True, binary=True)
	runs = F_.get_runs(x)
	G = {k: Guarded((B, T, H)) for k in ("V", "Z")}
	if layer:
		G["a"] = Guarded((B, T, H))
	G["zbits"] = Guarded((B, T, H // 32), torch.int32)
	G["y"] = Guarded((B, T, O))
	G["logits"] = Guarded((B, O))
	G["tstar"] = Guarded((B, O), torch.int32)
	G["W_effT"] = Guarded((H, H))
	ws_f = Guarded((max(int(lib.snnk_forward_workspace_bytes(ctypes.byref(desc))), 16),), torch.uint8)
	p = _cabi.ptr
	rc = lib.snnk_forward(ctypes.byref(desc), p(x), p(W_in), p(W_rec), p(mask), p(beta), p(W_out), p(b_out), None, None, None,
		p(G["V"].t), p(G["a"].t) if layer else None, p(G["Z"].t), p(G["zbits"].t), p(G["y"].t), p(G["logits"].t), p(G["tstar"].t),
		p(ws_f.t), ws_f.t.numel(), p(runs), p(G["W_effT"].t) if rec else None, _cabi.stream_ptr())
	_cabi.check(rc, "snnk_forward")
	torch.cuda.synchronize()
	for k, gb in G.items():
		gb.check(k, written=(k != "W_effT" or rec) and k not in ("zbits", "tstar"))
	ws_f.check("forward workspace", written=False)
	loss, logp, gl = F_.run_head_nll(G["logits"].t, labels)
	D = {"dW_in": Guarded((N, H)), "dW_out": Guarded((H, O)), "db": Guarded((O,))}
	if rec:
		D["dW_rec"] = Guarded((H, H))
	ws_b = Guarded((max(int(lib.snnk_backward_workspace_bytes(ctypes.byref(desc))), 16),), torch.uint8)
	rc = lib.snnk_backward(ctypes.byref(desc), p(x), p(W_rec), p(mask), p(beta), p(W_out), None, p(G["V"].t),
		p(G["a"].t) if layer else None, p(G["Z"].t), p(G["zbits"].t), None, p(gl), p(G["tstar"].t), None, None, None, p(D["dW_in"].t),
		p(D["dW_rec"].t) if rec else None, p(D["dW_out"].t), p(D["db"].t), p(ws_b.t), ws_b.t.numel(), p(runs),
		p(G["W_effT"].t) if rec else None, _cabi.stream_ptr())
	_cabi.check(rc, "snnk_backward")
	torch.cuda.synchronize()
	for k, gb in D.items():
		gb.check(k)
	ws_b.check("backward workspace", written=False)
	for k, gb in G.items():      # the backward pass must not have touched the forward's outputs or their surroundings
		gb.check(k + " (after backward)", written=False)


@pytest.mark.parametrize("B,T,H,layer,rec,tc,dedup", [
	(21, 10, 32, 1, True, False, False), (21, 10, 64, 0, True, True, True), (37, 23, 128, 1, True, True, True),
	(37, 23, 128, 1, True, True, False), (5, 7, 128, 0, False, True, True), (130, 9, 64, 1, False, True, False),
	(9, 100, 128, 1, False, True, True), (3, 5, 128, 1, True, False, False)])
def test_guard_bands_narrow(B, T, H, layer, rec, tc, dedup):
	_run(B, T, 64, H, 10, layer, rec, tc, dedup)


@pytest.mark.parametrize("B,T", [(21, 10), (8, 33), (1, 4), (70, 6)])
def test_guard_bands_tensor_core_recurrence(B, T, monkeypatch):
	monkeypatch.setenv("SNNK_MMA_RECUR", "1")      # recur_tc.cuh is selected from B >= 1024 on its own
	_run(B, T, 64, 128, 10, 1, True, True, True)
	_run(B, T, 64, 128, 10, 0, True, True, False)


@pytest.mark.parametrize("B,T,H,layer,tc", [
	(21, 10, 256, 1, True), (150, 7, 256, 0, True), (131, 5, 1024, 1, True), (9, 6, 2048, 0, True), (300, 4, 512, 1, True),
	(6, 5, 256, 1, False)])
def test_guard_bands_wide(B, T, H, layer, tc):
	_run(B, T, 64, H, 10, layer, True, tc, False)
