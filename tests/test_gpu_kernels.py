"""Kernel-level parity: every C-ABI compute entry point vs the CPU oracle on the
same seeded inputs (run on the B200 box: pytest -m gpu)."""

import ctypes

import numpy as np
import pytest

from tests import parity_util as pu
from tests.parity_util import orc

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def gpu(built_lib):
  import torch
  from adanet_b200 import _lib
  assert torch.cuda.is_available()
  _lib.check(built_lib.adn_init(), "adn_init")
  return built_lib


def _dev(a):
  import torch
  return torch.as_tensor(np.ascontiguousarray(a)).cuda()


def _sp():
  import torch
  return torch.cuda.current_stream().cuda_stream


PATHS = ["simt", "auto"]


def _set_path(name):
  from adanet_b200 import _lib
  _lib.set_dense_path({"simt": _lib.PATH_SIMT, "auto": _lib.PATH_AUTO, "tcgen05": _lib.PATH_TCGEN05}[name])


# fp32 GEMM tolerance: |err| <= 2e-6 * sum_k |a||b| bound, checked as relative-to-max
GEMM_RTOL = 3e-6


@pytest.mark.parametrize("path", PATHS)
@pytest.mark.parametrize("B,I,O,act", [
    (256, 100, 64, 1), (1024, 100, 1024, 1), (512, 1024, 1024, 1), (300, 784, 128, 1), (1024, 1024, 10, 0),
    (7, 5, 3, 0), (129, 33, 17, 1), (4096, 512, 512, 1), (128, 100, 10, 0),
])
def test_dense_fwd(gpu, path, B, I, O, act):
  import torch
  from adanet_b200 import _lib
  _set_path(path)
  rng = np.random.default_rng(B + I + O)
  x = rng.standard_normal((B, I)).astype(np.float32)
  w = orc.glorot_uniform(rng, I, O)
  b = rng.standard_normal(O).astype(np.float32) * 0.1
  want = x.astype(np.float64) @ w.astype(np.float64) + b
  if act:
    want = np.maximum(want, 0)
  xd, wd, bd = _dev(x), _dev(w), _dev(b)
  yd = torch.empty((B, O), dtype=torch.float32, device="cuda")
  fws_bytes = _lib.query(_lib.Q_DENSE_FWD_WS, B, I, O)
  fws = torch.empty((max(fws_bytes, 16),), dtype=torch.uint8, device="cuda")
  _lib.check(gpu.adn_dense_fwd(xd.data_ptr(), wd.data_ptr(), bd.data_ptr(), yd.data_ptr(), B, I, O, act,
                               fws.data_ptr(), fws_bytes, _sp()), "adn_dense_fwd")
  got = yd.cpu().numpy()
  scale = (np.abs(x).astype(np.float64) @ np.abs(w).astype(np.float64)).max()
  assert np.abs(got - want).max() <= GEMM_RTOL * scale, (np.abs(got - want).max(), scale)
  # no-bias variant
  _lib.check(gpu.adn_dense_fwd(xd.data_ptr(), wd.data_ptr(), None, yd.data_ptr(), B, I, O, 0, fws.data_ptr(), fws_bytes,
                               _sp()), "adn_dense_fwd")
  want2 = x.astype(np.float64) @ w.astype(np.float64)
  assert np.abs(yd.cpu().numpy() - want2).max() <= GEMM_RTOL * scale
  _set_path("auto")


@pytest.mark.parametrize("path", PATHS)
@pytest.mark.parametrize("B,I,O,mask,want_dx", [
    (256, 64, 10, 1, True), (1024, 1024, 1024, 1, True), (512, 100, 256, 0, False), (300, 128, 128, 1, True),
    (4096, 512, 512, 1, True), (7, 5, 3, 0, True), (129, 33, 17, 1, True), (2048, 1024, 10, 1, True),
])
def test_dense_bwd(gpu, path, B, I, O, mask, want_dx):
  import torch
  from adanet_b200 import _lib
  _set_path(path)
  rng = np.random.default_rng(B * 3 + I + O)
  x = rng.standard_normal((B, I)).astype(np.float32)
  if mask:
    x = np.maximum(x, 0)     # x is a ReLU output
  w = orc.glorot_uniform(rng, I, O)
  dz = (rng.standard_normal((B, O)) / B).astype(np.float32)
  x64, w64, dz64 = x.astype(np.float64), w.astype(np.float64), dz.astype(np.float64)
  want_dw = x64.T @ dz64
  want_db = dz64.sum(0)
  want_dxv = dz64 @ w64.T
  if mask:
    want_dxv = want_dxv * (x > 0)
  ws_bytes = _lib.query(_lib.Q_DENSE_BWD_WS, B, I, O)
  ws = torch.empty((ws_bytes,), dtype=torch.uint8, device="cuda")
  xd, wd, dzd = _dev(x), _dev(w), _dev(dz)
  dx = torch.full((B, I), 7.0, dtype=torch.float32, device="cuda") if want_dx else None
  dw = torch.empty((I, O), dtype=torch.float32, device="cuda")
  db = torch.empty((O,), dtype=torch.float32, device="cuda")
  _lib.check(gpu.adn_dense_bwd(xd.data_ptr(), wd.data_ptr(), dzd.data_ptr(), dx.data_ptr() if want_dx else None,
                               dw.data_ptr(), db.data_ptr(), B, I, O, mask, ws.data_ptr(), ws_bytes, _sp()),
             "adn_dense_bwd")
  s_dw = (np.abs(x64).T @ np.abs(dz64)).max()
  assert np.abs(dw.cpu().numpy() - want_dw).max() <= GEMM_RTOL * s_dw
  assert np.abs(db.cpu().numpy() - want_db).max() <= GEMM_RTOL * np.abs(dz64).sum(0).max()
  if want_dx:
    s_dx = (np.abs(dz64) @ np.abs(w64).T).max()
    assert np.abs(dx.cpu().numpy() - want_dxv).max() <= GEMM_RTOL * s_dx
  # determinism: a second launch gives bit-identical gradients
  dw2 = torch.empty_like(dw)
  _lib.check(gpu.adn_dense_bwd(xd.data_ptr(), wd.data_ptr(), dzd.data_ptr(), None, dw2.data_ptr(), db.data_ptr(),
                               B, I, O, mask, ws.data_ptr(), ws_bytes, _sp()), "adn_dense_bwd")
  assert torch.equal(dw, dw2)
  _set_path("auto")


@pytest.mark.parametrize("head,B,C", [(0, 256, 10), (0, 1000, 10), (0, 37, 3), (0, 4096, 16), (1, 300, 1), (2, 300, 1),
                                       (1, 128, 4), (0, 128, 64)])
def test_head_loss(gpu, head, B, C):
  import torch
  from adanet_b200 import _lib
  rng = np.random.default_rng(B + C + head)
  logits = (rng.standard_normal((B, C)) * 2).astype(np.float32)
  if head == 0:
    labels = rng.integers(0, C, B)
    want_l, want_g = orc.softmax_xent_mean(logits, labels)
    lab_d, labf_d = _dev(labels.astype(np.int64)), None
  else:
    labels = rng.standard_normal((B, C)).astype(np.float32) if head == 1 else (rng.random((B, C)) > 0.5).astype(np.float32)
    want_l, want_g = (orc.mse_mean if head == 1 else orc.sigmoid_xent_mean)(logits, labels)
    lab_d, labf_d = None, _dev(labels)
  ws_bytes = _lib.query(_lib.Q_HEAD_WS, B, C, 1)
  ws = torch.empty((ws_bytes,), dtype=torch.uint8, device="cuda")
  ld = _dev(logits)
  loss = torch.zeros((1,), dtype=torch.float32, device="cuda")
  g = torch.empty((B, C), dtype=torch.float32, device="cuda")
  _lib.check(gpu.adn_head_loss(head, ld.data_ptr(), lab_d.data_ptr() if lab_d is not None else None,
                               labf_d.data_ptr() if labf_d is not None else None, loss.data_ptr(), g.data_ptr(),
                               B, C, ws.data_ptr(), ws_bytes, _sp()), "adn_head_loss")
  assert abs(float(loss.item()) - float(want_l)) < 2e-6 * max(1.0, abs(float(want_l)))
  np.testing.assert_allclose(g.cpu().numpy(), want_g, atol=2e-7 + 1e-5 * np.abs(want_g).max())


@pytest.mark.parametrize("mix", ["scalar", "vector"])
@pytest.mark.parametrize("B,C,N,use_bias,lam,beta,mult", [
    (256, 10, 1, False, 0.0, 0.0, 2.0), (1000, 10, 2, False, 0.01, 0.001, 2.0), (4096, 10, 5, True, 0.1, 0.01, 2.0),
    (333, 3, 3, True, 0.05, 0.0, 1.0), (128, 16, 4, False, 0.0, 0.5, 2.0),
    (70001, 10, 3, True, 0.01, 0.001, 2.0),     # > 512 CTAs: two-level finalize, ragged last CTA
])
def test_ensemble_head(gpu, mix, B, C, N, use_bias, lam, beta, mult):
  import torch
  from adanet_b200 import _lib
  rng = np.random.default_rng(B + C + N)
  members = [(rng.standard_normal((B, C)) * 2).astype(np.float32) for _ in range(N)]
  labels = rng.integers(0, C, B)
  cx = [float(np.sqrt(k + 1)) for k in range(N)]
  if mix == "scalar":
    w = [np.float32(rng.uniform(-0.5, 1.0)) for _ in range(N)]
    w_arr = np.array(w, dtype=np.float32)
  else:
    w = [rng.uniform(-0.5, 1.0, C).astype(np.float32) for _ in range(N)]
    w_arr = np.stack(w)
  bias = (rng.standard_normal(C) * 0.1).astype(np.float32)
  ens = orc.ensemble_logits(mix, w, bias, members, None)
  want_loss, g = orc.softmax_xent_mean(ens, labels)
  want_reg = orc.complexity_regularization(w, cx, lam, beta)
  want_dw, want_db = orc.ensemble_grads(mix, w, cx, lam, beta, mult, g, members, None, True)
  md = [_dev(m) for m in members]
  ptrs = _lib.ptr_array([m.data_ptr() for m in md])
  gam = _lib.f32_array([float(orc.adanet_gamma(c, lam, beta)) for c in cx])
  wd, bd, lab = _dev(w_arr), _dev(bias), _dev(labels.astype(np.int64))
  out3 = torch.zeros((3,), dtype=torch.float32, device="cuda")
  dw = torch.zeros_like(wd)
  db = torch.zeros((C,), dtype=torch.float32, device="cuda")
  dens = torch.zeros((B, C), dtype=torch.float32, device="cuda")
  ens_out = torch.zeros((B, C), dtype=torch.float32, device="cuda")
  ws_bytes = _lib.query(_lib.Q_HEAD_WS, B, C, N)
  ws = torch.empty((ws_bytes,), dtype=torch.uint8, device="cuda")
  _lib.check(gpu.adn_ensemble_head(0, {"scalar": 0, "vector": 1}[mix], ptrs, N, wd.data_ptr(), bd.data_ptr(), gam,
                                   int(lam == 0.0 and beta == 0.0), mult, lab.data_ptr(), None, out3.data_ptr(),
                                   dw.data_ptr(), db.data_ptr() if use_bias else None, dens.data_ptr(),
                                   ens_out.data_ptr(), B, C, ws.data_ptr(), ws_bytes, _sp()), "adn_ensemble_head")
  o = out3.cpu().numpy()
  assert abs(o[0] - float(want_loss)) < 3e-6 * max(1.0, abs(float(want_loss)))
  assert abs(o[1] - float(want_reg)) < 1e-6
  assert abs(o[2] - float(want_loss + want_reg)) < 3e-6 * max(1.0, abs(float(want_loss)))
  np.testing.assert_allclose(ens_out.cpu().numpy(), ens, atol=1e-5)
  np.testing.assert_allclose(dens.cpu().numpy(), g, atol=2e-7 + 1e-5 * np.abs(g).max())
  want_dw_arr = np.array([np.asarray(d) for d in want_dw], dtype=np.float32).reshape(w_arr.shape)
  np.testing.assert_allclose(dw.cpu().numpy(), want_dw_arr, atol=5e-6)
  if use_bias:
    np.testing.assert_allclose(db.cpu().numpy(), want_db, atol=5e-6)


@pytest.mark.parametrize("spec", [("sgd", 0.05), ("momentum", 0.05, 0.9), ("rmsprop", 0.01), ("adam", 0.001),
                                  ("momentum_cosine", 0.05, 0.9, 4), ("momentum_cosine", 0.05, 0.9, 50, 0.1)])
def test_opt_step(gpu, spec):
  import torch
  from adanet_b200.core import engine as eng
  rng = np.random.default_rng(11)
  shapes = [(100, 64), (64,), (64, 10), (10,), (5000,), (3,)]
  ps = [rng.standard_normal(s).astype(np.float32) for s in shapes]
  ref = [p.copy() for p in ps]
  dev = [_dev(p) for p in ps]
  opt_o = orc.make_optimizer(spec)
  opt_e = eng._Optimizer(spec, dev)
  for step in range(5):
    gs = [rng.standard_normal(s).astype(np.float32) for s in shapes]
    opt_o.apply(ref, gs)
    opt_e.apply(gpu, [_dev(g) for g in gs], _sp())
  for a, b in zip(dev, ref):
    np.testing.assert_allclose(a.cpu().numpy(), b, rtol=2e-5, atol=2e-6)


def test_ema_and_l1(gpu):
  import torch
  from adanet_b200 import _lib
  state = torch.zeros((3,), dtype=torch.float32, device="cuda")
  loss = torch.zeros((1,), dtype=torch.float32, device="cuda")
  want = orc.ZeroDebiasEMA(0.999)
  got = []
  for l in (1.0, 0.5, 0.25):      # candidate_test.py:83-132 golden sequence
    loss.fill_(l)
    _lib.check(gpu.adn_ema_update(state.data_ptr(), loss.data_ptr(), 0.999, _sp()), "adn_ema_update")
    got.append(float(state[2].item()))
    assert abs(got[-1] - float(want.update(l))) < 1e-5
  np.testing.assert_allclose(got, [1.0, 0.750, 0.583], atol=1e-3)
  x = np.random.default_rng(3).standard_normal(12345).astype(np.float32)
  out = torch.zeros((1,), dtype=torch.float32, device="cuda")
  _lib.check(gpu.adn_l1_norm(_dev(x).data_ptr(), x.size, out.data_ptr(), _sp()), "adn_l1_norm")
  assert abs(float(out.item()) - float(np.abs(x.astype(np.float64)).sum())) < 1e-2


def test_record_and_counter(gpu):
  import torch
  from adanet_b200 import _lib
  a = torch.tensor([1.5], device="cuda")
  b = torch.tensor([2.5], device="cuda")
  step = torch.zeros((), dtype=torch.int64, device="cuda")
  trace = torch.zeros((4, 2), dtype=torch.float32, device="cuda")
  src = _lib.ptr_array([a.data_ptr(), b.data_ptr()])
  for i in range(6):
    a.fill_(float(i))
    _lib.check(gpu.adn_record_scalars(src, 2, trace.data_ptr(), 2, step.data_ptr(), 4, _sp()), "record")
    _lib.check(gpu.adn_counter_add(step.data_ptr(), 1, _sp()), "counter")
  assert int(step.item()) == 6
  np.testing.assert_allclose(trace.cpu().numpy()[:, 0], [4, 5, 2, 3])


@pytest.mark.parametrize("conv_path", ["tcgen05", "simt"])
@pytest.mark.parametrize("B,H,W,CIN,F", [(64, 32, 32, 3, 16), (5, 8, 8, 3, 16), (33, 28, 28, 1, 16), (16, 10, 10, 3, 32),
                                         (700, 32, 32, 3, 16), (3, 6, 4, 1, 48), (40, 28, 28, 1, 32), (9, 36, 20, 3, 16)])
def test_conv_stem_fwd_bwd(gpu, monkeypatch, conv_path, B, H, W, CIN, F):
  """SimpleCNN stem (customizing_adanet.ipynb SimpleCNNBuilder): conv3x3 same + ReLU + maxpool 2x2 + flatten,
  forward into split planes and the kernel / bias gradients, vs the oracle; the forward on both of its paths
  (tcgen05 implicit GEMM over pooled pixels, 3xTF32; exact-fp32 SIMT, which also serves shapes the former skips)."""
  import torch
  from adanet_b200 import _lib
  monkeypatch.setenv("ADN_CONV_PATH", conv_path)
  rng = np.random.default_rng(B * 7 + H + F)
  x = rng.uniform(0, 1, (B, H, W, CIN)).astype(np.float32)
  k = (rng.standard_normal((3, 3, CIN, F)) * np.sqrt(2.0 / (9 * CIN))).astype(np.float32)   # he_normal scale
  bias = (rng.standard_normal(F) * 0.1).astype(np.float32)
  want = orc.conv_stem_forward(k, bias, x)
  cols = (H // 2) * (W // 2) * F
  xd, kd, bd = _dev(x), _dev(k), _dev(bias)
  planes = torch.zeros((_lib.query(_lib.Q_PLANES_BYTES, B, cols) // 4,), dtype=torch.float32, device="cuda")
  arg = torch.zeros((B * cols // 16,), dtype=torch.int32, device="cuda")
  _lib.check(gpu.adn_conv_stem_fwd(xd.data_ptr(), kd.data_ptr(), bd.data_ptr(), planes.data_ptr(), arg.data_ptr(), B, H, W,
                                   CIN, F, _sp()), "adn_conv_stem_fwd")
  got = torch.empty((B, cols), dtype=torch.float32, device="cuda")
  _lib.check(gpu.adn_planes_merge(planes.data_ptr(), B, cols, got.data_ptr(), _sp()), "adn_planes_merge")
  got = got.cpu().numpy()
  np.testing.assert_allclose(got, np.asarray(want), rtol=0, atol=2e-6 * max(1.0, float(np.abs(want).max())))
  # sign bits = (pooled > 0): [ceil(cols/32) padded to whole k-blocks][B] words after the two planes
  f16 = _lib.plane_format() == _lib.PLANES_F16
  bk, esz = (64, 2) if f16 else (32, 4)
  nkbf = (cols + bk - 1) // bk
  plane_words = ((B * nkbf * bk + 127) // 128) * 128 * esz // 4
  nkb = nkbf * (bk // 32)
  words = planes.view(torch.int32)[2 * plane_words:2 * plane_words + nkb * B].cpu().numpy().view(np.uint32).reshape(nkb, B)
  padded = np.zeros((B, nkb * 32), dtype=bool)
  padded[:, :cols] = got > 0
  want_words = (padded.reshape(B, nkb, 32) * (np.uint64(1) << np.arange(32, dtype=np.uint64))).sum(axis=2).astype(np.uint32).T
  np.testing.assert_array_equal(words, want_words)
  # arg-max agrees with the oracle wherever the maximum is unique and active
  a = arg.cpu().numpy().view(np.uint32).reshape(B, cols // 16)
  pos = ((a[:, :, None] >> (2 * np.arange(16, dtype=np.uint32))) & 3).reshape(B, cols)
  o_arg = want.cache[1].reshape(B, cols)
  active = np.asarray(want) > 1e-4
  assert (pos[active] == o_arg[active]).mean() > 0.999
  # backward: dpooled already masked by (pooled > 0), as the first dense layer's dX epilogue delivers it
  g = (rng.standard_normal((B, cols)).astype(np.float32) / B) * (got > 0)
  dk_want, db_want = orc.conv_stem_backward(want, g)
  ws_bytes = _lib.query(_lib.Q_CONV_STEM_BWD_WS, B, CIN, F)
  ws = torch.empty((ws_bytes,), dtype=torch.uint8, device="cuda")
  dk = torch.empty((3, 3, CIN, F), dtype=torch.float32, device="cuda")
  db = torch.empty((F,), dtype=torch.float32, device="cuda")
  gd = _dev(g)
  for _ in range(2):     # twice: no state carried between calls
    _lib.check(gpu.adn_conv_stem_bwd(xd.data_ptr(), arg.data_ptr(), gd.data_ptr(), dk.data_ptr(), db.data_ptr(), B, H, W,
                                     CIN, F, ws.data_ptr(), ws_bytes, _sp()), "adn_conv_stem_bwd")
  tol = 2e-5 * max(1e-3, float(np.abs(dk_want).max()))
  np.testing.assert_allclose(dk.cpu().numpy(), dk_want, rtol=0, atol=tol)
  np.testing.assert_allclose(db.cpu().numpy(), db_want, rtol=0, atol=2e-5 * max(1e-3, float(np.abs(db_want).max())))


def test_conv_stem_rejects_bad_shapes(gpu):
  import torch
  from adanet_b200 import _lib
  t = torch.zeros((1 << 16,), dtype=torch.float32, device="cuda")
  p = t.data_ptr()
  for (h, w, c, f) in [(7, 8, 3, 16), (8, 8, 2, 16), (8, 8, 3, 24), (8, 8, 3, 128), (0, 8, 3, 16)]:
    assert gpu.adn_conv_stem_fwd(p, p, p, p, p, 2, h, w, c, f, _sp()) != 0
    assert b"adn_conv_stem_fwd" in gpu.adn_last_error()
  assert gpu.adn_conv_stem_bwd(p, p, p, p, p, 2, 8, 8, 3, 16, p, 16, _sp()) == _lib_err_workspace()


def _lib_err_workspace():
  return -12
