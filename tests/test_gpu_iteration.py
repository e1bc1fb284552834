"""Iteration-level parity: per-step losses, EMA, selection and growth of the GPU
engine vs the CPU oracle on identical seeded data and injected weights.

Tolerance: north_star's 1e-5 (fp32) on every per-step loss.  Training is a
chaotic map: two *correct* fp32 implementations that merely sum in a different
order drift apart, for some configurations by far more than 1e-5 (e.g. the
uncentred U[0,1) 784-feature data of SURVEY.md 8d at lr 0.05: the oracle
against itself with permuted feature order differs by 1.8e-4 after 40 steps).
So every parity configuration below is first shown to be well conditioned
(`test_parity_configs_are_well_conditioned`, CPU): the oracle's own
sensitivity -- to a permuted summation order AND to 2e-7 relative noise injected
into every dense forward/backward (the measured error level of the fp32 GPU
paths, tests/probe_accuracy.py) -- must be < 5e-6, half the 1e-5 budget.
"""

import numpy as np
import pytest

from tests import parity_util as pu
from tests.parity_util import orc

TOL = 1e-5
SENS_TOL = 5e-6
ENS = dict(optimizer=("sgd", 0.01), adanet_lambda=0.01, adanet_beta=0.001)


def _data(kind, n, d, c, seed):
  if kind == "tabular":
    return orc.make_tabular(n, d, c, seed=seed)
  if kind == "uniform":               # BASELINE configs[1] exactly as SURVEY.md 8d specifies it: X ~ U[0,1), uncentred
    return orc.make_uniform(n, d, c, seed=seed)
  if kind == "uniform_centered":      # BASELINE configs[1] shape, centred so that training is well conditioned
    x, y = orc.make_uniform(n, d, c, seed=seed)
    return (x - np.float32(0.5)).astype(np.float32), y
  if kind == "regression":
    rng = np.random.default_rng(seed)
    x = rng.standard_normal((n, d)).astype(np.float32)
    y = (x[:, :1] * 0.5 - x[:, 1:2] + 0.1 * rng.standard_normal((n, 1))).astype(np.float32)
    return x, y
  raise ValueError(kind)


# name -> dict(data=(kind, n, d, C, seed), cfgs=[(depth,width)], B, steps, iters, opt, ens, head, extra)
CONFIGS = {
    # BASELINE configs[1]: 784x10, 4 candidates (depth 1..2 x width 64/128), 3 iterations
    "config2": dict(data=("uniform_centered", 8192, 784, 10, 2234), cfgs=[(1, 64), (2, 64), (1, 128), (2, 128)],
                    B=1024, steps=40, iters=3, opt=("sgd", 0.05), ens=ENS),
    # north_star target: 100-feature 10-class tabular, 4-candidate DNN search, >= 100 steps
    "tabular4": dict(data=("tabular", 65536, 100, 10, 1234), cfgs=[(1, 64), (2, 128), (2, 256), (3, 512)],
                     B=512, steps=120, iters=2, opt=("sgd", 0.01), ens=ENS),
    "adam": dict(data=("tabular", 16384, 100, 10, 4321), cfgs=[(1, 128), (2, 128)], B=256, steps=60, iters=2,
                 # epsilon 1e-3: with small epsilon Adam turns a barely-alive ReLU unit (gradient 0 -> tiny) into a full
                 # lr-sized step: 2e-7 relative noise on the GEMMs makes the ORACLE itself jump by 3.5e-5 (eps 1e-8) / 1.4e-4 (1e-4)
                 opt=("adam", 0.0005, 0.9, 0.999, 1e-3),
                 ens=dict(optimizer=("adam", 0.0005, 0.9, 0.999, 1e-3), adanet_lambda=0.01, adanet_beta=0.001, use_bias=True,
                          mixture_weight_type="vector")),
    "rmsprop": dict(data=("tabular", 16384, 100, 10, 4321), cfgs=[(1, 128), (2, 128)], B=256, steps=60, iters=2,
                    opt=("rmsprop", 0.0005),
                    ens=dict(optimizer=("rmsprop", 0.0005), adanet_lambda=0.01, adanet_beta=0.001, use_bias=True,
                             mixture_weight_type="vector")),
    "momentum": dict(data=("tabular", 16384, 100, 10, 4321), cfgs=[(1, 128), (2, 128)], B=256, steps=60, iters=2,
                     opt=("momentum", 0.005, 0.9),
                     ens=dict(optimizer=("momentum", 0.005, 0.9), adanet_lambda=0.01, adanet_beta=0.001,
                              use_bias=True, mixture_weight_type="vector")),
    # BASELINE configs[4] shape in small: depth 1..8 in one iteration (mixed-depth layer waves, deep dZ ping-pong)
    "deep": dict(data=("tabular", 8192, 100, 10, 31), cfgs=[(1, 32), (8, 32), (4, 48), (6, 24), (2, 40)], B=256, steps=25,
                 iters=2, opt=("sgd", 0.01), ens=ENS),
    # MATRIX mixture weights (weighted.py:424-453): W_k [D_k, C] from zeros on every member's last layer, with bias
    "matrix": dict(data=("tabular", 8192, 100, 10, 77), cfgs=[(1, 64), (2, 96)], B=256, steps=30, iters=2,
                   opt=("sgd", 0.02),
                   ens=dict(optimizer=("sgd", 0.02), adanet_lambda=0.01, adanet_beta=0.001, use_bias=True,
                            mixture_weight_type="matrix")),
    # warm_start_mixture_weights (weighted.py:270-285,487-516): kept members + bias start from the previous ensemble's
    "warm_start": dict(data=("tabular", 8192, 100, 10, 12), cfgs=[(1, 48), (2, 48)], B=256, steps=25, iters=3,
                       opt=("sgd", 0.02),
                       ens=dict(optimizer=("sgd", 0.05), adanet_lambda=0.01, adanet_beta=0.001, use_bias=True,
                                mixture_weight_type="vector", warm_start_mixture_weights=True)),
    "warm_start_matrix": dict(data=("tabular", 8192, 100, 10, 13), cfgs=[(1, 48), (2, 48)], B=256, steps=25, iters=2,
                              opt=("sgd", 0.02),
                              ens=dict(optimizer=("sgd", 0.02), adanet_lambda=0.01, adanet_beta=0.001, use_bias=True,
                                       mixture_weight_type="matrix", warm_start_mixture_weights=True)),
    "default_ensembler": dict(data=("tabular", 8192, 100, 10, 99), cfgs=[(1, 64), (2, 64)], B=256, steps=30, iters=2,
                              opt=("sgd", 0.01), ens=dict(optimizer=None)),
    "force_grow": dict(data=("tabular", 8192, 100, 10, 5), cfgs=[(1, 32), (2, 32)], B=256, steps=10, iters=3,
                       opt=("sgd", 0.01), ens=ENS, force_grow=True),
    "replay": dict(data=("tabular", 8192, 100, 10, 5), cfgs=[(1, 32), (2, 32)], B=256, steps=10, iters=3,
                   opt=("sgd", 0.01), ens=ENS, replay=[1, 2, 1]),
    "regression": dict(data=("regression", 4096, 20, 1, 8), cfgs=[(1, 32), (2, 32)], B=128, steps=40, iters=2,
                       opt=("sgd", 0.02), ens=ENS, head="mse"),
    # BASELINE configs[2] -- the workload bench.py is quoted on: the exact 8 candidates 100->H->H->10 with the bench's
    # optimizers, at B=4096 (B=32768: test_bench_workload_parity_full_batch)
    "bench_shape": dict(data=("tabular", 4096 * 8, 100, 10, 1234), cfgs=[(2, h) for h in (64, 128, 192, 256, 384, 512, 768, 1024)],
                        B=4096, steps=20, iters=1, opt=("sgd", 0.05), ens=ENS),
    # tf.layers.dropout(rate .25) after every hidden layer in TRAIN mode (simple_dnn.py:80-81); frozen members replay
    # without it; the keep mask is injected data shared with the oracle (dropout_keep_mask)
    "dropout": dict(data=("tabular", 8192, 100, 10, 41), cfgs=[(1, 64), (2, 48), (3, 40)], B=256, steps=30, iters=2,
                    opt=("sgd", 0.01), ens=ENS, dropout=(0.25, 7)),
    # edge cases: batch not a multiple of any tile, widths 3, single candidate, 3 classes
    "ragged": dict(data=("tabular", 1000, 7, 3, 3), cfgs=[(1, 3)], B=37, steps=15, iters=2, opt=("sgd", 0.05),
                   ens=ENS),
}


def _oracle_run(cfg, perm=None):
  kind, n, d, c, seed = cfg["data"]
  x, y = _data(kind, n, d, c, seed)
  if perm is not None:
    x = np.ascontiguousarray(x[:, perm])

  def space(t, frozen):
    specs = pu.make_specs(cfg["cfgs"], d, c, t, cfg["opt"], dropout=cfg.get("dropout"))[0]
    if perm is not None:
      for s in specs:
        s.ws[0] = np.ascontiguousarray(s.ws[0][perm])
    return specs

  res, _ = orc.run_adanet(space, x, y, cfg["B"], cfg["steps"], cfg["iters"], orc.EnsemblerSpec(**cfg["ens"]), c,
                          head=cfg.get("head", "softmax_xent"), force_grow=cfg.get("force_grow", False),
                          replay_indices=cfg.get("replay"))
  return res


def _max_trace_diff(a, b):
  worst = 0.0
  for ra, rb in zip(a, b):
    for name in ra.traces:
      for f in ("sub_loss", "ens_loss", "adanet_loss", "ema"):
        worst = max(worst, float(np.abs(np.asarray(ra.traces[name][f], np.float64) -
                                        np.asarray(rb.traces[name][f], np.float64)).max()))
  return worst


@pytest.mark.parametrize("name", sorted(CONFIGS))
def test_parity_configs_are_well_conditioned(name):
  """CPU: the oracle against itself (a) with permuted input-feature order (a pure summation-order
  change) and (b) with 2e-7 relative noise on every dense forward / weight gradient."""
  cfg = CONFIGS[name]
  d = cfg["data"][2]
  perm = np.random.default_rng(0).permutation(d)
  a, b = _oracle_run(cfg), _oracle_run(cfg, perm)
  sens = _max_trace_diff(a, b)
  assert [r.best_index for r in a] == [r.best_index for r in b]
  assert sens < SENS_TOL, "config %s is ill conditioned: oracle self-sensitivity %.3g" % (name, sens)
  for seed in (0, 1, 2):
    with pu.oracle_noise(2e-7, seed):
      c = _oracle_run(cfg)
    sens = _max_trace_diff(a, c)
    assert [r.best_index for r in a] == [r.best_index for r in c]
    assert sens < SENS_TOL, "config %s is ill conditioned: 2e-7 noise (seed %d) moves the oracle by %.3g" % (
        name, seed, sens)


def _engine_run(cfg, use_graph=True, multi_stream=True):
  from adanet_b200.core import engine as eng
  from adanet_b200.core import search as srch
  kind, n, d, c, seed = cfg["data"]
  x, y = _data(kind, n, d, c, seed)
  space = lambda t, frozen: pu.make_specs(cfg["cfgs"], d, c, t, cfg["opt"], dropout=cfg.get("dropout"))[1]
  s = srch.AdaNetSearch(space, eng.EnsemblerPlanSpec(**cfg["ens"]), d, c, cfg["B"], head=cfg.get("head", "softmax_xent"),
                        use_cuda_graph=use_graph, multi_stream=multi_stream, force_grow=cfg.get("force_grow", False),
                        replay_indices=cfg.get("replay"))
  reps = s.run(srch.consecutive_batches(x, y, cfg["B"]), cfg["steps"], cfg["iters"])
  return reps, s


def _check(o_res, reps, tol=TOL):
  worst = 0.0
  for o, r in zip(o_res, reps):
    assert r.candidate_names == o.candidate_names
    for name, tr in o.traces.items():
      for f in ("sub_loss", "ens_loss", "adanet_loss", "ema"):
        want = np.asarray(tr[f], dtype=np.float64)
        got = r.traces[name][f].astype(np.float64)
        assert got.shape == want.shape
        err = np.abs(got - want).max()
        worst = max(worst, err)
        assert err < tol, "iteration %d %s/%s: max abs err %.3g (first step err %.3g)" % (
            o.iteration, name, f, err, abs(got[0] - want[0]))
    assert r.best_index == o.best_index, (r.ema_losses, o.ema_losses)
    assert r.architecture == o.architecture
    np.testing.assert_allclose(r.ema_losses, o.ema_losses, atol=tol)
  return worst


@pytest.mark.gpu
@pytest.mark.parametrize("path", ["simt", "auto"])
@pytest.mark.parametrize("name", sorted(CONFIGS))
def test_iteration_parity(built_lib, name, path):
  from adanet_b200 import _lib
  cfg = CONFIGS[name]
  if name in ("matrix", "warm_start_matrix", "dropout") and path == "simt":
    pytest.skip("MATRIX mixture weights and dropout run on the plane path only")
  _lib.set_dense_path(_lib.PATH_SIMT if path == "simt" else _lib.PATH_AUTO)
  try:
    o = _oracle_run(cfg)
    r, s = _engine_run(cfg)
    worst = _check(o, r)
    print("%s[%s] worst per-step abs err %.3g" % (name, path, worst))
    assert len(s.frozen) == len(r[-1].architecture)
    if name == "default_ensembler":
      # weighted.py:612-613: optimizer None -> no_op, weights stay 1/N; lambda=beta=0 -> reg exactly 0
      np.testing.assert_allclose(r[-1].mixture_weights, np.full_like(r[-1].mixture_weights, 1.0 / len(r[-1].architecture)))
      for tr in r[0].traces.values():
        np.testing.assert_array_equal(tr["ens_loss"], tr["adanet_loss"])
    if name == "force_grow":
      assert len(r[-1].architecture) == 3   # a subnetwork is added every iteration (estimator_test.py:3002-3078)
    if name == "replay":
      assert [rep.best_index for rep in r] == [1, 2, 1]   # estimator_test.py:3235-3311
  finally:
    _lib.set_dense_path(_lib.PATH_AUTO)


@pytest.mark.gpu
def test_bench_workload_parity_full_batch(built_lib):
  """bench.py's configuration itself (BASELINE configs[2]: 8 candidates 100->H->H->10, H in 64..1024, B=32768, SGD .05 /
  mixture SGD .01, lambda .01, beta .001) against the oracle: per-step losses of every candidate within 1e-5 and
  the same winner.  5 steps (the oracle needs ~3 s per step at this size)."""
  cfg = dict(data=("tabular", 32768 * 5, 100, 10, 1234), cfgs=[(2, h) for h in (64, 128, 192, 256, 384, 512, 768, 1024)],
             B=32768, steps=5, iters=1, opt=("sgd", 0.05), ens=ENS)
  o = _oracle_run(cfg)
  r, _ = _engine_run(cfg)
  worst = _check(o, r)
  print("bench workload B=32768 worst per-step abs err %.3g" % worst)


@pytest.mark.gpu
def test_bench_dump_outputs_hold_the_last_step(built_lib, tmp_path):
  """bench.py --dump-outputs writes the plan's state after its last step, that step's loss row and the logits of
  its forward pass: the subnetwork loss recomputed from the dumped logits and labels is the dumped one."""
  import bench
  from adanet_b200.core import engine as eng
  from adanet_b200.core import search as srch
  B, D, C, steps = 256, 100, 10, 3
  x, y = orc.make_tabular(B * 4, D, C, seed=5)
  s = srch.AdaNetSearch(lambda t, frozen: pu.make_specs([(1, 64), (2, 128)], D, C, t, ("sgd", 0.05))[1],
                        eng.EnsemblerPlanSpec(**ENS), D, C, B, keep_traces=False)
  plan = s.build_iteration()
  batches = srch.consecutive_batches(x, y, B)
  for _ in range(steps):
    plan.train_step(*next(batches))
  bench.dump_outputs(plan, str(tmp_path))
  last = plan.last_losses()
  labels = y[(steps - 1) * B:steps * B]
  for k, c in enumerate(plan.candidates):
    def load(key):
      a = np.load(str(tmp_path / ("%s.%s.npy" % (c.spec.name, key))))
      assert a.dtype in (np.float32, np.float64)
      return a
    for key, want in c.state_dict().items():
      if key != "trace":
        np.testing.assert_array_equal(load(key), want)
    np.testing.assert_array_equal(load("losses"), last[k])
    logits = load("logits").astype(np.float64)
    assert logits.shape == (B, C)
    z = logits - logits.max(axis=1, keepdims=True)
    xent = np.mean(np.log(np.exp(z).sum(axis=1)) - z[np.arange(B), labels])
    assert abs(xent - last[k][0]) < 1e-5


@pytest.mark.gpu
def test_config5_sweep_at_real_widths(built_lib):
  """BASELINE configs[4] at its real size for one iteration: 32 candidates, depth 1..8 x width {128,256,512,1024},
  B=4096 (241 MFLOP per example summed over the candidates), 3 steps against the oracle."""
  cfgs = [(l, h) for l in range(1, 9) for h in (128, 256, 512, 1024)]
  cfg = dict(data=("tabular", 4096 * 3, 100, 10, 1234), cfgs=cfgs, B=4096, steps=3, iters=1, opt=("sgd", 0.01), ens=ENS)
  o = _oracle_run(cfg)
  r, _ = _engine_run(cfg)
  worst = _check(o, r)
  print("configs[4] 32-candidate sweep worst per-step abs err %.3g" % worst)


# BASELINE configs[1] on the data SURVEY.md 8d specifies, X ~ U[0,1) UNCENTRED: every feature has mean 0.5, so the
# first-layer pre-activations share a large common component and SGD at lr 0.05 amplifies rounding differences --
# the oracle run against itself with a permuted feature order (a pure change of summation order) already differs by
# ~2e-4 after 40 steps (module docstring).  1e-5 is therefore not a property of ANY fp32 implementation there; what
# is checked is the first steps at 1e-5 (before amplification), the whole trace at a bound a few times the
# oracle's own sensitivity, and identical selection.
UNCENTRED_TOL = 2e-3


@pytest.mark.gpu
def test_config2_uncentred_data(built_lib):
  cfg = dict(CONFIGS["config2"], data=("uniform", 8192, 784, 10, 2234))
  o = _oracle_run(cfg)
  perm = np.random.default_rng(0).permutation(784)
  sens = _max_trace_diff(o, _oracle_run(cfg, perm))
  r, _ = _engine_run(cfg)
  worst = _check(o, r, tol=UNCENTRED_TOL)
  early = 0.0
  for name, tr in o[0].traces.items():
    for f in ("sub_loss", "adanet_loss"):
      early = max(early, float(np.abs(r[0].traces[name][f][:3].astype(np.float64) - np.asarray(tr[f][:3], np.float64)).max()))
  print("config2 uncentred: worst %.3g (oracle self-sensitivity %.3g), first 3 steps %.3g" % (worst, sens, early))
  assert early < TOL
  assert worst < max(10 * sens, 1e-4)


@pytest.mark.gpu
def test_fp16_plane_overflow_falls_back_to_tf32_planes(built_lib):
  """A feature column of magnitude 3e5 does not fit the fp16 split planes: the input split raises the sticky flag, the
  search discards the iteration, switches the process to TF32 planes and trains it again (core/search.py
  restart_on_tf32_if_overflowed) -- the reported traces are those of the TF32 run and match the oracle.  (The
  subnetworks' weights for that column are scaled down and their optimizer is frozen, so the run itself is benign;
  the mixture weights still train.)"""
  from adanet_b200 import _lib
  from adanet_b200.core import engine as eng
  from adanet_b200.core import search as srch
  if _lib.plane_format() != _lib.PLANES_F16:
    pytest.skip("needs the fp16 plane format as the starting point")
  d, c, B, steps, iters = 100, 10, 256, 10, 2
  x, y = orc.make_tabular(4096, d, c, seed=61)
  x = x.copy()
  x[:, 3] *= np.float32(3e5)
  cfgs = [(1, 32), (2, 24)]

  def space(which):
    def fn(t, frozen):
      specs = pu.make_specs(cfgs, d, c, t, ("sgd", 0.0))[which]
      for sp in specs:
        sp.ws[0][3, :] *= np.float32(1e-5)
      return specs
    return fn

  o, _ = orc.run_adanet(space(0), x, y, B, steps, iters, orc.EnsemblerSpec(**ENS), c)
  s = srch.AdaNetSearch(space(1), eng.EnsemblerPlanSpec(**ENS), d, c, B)
  reps = s.run(srch.consecutive_batches(x, y, B), steps, iters)
  assert s.tf32_fallbacks == 1 and _lib.plane_format() == _lib.PLANES_TF32
  # the re-run consumed the batches that followed the discarded attempt: compare with the oracle started there
  o2, _ = orc.run_adanet(space(0), np.roll(x, -steps * B, axis=0), np.roll(y, -steps * B), B, steps, iters,
                         orc.EnsemblerSpec(**ENS), c)
  worst = _check(o2, reps)
  print("fallback run worst per-step abs err %.3g" % worst)
  assert all(np.isfinite(r.ema_losses).all() for r in reps)


@pytest.mark.gpu
def test_eager_launches_match_cuda_graph(built_lib):
  """Plain stream launches (no graph, single stream) and the captured multi-stream graph agree bit for bit."""
  cfg = CONFIGS["config2"]
  a, _ = _engine_run(cfg, use_graph=False, multi_stream=False)
  b, _ = _engine_run(cfg, use_graph=True, multi_stream=True)
  for ra, rb in zip(a, b):
    for name in ra.traces:
      for f in ("sub_loss", "ens_loss", "adanet_loss", "ema"):
        np.testing.assert_array_equal(ra.traces[name][f], rb.traces[name][f])
    assert ra.best_index == rb.best_index


@pytest.mark.gpu
def test_full_size_properties(built_lib):
  """BASELINE-size step (B=32768, H=1024) checked through size-independent properties:
  determinism (two fresh runs bit-identical), exact power-of-two linearity of the dense
  backward, and the ReLU-mask structure of dX."""
  import torch
  from adanet_b200 import _lib
  from adanet_b200.core import engine as eng
  from adanet_b200.core import search as srch
  B, D, C = 32768, 100, 10
  x, y = orc.make_tabular(B * 2, D, C, seed=1234)
  losses = []
  for _ in range(2):
    s = srch.AdaNetSearch(lambda t, f: pu.make_specs([(2, 1024)], D, C, t, ("sgd", 0.05))[1],
                          eng.EnsemblerPlanSpec(optimizer=("sgd", 0.01), adanet_lambda=0.01), D, C, B)
    reps = s.run(srch.consecutive_batches(x, y, B), 2, 1)
    losses.append(next(iter(reps[0].traces.values()))["sub_loss"].copy())
  np.testing.assert_array_equal(losses[0], losses[1])
  assert np.isfinite(losses[0]).all()
  lib = _lib.load()
  I, O = 1024, 1024
  rng = np.random.default_rng(0)
  xd = torch.as_tensor(np.maximum(rng.standard_normal((B, I)), 0).astype(np.float32)).cuda()
  wd = torch.as_tensor(orc.glorot_uniform(rng, I, O)).cuda()
  dz = torch.as_tensor((rng.standard_normal((B, O)) / B).astype(np.float32)).cuda()
  ws_bytes = _lib.query(_lib.Q_DENSE_BWD_WS, B, I, O)
  ws = torch.empty((ws_bytes,), dtype=torch.uint8, device="cuda")
  outs = []
  for scale in (1.0, 2.0):
    d = dz * scale
    dw = torch.empty((I, O), device="cuda")
    db = torch.empty((O,), device="cuda")
    dx = torch.empty((B, I), device="cuda")
    _lib.check(lib.adn_dense_bwd(xd.data_ptr(), wd.data_ptr(), d.data_ptr(), dx.data_ptr(), dw.data_ptr(), db.data_ptr(),
                                 B, I, O, 1, ws.data_ptr(), ws_bytes, torch.cuda.current_stream().cuda_stream), "bwd")
    outs.append((dw, db, dx))
  for a, b in zip(outs[0], outs[1]):
    assert torch.equal(a * 2.0, b)
  assert float(outs[0][2][xd == 0].abs().max()) == 0.0
  # spot-check 64 random dW entries against fp64
  ii = rng.integers(0, I, 64)
  oo = rng.integers(0, O, 64)
  xs = xd[:, torch.as_tensor(ii).cuda()].double()
  ds = dz[:, torch.as_tensor(oo).cuda()].double()
  want = (xs * ds).sum(0).cpu().numpy()
  got = outs[0][0][torch.as_tensor(ii).cuda(), torch.as_tensor(oo).cuda()].cpu().numpy()
  scale = float((xs.abs() * ds.abs()).sum(0).max())
  assert np.abs(got - want).max() <= 3e-6 * scale


STRATEGY_CASES = {
    # adanet/ensemble/strategy.py:79-117: several candidate ensembles share the iteration's subnetworks
    "all_solo_grow": dict(strategies=("all", "solo", "grow"), ens=dict(optimizer=("sgd", 0.01), adanet_lambda=0.01,
                                                                       adanet_beta=0.001, use_bias=True)),
    "solo_only": dict(strategies=("solo",), ens=ENS),
    # data seed 22: with seed 21 iteration 2 / step 14 sits on a discrete boundary (a ReLU flip that MATRIX weights see
    # through the last layers): the ORACLE itself jumps by 2.7e-5 there under 2e-7 relative noise on its GEMMs
    # (test_strategy_cases_are_well_conditioned keeps every case honest)
    "all_matrix": dict(strategies=("all",), seed=22, ens=dict(optimizer=("sgd", 0.02), adanet_lambda=0.01, use_bias=True,
                                                              mixture_weight_type="matrix")),
    # adanet/ensemble/mean.py:92-135: mean of the new subnetworks' logits, nothing trained
    "mean_grow": dict(strategies=("grow",), mean=True, ens=dict(optimizer=None)),
    "mean_all": dict(strategies=("all",), mean=True, ens=dict(optimizer=None)),
}


def _strategy_oracle(case):
  d, c, B, steps, iters = 100, 10, 256, 20, 3
  x, y = orc.make_tabular(8192, d, c, seed=case.get("seed", 21))
  cfgs = [(1, 48), (2, 32), (3, 24)]
  o, _ = orc.run_adanet_strategies(lambda t, frozen: pu.make_specs(cfgs, d, c, t, ("sgd", 0.02))[0], x, y, B, steps, iters,
                                   orc.EnsemblerSpec(**case["ens"]), c, strategies=case["strategies"],
                                   mean_ensembler=case.get("mean", False))
  return o, (d, c, B, steps, iters, x, y, cfgs)


@pytest.mark.parametrize("name", sorted(STRATEGY_CASES))
def test_strategy_cases_are_well_conditioned(name):
  """CPU: every strategy parity case against itself under 2e-7 relative noise on the oracle's GEMMs (see
  test_parity_configs_are_well_conditioned)."""
  a, _ = _strategy_oracle(STRATEGY_CASES[name])
  for seed in (0, 1):
    with pu.oracle_noise(2e-7, seed):
      b, _ = _strategy_oracle(STRATEGY_CASES[name])
    assert [r.best_index for r in a] == [r.best_index for r in b]
    worst = 0.0
    for ra, rb in zip(a, b):
      for cname in ra.traces:
        for f in ("sub_loss", "ens_loss", "adanet_loss", "ema"):
          e = np.abs(np.asarray(ra.traces[cname][f], np.float64) - np.asarray(rb.traces[cname][f], np.float64))
          worst = max(worst, float(np.nanmax(e)) if not np.all(np.isnan(e)) else 0.0)
    assert worst < SENS_TOL, "strategy case %s is ill conditioned: 2e-7 noise moves the oracle by %.3g" % (name, worst)


@pytest.mark.gpu
@pytest.mark.parametrize("name", sorted(STRATEGY_CASES))
def test_strategy_parity(built_lib, name):
  from adanet_b200.core import engine as eng
  from adanet_b200.core import search as srch
  case = STRATEGY_CASES[name]
  o, (d, c, B, steps, iters, x, y, cfgs) = _strategy_oracle(case)
  e_ens = eng.EnsemblerPlanSpec(kind="mean" if case.get("mean") else "complexity_regularized", **case["ens"])
  s = srch.AdaNetSearch(lambda t, frozen: pu.make_specs(cfgs, d, c, t, ("sgd", 0.02))[1], e_ens, d, c, B,
                        strategies=case["strategies"])
  reps = s.run(srch.consecutive_batches(x, y, B), steps, iters)
  for ro, r in zip(o, reps):
    assert r.candidate_names == ro.candidate_names
    for cname, tr in ro.traces.items():
      for f in ("sub_loss", "ens_loss", "adanet_loss", "ema"):
        np.testing.assert_allclose(r.traces[cname][f], np.asarray(tr[f], dtype=np.float64), atol=TOL, rtol=0, equal_nan=True)
    assert r.best_index == ro.best_index and r.architecture == ro.architecture
    np.testing.assert_allclose(r.ema_losses, ro.ema_losses, atol=TOL)
  assert [m.name for m in s.frozen] == [n for _, n in o[-1].architecture]


@pytest.mark.gpu
@pytest.mark.parametrize("strategies", [("grow",), ("all", "grow")])
def test_two_ensemblers_parity(built_lib, strategies):
  """Several ensemblers per iteration (adanet/core/iteration.py:683-693): every strategy candidate is built by a
  trained ComplexityRegularizedEnsembler (VECTOR weights, bias, warm start), by a second one with other settings and
  by the MeanEnsembler; candidates are named t{t}_{candidate}_{ensembler}, the subnetworks are trained once, and only
  the heads of the ensembler that built the previous winner warm-start from it."""
  from adanet_b200.core import engine as eng
  from adanet_b200.core import search as srch
  d, c, B, steps, iters = 100, 10, 256, 15, 3
  x, y = orc.make_tabular(8192, d, c, seed=23)
  cfgs = [(1, 48), (2, 32)]
  e1 = dict(optimizer=("sgd", 0.05), adanet_lambda=0.01, adanet_beta=0.001, use_bias=True, mixture_weight_type="vector",
            warm_start_mixture_weights=True, name="cr_vector")
  e2 = dict(optimizer=("sgd", 0.01), adanet_lambda=0.1, name="cr_scalar")
  e3 = dict(optimizer=None, name="mean", kind="mean")
  o, _ = orc.run_adanet_strategies(lambda t, frozen: pu.make_specs(cfgs, d, c, t, ("sgd", 0.02))[0], x, y, B, steps, iters,
                                   [orc.EnsemblerSpec(**e) for e in (e1, e2, e3)], c, strategies=strategies)
  s = srch.AdaNetSearch(lambda t, frozen: pu.make_specs(cfgs, d, c, t, ("sgd", 0.02))[1],
                        [eng.EnsemblerPlanSpec(**e) for e in (e1, e2, e3)], d, c, B, strategies=strategies)
  reps = s.run(srch.consecutive_batches(x, y, B), steps, iters)
  n_cand = (len(cfgs) if "grow" in strategies else 0) + (1 if "all" in strategies else 0)
  assert len(reps[0].candidate_names) == 3 * n_cand
  assert reps[0].candidate_names[:3] == ["t0_%s_%s" % ("all" if strategies[0] == "all" else "1_layer_dnn_grow", n)
                                         for n in ("cr_vector", "cr_scalar", "mean")]
  for ro, r in zip(o, reps):
    assert r.candidate_names == ro.candidate_names
    for cname, tr in ro.traces.items():
      for f in ("sub_loss", "ens_loss", "adanet_loss", "ema"):
        np.testing.assert_allclose(r.traces[cname][f], np.asarray(tr[f], dtype=np.float64), atol=TOL, rtol=0, equal_nan=True,
                                   err_msg="%s/%s" % (cname, f))
    assert r.best_index == ro.best_index and r.architecture == ro.architecture
    np.testing.assert_allclose(r.ema_losses, ro.ema_losses, atol=TOL)


@pytest.mark.gpu
def test_partial_pruning_parity(built_lib):
  """A custom Strategy that keeps only part of the previous ensemble (adanet/core/ensemble_builder.py:367-388): next
  to the plain `grow` candidates, `prune_oldest` drops the oldest member and `keep_newest` keeps only the newest one,
  with VECTOR weights warm-started for exactly the members that stay."""
  from adanet_b200.core import engine as eng
  from adanet_b200.core import search as srch
  d, c, B, steps, iters = 100, 10, 256, 12, 4
  x, y = orc.make_tabular(8192, d, c, seed=29)
  cfgs = [(1, 40), (2, 24)]
  ens = dict(optimizer=("sgd", 0.05), adanet_lambda=0.02, adanet_beta=0.001, use_bias=True, mixture_weight_type="vector",
             warm_start_mixture_weights=True)

  def cands(t, names, n_frozen):
    out = [("%s_grow" % n, [i], True) for i, n in enumerate(names)]
    if n_frozen >= 2:
      out.append(("%s_prune_oldest" % names[0], [0], list(range(1, n_frozen))))
      out.append(("%s_keep_newest" % names[1], [1], [n_frozen - 1]))
    return out

  o, o_frozen = orc.run_adanet_strategies(lambda t, frozen: pu.make_specs(cfgs, d, c, t, ("sgd", 0.02))[0], x, y, B, steps, iters,
                                          orc.EnsemblerSpec(**ens), c, candidates_fn=cands, force_grow=True)
  s = srch.AdaNetSearch(lambda t, frozen: pu.make_specs(cfgs, d, c, t, ("sgd", 0.02))[1], eng.EnsemblerPlanSpec(**ens), d, c, B,
                        force_grow=True,
                        candidates_fn=lambda specs, n_frozen: [srch.EnsembleCandidate(n, b, k) for n, b, k in
                                                               cands(None, [sp.name for sp in specs], n_frozen)])
  reps = s.run(srch.consecutive_batches(x, y, B), steps, iters)
  assert any("prune_oldest" in n for n in reps[-1].candidate_names)
  for ro, r in zip(o, reps):
    assert r.candidate_names == ro.candidate_names
    for cname, tr in ro.traces.items():
      for f in ("sub_loss", "ens_loss", "adanet_loss", "ema"):
        np.testing.assert_allclose(r.traces[cname][f], np.asarray(tr[f], dtype=np.float64), atol=TOL, rtol=0, err_msg="%s/%s" % (cname, f))
    assert r.best_index == ro.best_index and r.architecture == ro.architecture
  assert [m.name for m in s.frozen] == [m.name for m in o_frozen]


# BASELINE config 4: simple_cnn subnetworks on CIFAR-shaped synthetic images (customizing_adanet.ipynb: SimpleCNNBuilder,
# Momentum(0.9) under cosine decay of the iteration step, mixture weights not trained, adanet_loss_decay=.99)
CNN_CASES = {
    "cifar_shaped": dict(image=(32, 32, 3), filters=16, hidden=64, seeds=(0, 1, 2, 3), n=1024, B=64, steps=12, iters=2,
                         opt=lambda steps: ("momentum_cosine", 0.003, 0.9, steps)),
    "mnist_shaped_sgd": dict(image=(28, 28, 1), filters=16, hidden=32, seeds=(0, 1), n=600, B=50, steps=10, iters=3,
                             opt=lambda steps: ("sgd", 0.02)),
    "wide_stem": dict(image=(12, 12, 3), filters=32, hidden=24, seeds=(5,), n=512, B=128, steps=8, iters=2,
                      opt=lambda steps: ("momentum", 0.02, 0.9)),
}


def _cnn_data(case, classes=10):
  h, w, c = case["image"]
  # SURVEY.md 8d: X ~ U[0,1) NHWC, labels randint(0, 10); centred like the tutorial's `images / 127.5 - 1`
  # preprocessing so that the short parity runs train smoothly (no loss spikes amplifying rounding differences)
  rng = np.random.default_rng(3234)
  return (rng.uniform(0, 1, (case["n"], h, w, c)) * 2 - 1).astype(np.float32), rng.integers(0, classes, case["n"])


@pytest.mark.gpu
@pytest.mark.parametrize("name", sorted(CNN_CASES))
def test_simple_cnn_parity(built_lib, name):
  from adanet_b200.core import engine as eng
  from adanet_b200.core import search as srch
  case = CNN_CASES[name]
  C = 10
  x, y = _cnn_data(case, C)
  opt = case["opt"](case["steps"])
  mk = lambda t, which: pu.make_cnn_specs(case["seeds"], case["image"], case["filters"], case["hidden"], C, t, opt)[which]
  o, o_frozen = orc.run_adanet(lambda t, frozen: mk(t, 0), x, y, case["B"], case["steps"], case["iters"], orc.EnsemblerSpec(),
                               C, adanet_loss_decay=0.99)
  s = srch.AdaNetSearch(lambda t, frozen: mk(t, 1), eng.EnsemblerPlanSpec(), int(np.prod(case["image"])), C, case["B"],
                        adanet_loss_decay=0.99)
  reps = s.run(srch.consecutive_batches(x, y, case["B"]), case["steps"], case["iters"])
  worst = _check(o, reps)
  print("%s worst per-step abs err %.3g" % (name, worst))
  # the trained stem and dense weights of the selected members
  for m, mo in zip(s.frozen, o_frozen):
    ws, bs = m.numpy_params()
    assert ws[0].ndim == 4
    for a, b in zip(ws + bs, list(mo.ws) + list(mo.bs)):
      np.testing.assert_allclose(a, b, atol=5e-5)


@pytest.mark.gpu
@pytest.mark.parametrize("opt", [("sgd", 0.05), ("adam", 0.003)])
def test_bagged_subnetworks_parity(built_lib, opt):
  """Bagging (adanet/autoensemble/common.py:63-93,151-180): candidates 0 and 2 train on minibatches of their own
  input (one step BEFORE the main pass, :43-56), candidate 1 on the shared minibatch; every ensemble head reads the
  forwards on the shared minibatch."""
  from adanet_b200.core import engine as eng
  from adanet_b200.core import search as srch
  d, c, B, steps, iters = 100, 10, 256, 15, 3
  x, y = orc.make_tabular(8192, d, c, seed=51)
  bags = {0: orc.make_tabular(B * 4, d, c, seed=52), 2: orc.make_tabular(B * 6, d, c, seed=53)}
  cfgs = [(1, 48), (2, 32), (2, 64)]
  ens = dict(optimizer=("sgd", 0.01), adanet_lambda=0.01, adanet_beta=0.001)

  def o_space(t, frozen):
    specs = pu.make_specs(cfgs, d, c, t, opt)[0]
    for i, data in bags.items():
      specs[i].own_data = data
    return specs

  def e_space(t, frozen):
    specs = pu.make_specs(cfgs, d, c, t, opt)[1]
    for i in bags:
      specs[i].own_input = True
    return specs

  want, _ = orc.run_adanet(o_space, x, y, B, steps, iters, orc.EnsemblerSpec(**ens), c)
  s = srch.AdaNetSearch(e_space, eng.EnsemblerPlanSpec(**ens), d, c, B)
  batches = srch.consecutive_batches(x, y, B)
  for t in range(iters):
    plan = s.build_iteration()
    if t == 0:
      with pytest.raises(ValueError):      # a bagged subnetwork without its minibatch is an error, not a silent reuse
        plan.train_step(*next(srch.consecutive_batches(x, y, B)))
    for step in range(steps):
      own = {}
      for i, (xo, yo) in bags.items():
        o = (step % (xo.shape[0] // B)) * B
        own[i] = (xo[o:o + B], yo[o:o + B])
      plan.train_step(*next(batches), own_batches=own)
    s.finish_iteration()
  worst = _check(want, s.reports)
  print("bagging %s worst per-step abs err %.3g" % (opt[0], worst))
