"""CPU tests of the host-side logic that needs no GPU: gin-compatible config surface, TF SAME padding
arithmetic, dataset surface, metric math against the oracle and the reference's golden FID."""
import json
import os

import numpy as np
import pytest

from compare_gan_b200 import datasets
from compare_gan_b200 import gin_lite as gin
from compare_gan_b200 import kernels as K
from compare_gan_b200.metrics import fid_score, inception_score, kid_score
from oracle import metrics as ometrics
from oracle import tf_ops as T


def test_same_padding_matches_oracle():
  for n in range(1, 20):
    for k in (1, 3, 4, 5):
      for s in (1, 2):
        out, before, _ = T._same_pads(n, k, s)
        assert K.same_pad(n, k, s) == (out, before)


def test_gin_bindings_scopes_and_refs():
  gin.clear_config()

  @gin.configurable("hp_test_fn", module="tmod")
  def f(a, b=2, c=gin.REQUIRED):
    return a, b, c
  with pytest.raises(ValueError):
    f(1)
  gin.parse_config("hp_test_fn.c = 7\nscope1/hp_test_fn.b = 5\nX = 3\nhp_test_fn.b = %X")
  assert f(1) == (1, 3, 7)
  with gin.config_scope("scope1"):
    assert f(1) == (1, 5, 7)
  assert f(1, b=9) == (1, 9, 7)
  with pytest.raises(ValueError):
    gin.parse_config("hp_test_fn.nope = 1")
  gin.clear_config()


def test_example_config_parses_and_binds():
  from compare_gan_b200.gans import modular_gan  # noqa: F401
  from compare_gan_b200 import runner_lib  # noqa: F401
  gin.clear_config()
  # a literal copy of the bindings of example_configs/resnet_cifar10.gin (the file itself lives in the read-only
  # reference tree, which is absent on the GPU box)
  text = """
dataset.name = "cifar10"
options.architecture = "resnet_cifar_arch"
options.batch_size = 64
options.gan_class = @ModularGAN
options.lamba = 1
options.training_steps = 40000
options.z_dim = 128
G.batch_norm_fn = @batch_norm
standardize_batch.decay = 0.9
standardize_batch.epsilon = 1e-5
options.disc_iters = 5
D.spectral_norm = True
loss.fn = @non_saturating
penalty.fn = @no_penalty
ModularGAN.g_lr = 0.0002
ModularGAN.g_optimizer_fn = @tf.train.AdamOptimizer
tf.train.AdamOptimizer.beta1 = 0.5
tf.train.AdamOptimizer.beta2 = 0.999
"""
  gin.parse_config(text)
  opts = runner_lib.get_options_dict()
  assert opts["architecture"] == "resnet_cifar_arch" and opts["disc_iters"] == 5 and opts["lambda"] == 1
  assert opts["gan_class"] is modular_gan.ModularGAN
  assert gin.query_parameter("standardize_batch.decay") == 0.9
  # every example config the reference ships, restated in configs.py, must bind exactly the values the original file
  # binds: the golden holds the operative config of each original example_configs/*.gin as parsed by gin_lite
  from compare_gan_b200 import configs
  golden = json.load(open(os.path.join(os.path.dirname(__file__), "golden", "example_configs_operative.json")))
  for name, from_file in sorted(golden.items()):
    gin.clear_config()
    gin.parse_config(configs.CONFIGS[name])
    assert runner_lib.get_options_dict()["gan_class"] is modular_gan.ModularGAN
    assert gin.operative_config_str() == from_file, name
  gin.clear_config()


def test_dataset_surface():
  ds = datasets.get_dataset("cifar10")
  assert ds.image_shape == (32, 32, 3) and ds.num_classes == 10 and ds.eval_test_samples == 10000
  x = ds.sample_images(4)
  assert x.shape == (4, 32, 32, 3) and x.dtype == np.float32 and 0 <= x.min() and x.max() < 1
  assert datasets.get_dataset("imagenet_128").eval_test_samples == 50000
  with pytest.raises(ValueError):
    datasets.get_dataset("nope")


def test_fid_golden_and_streaming_moments():
  real = np.ones((100, 2)); real[:50, 0] = 2
  gen = np.ones((100, 2)) * 9; gen[50:, 0] = 2
  assert abs(fid_score.compute_fid_from_activations(gen, real) - 89.091) < 1e-4   # fid_score_test.py:31-40
  rng = np.random.RandomState(0)
  a = rng.randn(500, 12) * 2 + 1
  mu, sigma = fid_score.moments_from_sums(a.sum(0), a.T @ a, 500)
  np.testing.assert_allclose(mu, a.mean(0), rtol=1e-12)
  np.testing.assert_allclose(sigma, np.cov(a, rowvar=False), rtol=1e-9, atol=1e-12)


def test_is_and_kid_match_oracle():
  rng = np.random.RandomState(1)
  logits = rng.randn(200, 30)
  assert abs(inception_score.classifier_score_from_logits(logits) - ometrics.inception_score_from_logits(logits)) < 1e-12
  a, b = rng.randn(2100, 16), rng.randn(2500, 16) + 0.3
  assert abs(kid_score.kid(a, b, gram=lambda x, y: x @ y.T) - ometrics.kid(a, b)) < 1e-12


def test_inception_topology_statics():
  """The Inception-v3 layer table (2015 classify_image graph): 94 convolutions + logits, 2048-d pool_3, channel widths of
  every concat, and the FLOP count that bench.py reports per FID sample.  Pure host logic, no kernels."""
  from compare_gan_b200 import inception as inc
  from oracle import inception as oinc
  convs = inc.walk_convs()
  assert len(convs) == 94
  assert inc._channels(inc.SPEC, 3) == inc.POOL_DIM == 2048
  widths = [inc._channels([it], c) for it, c in ((inc.SPEC[7], 192), (inc.SPEC[8], 256), (inc.SPEC[10], 288),
                                                  (inc.SPEC[11], 768), (inc.SPEC[15], 768), (inc.SPEC[16], 1280))]
  assert widths == [256, 288, 768, 768, 1280, 2048]
  assert abs(inc.flops_per_image() / 1e9 - 11.43) < 0.01
  w = inc.synthetic_weights(0)
  assert len(w) == 2 * 94 + 2 and w["inception/logits/kernel"].shape == (2048, inc.NUM_CLASSES)
  # the CPU oracle walks the same table: same variable names and shapes
  assert sorted(w) == sorted(oinc.synthetic_weights(0)) if hasattr(oinc, "synthetic_weights") else True


def test_reference_arm_prints_contract_line():
  """`bench.py --impl reference` (the CPU restatement timed on the host cores) prints one JSON line with the contract's
  keys; runs a single bounded cycle here."""
  import json
  import os
  import subprocess
  import sys
  root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
  env = dict(os.environ, CGAN_REF_BATCH="4", CGAN_REF_SKIP_EVAL="1")      # the contract, not the number: a tiny sample
  out = subprocess.run([sys.executable, os.path.join(root, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "0"],
                       capture_output=True, text=True, timeout=900, cwd=root, env=env)
  assert out.returncode == 0, out.stderr[-2000:]
  line = json.loads(out.stdout.strip().splitlines()[-1])
  for key in ("impl", "metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
              "vs_baseline", "dtype", "data", "config", "cpu_baseline", "e2e"):
    assert key in line, key
  assert line["impl"] == "reference" and line["unit"] == "images/sec" and line["value"] > 0
  assert line["cpu_baseline"]["kind"] == "port" and line["cpu_baseline"]["cores"] >= 1
  assert line["e2e"]["h2d_bytes_per_step"] == 0 and line["e2e"]["d2h_bytes_per_step"] == 0


def test_task_manager_checkpoint_polling_and_csv(tmp_path):
  """TaskManager / TaskManagerWithCsvResults (reference runner_lib.py:114-232): unevaluated checkpoints come in step
  order, `eval_every_steps` keeps the positive multiples only, results land in scores.csv as checkpoint_path, step,
  sorted result keys, sorted operative-config keys (floats with three decimals), evaluated checkpoints are not offered
  again, and the config of a step is the latest operative_config saved at or before it."""
  import csv
  import os
  from compare_gan_b200 import runner_lib
  md = str(tmp_path)
  for step in (0, 5000, 10000, 12500):
    open(os.path.join(md, "model.ckpt-%d.npz" % step), "w").close()
  open(os.path.join(md, "operative_config-0.gin"), "w").write("options.batch_size = 64\nloss.fn = @hinge\n")
  open(os.path.join(md, "operative_config-10000.gin"), "w").write("options.batch_size = 128\nloss.fn = @hinge\n")
  tm = runner_lib.TaskManagerWithCsvResults(md)
  assert not tm.is_training_done()
  tm.mark_training_done()
  assert tm.is_training_done() and os.path.exists(os.path.join(md, "TRAIN_DONE"))
  todo = list(tm.unevaluated_checkpoints(timeout=0))
  assert [os.path.basename(c) for c in todo] == ["model.ckpt-0.npz", "model.ckpt-5000.npz", "model.ckpt-10000.npz",
                                                  "model.ckpt-12500.npz"]
  assert [os.path.basename(c) for c in tm.unevaluated_checkpoints(timeout=0, eval_every_steps=5000)] == [
      "model.ckpt-5000.npz", "model.ckpt-10000.npz"]
  tm.add_eval_result(todo[1], {"fid_score_mean": 12.34567, "inception_score_mean": 7.0, "note": "ok"}, -1.0)
  tm.add_eval_result(todo[2], {"fid_score_mean": 11.0, "inception_score_mean": 7.5, "note": "ok"}, -1.0)
  rows = list(csv.reader(open(os.path.join(md, "scores.csv"))))
  assert rows[0] == ["checkpoint_path", "step", "fid_score_mean", "inception_score_mean", "note", "loss.fn", "options.batch_size"]
  assert rows[1][1:] == ["5000", "12.346", "7.000", "ok", "@hinge", "64"]
  assert rows[2][1:] == ["10000", "11.000", "7.500", "ok", "@hinge", "128"]
  assert tm.get_checkpoints_with_results() == {todo[1], todo[2]}
  assert [os.path.basename(c) for c in tm.unevaluated_checkpoints(timeout=0)] == ["model.ckpt-0.npz", "model.ckpt-12500.npz"]
  # the base class keeps no results: everything stays unevaluated
  assert len(list(runner_lib.TaskManager(md).unevaluated_checkpoints(timeout=0))) == 4


def test_get_losses_routes_every_objective_to_the_fused_kernel(monkeypatch):
  """loss_lib.get_losses(fn=...) hands the logits to `kernels.gan_losses` with the objective's name, whatever the order
  in which the reference declares the (probability, logit) arguments (loss_lib.py:53-154)."""
  from compare_gan_b200 import kernels as K
  from compare_gan_b200.gans import loss_lib
  gin.clear_config()

  class T(object):
    shape = (4, 1)
  calls = []
  monkeypatch.setattr(K, "gan_losses", lambda kind, real, fake: calls.append((kind, real, fake)) or "out")
  d_real, d_fake, lr, lf = T(), T(), T(), T()
  for fn in (loss_lib.non_saturating, loss_lib.wasserstein, loss_lib.least_squares, loss_lib.hinge):
    assert loss_lib.get_losses(fn=fn, d_real=d_real, d_fake=d_fake, d_real_logits=lr, d_fake_logits=lf) == "out"
  assert [c[0] for c in calls] == ["non_saturating", "wasserstein", "least_squares", "hinge"]
  assert all(c[1] is lr and c[2] is lf for c in calls)
  gin.parse_config("loss.fn = @hinge")
  loss_lib.get_losses(d_real=d_real, d_fake=d_fake, d_real_logits=lr, d_fake_logits=lf)
  assert calls[-1][0] == "hinge"
  gin.clear_config()


def test_kid_follows_the_reference_block_estimator_for_unequal_sets():
  """metrics/kid_score.py:44-149 incl. its bin-size quirks: the host code (Gram matrices injected, so no GPU) against
  the line-by-line restatement in the oracle, for equal and unequal set sizes and several blocks."""
  from compare_gan_b200.metrics import kid_score
  from oracle import metrics as ometrics
  rng = np.random.RandomState(0)
  gram = lambda a, b: np.asarray(a, np.float64) @ np.asarray(b, np.float64).T
  for n_real, n_fake, block in [(12, 12, 1024), (50, 50, 16), (37, 41, 10), (64, 50, 16), (41, 37, 10), (200, 190, 64), (17, 23, 5)]:
    real, fake = rng.randn(n_real, 6), rng.randn(n_fake, 6) + 0.2
    np.testing.assert_allclose(kid_score.kid(fake, real, max_batch_size=block, gram=gram),
                               ometrics.kid(fake, real, max_batch_size=block), rtol=1e-12, err_msg=str((n_real, n_fake, block)))
