"""inference.evaluate() against a numpy restatement of the reference's EVAL metrics
(imagenet_train_eval.py:577-606): argmax accuracy, tf.nn.in_top_k(k=5) accuracy (ties at the boundary count as
inside, non-finite logits as outside) and the label-smoothed softmax cross-entropy, mean over the batch."""
import numpy as np
import pytest
import torch

from rigl_b200.inference import evaluate


def _numpy_metrics(z, labels, ls):
  z = z.astype(np.float64)
  n, k = z.shape
  top1 = np.mean(np.argmax(z, axis=1) == labels)
  t = z[np.arange(n), labels]
  top5 = np.mean([(np.sum(z[i] > t[i]) < 5) and np.isfinite(t[i]) for i in range(n)])
  soft = np.full((n, k), ls / k)
  soft[np.arange(n), labels] += 1.0 - ls
  m = z.max(axis=1, keepdims=True)
  logp = z - m - np.log(np.exp(z - m).sum(axis=1, keepdims=True))
  return top1, top5, np.mean(-(soft * logp).sum(axis=1))


@pytest.mark.parametrize('ls', [0.0, 0.1])
@pytest.mark.parametrize('dtype', [torch.float32, torch.bfloat16])
def test_evaluate_matches_numpy(ls, dtype):
  rng = np.random.RandomState(3)
  n, k = 300, 1000
  z = rng.standard_normal((n, k)).astype(np.float32) * 3
  labels = rng.randint(0, k, n)
  z[:50, labels[:50]] = z[:50].max(axis=1) + 1          # some rows right
  z[50:60] = np.round(z[50:60])                         # ties everywhere, incl. at the top-5 boundary
  z[60, 7] = np.nan                                     # a non-finite row
  labels[60] = 7
  zt = torch.from_numpy(z).to(dtype)
  got = evaluate(zt, torch.from_numpy(labels), ls)
  top1, top5, cross = _numpy_metrics(zt.float().numpy(), labels, ls)
  assert got['eval_accuracy'] == pytest.approx(top1, abs=1e-12)
  assert got['top_5_eval_accuracy'] == pytest.approx(top5, abs=1e-12)
  finite = np.isfinite(zt.float().numpy()).all(axis=1)
  assert not np.isfinite(got['cross_loss']) or not finite.all()
  got_f = evaluate(zt[torch.from_numpy(finite)], torch.from_numpy(labels[finite]), ls)
  want_f = _numpy_metrics(zt.float().numpy()[finite], labels[finite], ls)
  assert got_f['cross_loss'] == pytest.approx(want_f[2], rel=1e-12)


def test_evaluate_top5_ties_at_the_boundary_count_as_inside():
  z = torch.tensor([[5., 4., 3., 2., 1., 1., 1., 0.]])
  assert evaluate(z, torch.tensor([6]), 0.0)['top_5_eval_accuracy'] == 1.0   # 4 strictly larger
  assert evaluate(z, torch.tensor([7]), 0.0)['top_5_eval_accuracy'] == 0.0   # 7 strictly larger
  assert evaluate(z, torch.tensor([0]), 0.0)['eval_accuracy'] == 1.0
