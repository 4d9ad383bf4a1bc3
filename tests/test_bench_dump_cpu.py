"""bench.py --dump-outputs: what it writes is float, bounded in size, and the same from run to run for the same model."""
import os

import numpy as np

import bench
import paddle_b200 as paddle
from paddle_b200 import models


def test_dump_outputs_is_bounded_and_repeatable(tmp_path, monkeypatch):
    paddle.seed(0)
    m = models.LlamaForCausalLM(models.llama_tiny(vocab_size=4096))
    ids = paddle.randint(0, 4096, [2, 17])
    loss = m(ids[:, :-1], ids[:, 1:])
    monkeypatch.setattr(bench, "DUMP_BUDGET_BYTES", 1 << 20)
    bench.dump_outputs(str(tmp_path / "a"), loss, m)
    bench.dump_outputs(str(tmp_path / "b"), loss.item(), m)
    names = sorted(os.listdir(tmp_path / "a"))
    params = dict(m.named_parameters())
    assert names == sorted(os.listdir(tmp_path / "b")) and names == sorted(["loss.npy"] + [f"{k}.npy" for k in params])
    per_param = (1 << 20) // 4 // len(params)
    total = 0
    for f in names:
        a, b = np.load(tmp_path / "a" / f), np.load(tmp_path / "b" / f)
        assert a.dtype in (np.float32, np.float64) and np.array_equal(a, b), f
        total += a.nbytes
        if f != "loss.npy":
            p = params[f[:-4]].numpy().astype(np.float32).reshape(-1)
            if p.size <= per_param:
                np.testing.assert_array_equal(a, p)
            else:
                assert a.size == per_param and np.isin(a, p).all()   # a sample of the parameter's own values
    assert total <= (1 << 20) + 8
    assert np.load(tmp_path / "a" / "loss.npy")[0] == np.float64(loss.item())
