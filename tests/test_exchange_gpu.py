"""(e) multi-GPU: NCCL all-to-all exchange + partial/exchange/final plan on >= 2 GPUs of one box."""
import os
import subprocess
import sys

import pytest

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _ngpus():
    try:
        out = subprocess.run(["nvidia-smi", "-L"], capture_output=True, text=True, timeout=30).stdout
        return len([line for line in out.splitlines() if line.startswith("GPU ")])
    except Exception:
        return 0


def test_exchange_single_rank_is_identity(b2):
    """world = 1: the exchange degenerates to partition + (self) copy — runs on the 1-GPU box"""
    import numpy as np
    from oracle import spark_cpu as O
    from oracle import spark_hash as H
    from tests import datagen as G
    rng = np.random.default_rng(2)
    cols = [G.gen_column(rng, (O.INT64, 0, 0), 5000, distinct=100), G.gen_column(rng, (O.STRING, 0, 0), 5000), G.gen_column(rng, (O.DECIMAL128, 30, 2), 5000)]
    comm = b2.Comm(b2.Comm.unique_id(), 0, 1)
    part, offs = b2.hash_partition(G.to_b2_table(b2, cols), [0], 1)
    got = comm.exchange(part, offs)
    exp, _ = H.hash_partition(cols, [0], 1)
    for i in range(3):
        G.assert_col_equal(got.column(i), exp[i])
    comm.close()


@pytest.mark.skipif(_ngpus() < 2, reason="needs 2 GPUs")
def test_exchange_two_ranks():
    n = min(_ngpus(), 4)
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", str(n), "--master-addr", "127.0.0.1",
                        "--master-port", "29517", os.path.join(ROOT, "scripts", "exchange_check.py")], capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-3000:]
    assert "exchange_check ok" in r.stdout
