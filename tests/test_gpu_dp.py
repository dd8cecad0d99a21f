"""Data-parallel correctness on real GPUs (needs >= 2; skipped on a one-GPU box): tools/dp_check.py under torchrun --
NCCL through the C-ABI communicator, DP step == single-GPU step on replicated data, bit-identical parameters across ranks on sharded
data, the reference's parameter averaging (J:325-330), sync_bn "W x N/W == 1 x N" (SURVEY.md 8e), bf16 gradient payload, and the
overlapped two-bucket all-reduce."""
import json
import os
import subprocess
import sys

import pytest

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _gpus():
    try:
        import torch
        return torch.cuda.device_count()
    except Exception:
        return 0


@pytest.mark.parametrize("overlap,p2p", [("0", "1"), ("0", "0"), ("1", "0")], ids=["peer-memory all-reduce", "nccl", "nccl two-bucket overlap"])
def test_two_rank_data_parallel(overlap, p2p, tmp_path):
    if _gpus() < 2:
        pytest.skip("needs two GPUs")
    env = dict(os.environ, B2G_AR_OVERLAP=overlap, B2G_P2P_AR=p2p)
    result = tmp_path / "dp_check_rank0.json"
    out = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr", "127.0.0.1", "--master-port", str(29531 + int(overlap) + 2 * int(p2p)),
                          os.path.join(ROOT, "tools", "dp_check.py"), str(result)], capture_output=True, text=True, timeout=900, env=env, cwd=ROOT)
    assert out.returncode == 0, out.stdout[-800:] + out.stderr[-1500:]
    d = json.loads(result.read_text())
    assert d["world"] == 2 and d["allreduce"] == "ok" and d["ar_overlap_env"] == overlap
    assert d["allreduce_transport"] == ("peer-memory kernel" if p2p == "1" else "nccl"), d["allreduce_transport"]
    for k in ("sharded_fp32_G_identical", "sharded_fp32_D_identical", "sharded_bf16_G_identical", "sharded_bf16_D_identical", "bf16_payload_G_identical", "bf16_payload_D_identical"):
        assert d[k] is True, k
    assert d["parameter_averaging_max_abs_err"] < 1e-6
    assert d["sync_bn"]["max_abs_dG"] < 4.5e-3 and d["sync_bn"]["max_abs_dD"] < 4.5e-3 and d["sync_bn"]["mean_abs_dG"] < 5e-5 and d["sync_bn"]["mean_abs_dD"] < 5e-5
