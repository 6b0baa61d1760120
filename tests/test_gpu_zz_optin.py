"""The previous defaults and the measured-slower experiments stay in the tree as opt-in switches (profiles/r1_g_side_stream.md, r1_c_loop_kernel.md); this keeps them
parity-green: the golden-fixture and shape-variant parity tests are re-run in a child process with the switches on (they are read
once per process, hence the subprocess).  Runs last (file name) so that a regression here cannot hide the default path's results."""
import os
import subprocess
import sys

import pytest

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SELECT = "test_losses_hiddens_grads_match_reference_golden or test_shape_variants_against_oracle or cuda_graph or full_size or greedy"


@pytest.mark.parametrize("switches", [
    {"RECNET_SIDE": "0"},                                                     # everything on one stream (the pre-r2_h default)
    {"RECNET_PERSIST": "0", "RECNET_PERSIST_BWD": "0", "RECNET_PDL": "1"},    # kernel-per-phase reconstructor loops (the pre-r2 default) + programmatic dependent launch
    {"RECNET_OPTIMIZER": "torch", "RECNET_GEMM_PERSIST": "0"},               # r1_f optimiser, one-tile-per-CTA GEMMs
    {"RECNET_DEC_CLUSTER": "0", "RECNET_PERSIST_GLOBAL": "0", "RECNET_GREEDY_PF": "0"},   # decoder forward loop / global reconstructor / greedy on the kernel-per-phase paths
], ids=["one_stream", "kernel_per_phase+pdl", "r1_f_paths", "r1_loops"])
def test_opt_in_paths_stay_parity_green(switches):
    env = dict(os.environ, **switches)
    r = subprocess.run([sys.executable, "-m", "pytest", os.path.join(ROOT, "tests", "test_gpu_parity.py"), "-m", "gpu", "-q", "-x",
                        "-p", "no:cacheprovider", "-k", SELECT], capture_output=True, text=True, timeout=900, cwd=ROOT, env=env)
    tail = (r.stdout + r.stderr)[-3000:]
    assert r.returncode == 0, tail
    assert " passed" in r.stdout and " failed" not in r.stdout, tail


def test_nvlink_allreduce_kernel_matches_nccl_on_two_gpus():
    """csrc/allreduce.cuh under torchrun on 2 GPUs of this box: gradients averaged in place in symmetric memory (NVSwitch multicast path
    and peer-pointer path) equal NCCL's all_reduce(AVG) of a copy, and every rank ends with bitwise identical buffers.  Skipped on a
    single-GPU box (the driver's scaling run exercises the kernel there; tools/dp_nvlink_check.py is the same check by hand)."""
    import json
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs >= 2 GPUs on this box")
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr", "127.0.0.1",
                        "--master-port", "29577", os.path.join(ROOT, "tools", "dp_nvlink_check.py")],
                       capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert r.returncode == 0, (r.stdout + r.stderr)[-3000:]
    out = json.loads([l for l in r.stdout.splitlines() if l.startswith("{")][-1])
    for mode in ("multicast", "peer"):
        assert out[mode + "_worst_rel_err_vs_nccl"] < 1e-5 and out[mode + "_identical_on_all_ranks"], out
