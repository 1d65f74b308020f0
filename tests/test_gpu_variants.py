"""The A/B variants that ship in libnerfpp_b200.so behind environment switches (read once per process) stay correct: each is run in a fresh
process through the parity tests of the default path.
  NRF_NERF_CLUSTER=2    classic-NeRF forward with 2-CTA clusters sharing one multicast weight stream (csrc/mlp_nerf_tc.cu)
  NRF_LERF_EPI_WARPS=8  eight epilogue warps in the LeRF SIGMA / HIDDEN programs (csrc/lerf_tc.cu)
  NRF_ADAM_L2HINT=0     Adam without the L2 eviction-priority hints (csrc/optim.cu)
  NRF_RENDER_REUSE=0    nrf_render_rays_fwd evaluating every merged row of the fine pass instead of the importance samples only (csrc/render.cu):
                        the test compares it with the composed path, which reuses — bit for bit
  NRF_HASH_SPLIT=0      hash forward with one thread per point instead of four lanes per point (csrc/hash_encode.cu)
  NRF_PDL=1             programmatic dependent launch along the step's kernel chain (csrc/common.cuh launch_kernel / pdl_prologue)
  NRF_SAMPLER_BLOCK=0   warp-per-ray sampler also for training-sized batches (csrc/sampler.cu)"""
import os
import subprocess
import sys

import pytest

pytestmark = pytest.mark.gpu
HERE = os.path.dirname(os.path.abspath(__file__))

VARIANTS = [
    ({"NRF_NERF_CLUSTER": "2"}, ["test_gpu_mlp_nerf.py"], "forward_matches_oracle or repeatable"),
    ({"NRF_LERF_EPI_WARPS": "8"}, ["test_gpu_lerf.py"], "fixture or oracle"),
    ({"NRF_ADAM_L2HINT": "0"}, ["test_gpu_render.py"], "adam"),
    ({"NRF_RENDER_REUSE": "0"}, ["test_gpu_pipeline.py"], "fused_render_entry"),
    ({"NRF_HASH_SPLIT": "0"}, ["test_gpu_hash.py"], "fixture or reuse or rays"),
    ({"NRF_PDL": "1"}, ["test_gpu_pipeline.py"], "graph or gradients or trains or reuse or render"),
    ({"NRF_SAMPLER_BLOCK": "0"}, ["test_gpu_render.py"], "sample_pdf or merge or sampler"),
]


@pytest.mark.parametrize("env,files,expr", VARIANTS, ids=[",".join(f"{k}={v}" for k, v in e.items()) for e, _, _ in VARIANTS])
def test_variant_passes_the_default_paths_parity_tests(env, files, expr):
    cmd = [sys.executable, "-m", "pytest", "-q", "-x", "--no-header", "-k", expr] + [os.path.join(HERE, f) for f in files]
    out = subprocess.run(cmd, capture_output=True, text=True, timeout=600, env={**os.environ, **env})
    assert out.returncode == 0 and " passed" in out.stdout, out.stdout[-3000:] + out.stderr[-2000:]
