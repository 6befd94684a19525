"""GPU tests of the training-step engine AT THE BENCHMARKED CONFIGURATION (BASELINE.json configs[2]: ImageFillOrigin,
512x512, batch 8, bf16): the CUDA-graph replay of `engine.TrainStep` -- side streams, gradient sinks, mask stream, operand
prefetch, everything bench.py times -- against the ORACLE (oracle/pconv_torch.py, pinned bit-for-bit to the reference by
tests/golden/net_ImageFillOrigin_512.npz), not against the engine's own eager mode.

Tolerances: the loss within 2e-3 of the fp32 oracle; every checked gradient within 3e-2 of max|ref| of the oracle run under
the SAME storage precision (oracle.pconv_torch.storage(bfloat16): activations / activation gradients rounded to bf16 at the
kernel hand-over points, fp32 everywhere else) -- the comparison that isolates the kernels from the precision policy.
"""
import os
import socket
import subprocess
import sys

import pytest
import torch

from gpu_cases import ROOT, relerr
from oracle import pconv_torch as O
from oracle.detfill import det_fill_state_dict, det_tensor

pytestmark = pytest.mark.gpu

GRAD_KEYS = ["decoder.7.0.feature_conv.weight", "decoder.6.0.0.feature_conv.weight", "decoder.5.0.0.feature_conv.weight",
             "decoder.4.0.0.feature_conv.weight", "decoder.6.0.1.bn_act.0.weight", "decoder.6.0.1.bn_act.0.bias",
             "decoder.5.0.1.bn_act.0.weight", "decoder.7.0.feature_conv.bias"]


@pytest.fixture(scope="module")
def dev():
    return torch.device("cuda:0")


def _inputs(batch, hw, seed=21):
    from text_segmentation_image_inpainting_b200.synthetic import random_hole_masks
    x = det_tensor("engine.x", (batch, 3, hw, hw))
    mask = torch.from_numpy(random_hole_masks(batch, hw, hw, seed=seed))
    return x, mask


def _oracle_step(sd0, x, mask):
    """fwd (fp32) and fwd + bwd (bf16 storage emulation) of the reference algorithm on the host cores."""
    from gpu_cases import oracle_bf16_step
    with torch.no_grad():
        loss32 = float(O.image_fill_origin(O.clone_state_dict(sd0), x * mask, mask, training=True).abs().mean())
    loss16, grads = oracle_bf16_step("ImageFillOrigin", x, mask, sd0)
    return loss32, loss16, grads


def test_train_step_graph_512_batch8_matches_oracle(dev):
    from text_segmentation_image_inpainting_b200 import _lib
    from text_segmentation_image_inpainting_b200.engine import TrainStep
    from text_segmentation_image_inpainting_b200.models.image_inpainting import ImageFillOrigin

    torch.set_num_threads(max(1, min(32, os.cpu_count() or 1)))
    net = ImageFillOrigin()
    sd0 = det_fill_state_dict(net.state_dict())
    net.load_state_dict(sd0)
    x, mask = _inputs(8, 512)
    ref_loss, ref_loss16, ref_grads = _oracle_step(sd0, x, mask)

    net = net.to(dev)
    # lr = 0: the eager warm-up steps and the capture run leave the weights where the oracle has them
    ts = TrainStep(net, compute_dtype=torch.bfloat16, lr=0.0, momentum=0.0, weight_decay=0.0, nesterov=False, use_graph=True)
    xd, md = x.to(dev), mask.to(dev)
    ts.warmup_and_capture(xd, md, eager_warmup=2)
    assert ts.graph is not None
    loss = float(ts.step(xd, md))                       # CUDA-graph replay: the path bench.py times
    torch.cuda.synchronize()
    code = _lib.ctypes.c_int(0)
    _lib.check(_lib.load().pcb_debug_pipeline_status(_lib.ctypes.byref(code)))
    assert code.value == 0, f"a tensor-core pipeline wait timed out (code {code.value})"
    assert abs(loss - ref_loss) <= 2e-3 * abs(ref_loss) and abs(loss - ref_loss16) <= 1e-3 * abs(ref_loss16), (loss, ref_loss, ref_loss16)
    params = dict(net.named_parameters())
    errs = {k: relerr(params[k].grad, ref_grads[k]) for k in ref_grads}
    worst = sorted(errs.items(), key=lambda kv: -kv[1])[:6]
    assert all(errs[k] <= 3e-2 for k in GRAD_KEYS), worst
    # the count-8 BatchNorms at the bottom of the U (2x2 maps) make the deepest gradients ill-conditioned: looser there
    assert max(errs.values()) <= 1e-1, worst

    # ADVICE r1: graph -> eager evaluation -> graph.  The eager pass re-lays-out the weights into NEW buffers (the optimiser
    # bumped the weight epoch); the graph must keep replaying on its own (pinned) operand buffers.
    net.eval()
    with torch.no_grad():
        xin, hm = ts._prepare(xd, md)
        out_eval = net((xin, hm))
    assert torch.isfinite(out_eval.float()).all()
    net.train()
    junk = [torch.empty(1 << 22, device=dev).normal_() for _ in range(8)]     # churn the allocator over any freed block
    loss2 = float(ts.step(xd, md))
    torch.cuda.synchronize()
    del junk
    assert loss2 == loss, (loss, loss2)               # forward has no unordered atomics: bitwise repeatable


def test_train_step_updates_match_oracle_sgd(dev):
    """Three graph steps WITH the optimiser (SGD + Nesterov + weight decay, checkpoints/ReadME.md:4) at 256x256 batch 2 against
    three oracle steps with torch.optim.SGD on CPU: the loss trajectory must agree."""
    from text_segmentation_image_inpainting_b200.engine import TrainStep
    from text_segmentation_image_inpainting_b200.models.image_inpainting import ImageFillOrigin
    net = ImageFillOrigin()
    sd0 = det_fill_state_dict(net.state_dict())
    net.load_state_dict(sd0)
    x, mask = _inputs(2, 256, seed=5)
    sd = O.clone_state_dict(sd0, requires_grad=True)
    opt = torch.optim.SGD([v for v in sd.values() if v.requires_grad], lr=1e-3, momentum=0.9, weight_decay=1e-4, nesterov=True)
    ref = []
    for _ in range(4):
        opt.zero_grad(set_to_none=True)
        out = O.image_fill_origin(sd, x * mask, mask, training=True)
        loss = out.abs().mean()
        loss.backward()
        opt.step()
        ref.append(float(loss))
    ts = TrainStep(net.to(dev), lr=1e-3, momentum=0.9, weight_decay=1e-4, nesterov=True, use_graph=False)
    xd, md = x.to(dev), mask.to(dev)
    got = [float(ts.step(xd, md)) for _ in range(4)]
    assert all(abs(a - b) <= 1e-2 * abs(b) for a, b in zip(got, ref)), (got, ref)
    assert ref[-1] != ref[0]


def test_bench_dump_outputs_writes_the_last_timed_step(tmp_path):
    """`bench.py --dump-outputs DIR`: one JSON line, and float32 / float64 arrays of the last timed step (loss, updated parameters,
    gradients, BatchNorm statistics) of at most 64 MB in all.  Two runs with the same arguments see the same inputs and so dump
    the same values (up to the unordered fp32 adds of the weight gradients); one more timed step moves the dumped state."""
    import json

    import numpy as np
    from text_segmentation_image_inpainting_b200.models.image_inpainting import ImageFillOrigin

    def run(steps, name):
        out = tmp_path / name
        r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--gpus", "1", "--steps", str(steps), "--warmup", "1",
                            "--no-cpu-baseline", "--dump-outputs", str(out)], capture_output=True, text=True, timeout=90, cwd=ROOT)
        assert r.returncode == 0, r.stderr[-3000:]
        lines = [ln for ln in r.stdout.splitlines() if ln.strip()]
        assert len(lines) == 1 and json.loads(lines[0])["steps"] == steps, r.stdout[:500]
        assert sum(f.stat().st_size for f in out.iterdir()) <= 64 << 20
        return {f.stem: np.load(f) for f in out.iterdir()}

    one, two, again = run(1, "one"), run(2, "two"), run(2, "again")
    assert set(two) == {"loss", "params", "grads", "bn_stats"}
    assert all(a.dtype in (np.float32, np.float64) and np.isfinite(a).all() for a in two.values())
    n_params = sum(p.numel() for p in ImageFillOrigin().parameters() if p.requires_grad)
    assert two["params"].shape == two["grads"].shape == (min(n_params, 1 << 22),)
    assert two["loss"].shape == (1,) and two["loss"][0] > 0 and np.abs(two["grads"]).max() > 0

    def diff(a, b, name):
        return float(np.abs(a[name].astype(np.float64) - b[name]).max())
    # same arguments: same inputs, same trajectory
    assert diff(two, again, "loss") <= 1e-3 * abs(float(two["loss"][0])), (two["loss"], again["loss"])
    for name in ("params", "grads", "bn_stats"):
        assert diff(two, again, name) <= 1e-3 * float(np.abs(two[name]).max()), name
    # --steps sets the number of timed (optimiser) steps: one more step moves the parameters and the loss by far more than
    # the run-to-run noise above
    assert diff(one, two, "params") > 100 * diff(two, again, "params")
    assert diff(one, two, "loss") > 100 * diff(two, again, "loss")


# ------------------------------------------------------------------------------------------------------------------
# two ranks over NCCL: the averaged gradient arena == the single-process gradient of the concatenated batch
# ------------------------------------------------------------------------------------------------------------------
_RANK_SCRIPT = r"""
import os, sys, json
import torch, torch.distributed as dist
sys.path.insert(0, {root!r})
from oracle.detfill import det_fill_state_dict, det_tensor
from text_segmentation_image_inpainting_b200.engine import TrainStep
from text_segmentation_image_inpainting_b200.models.image_inpainting import ImageFillOrigin
from text_segmentation_image_inpainting_b200.synthetic import random_hole_masks
rank, world = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"])
torch.cuda.set_device(rank)
dev = torch.device("cuda", rank)
dist.init_process_group("nccl", device_id=dev)
net = ImageFillOrigin()
net.load_state_dict(det_fill_state_dict(net.state_dict()))
if rank == 1:                                   # a replica that starts from different weights must adopt rank 0's
    with torch.no_grad():
        for p in net.parameters():
            p.add_(0.5)
B, HW = 2, 256
x = det_tensor("ddp.x", (world * B, 3, HW, HW))[rank * B:(rank + 1) * B].to(dev)
mask = torch.from_numpy(random_hole_masks(world * B, HW, HW, seed=31))[rank * B:(rank + 1) * B].to(dev)
ts = TrainStep(net.to(dev), lr=0.0, momentum=0.0, weight_decay=0.0, nesterov=False, process_group=dist.group.WORLD,
               use_graph={graph})
ts.warmup_and_capture(x, mask, eager_warmup=2)
loss = float(ts.step(x, mask))
torch.cuda.synchronize()
g = ts.flat.flat_g.clone() * ts.grad_scale        # the 1/world factor is folded into the optimiser kernel
if rank == 0:
    torch.save({{"g": g.cpu(), "loss": loss, "overlapped": bool(ts.overlap_active)}}, {out!r})
ts.close()                                        # graphs with captured collectives must die before the communicator
dist.barrier()
dist.destroy_process_group()
"""


@pytest.mark.parametrize("graph", [False, True])
def test_two_rank_nccl_gradient_average_matches_single_process(tmp_path, graph):
    """BatchNorm statistics are rank-local (the reference has no SyncBN), so the data-parallel gradient is the MEAN of the two
    per-rank gradients: check the all-reduced arena of a 2-rank job (bucketed, overlapped with backward) against the mean of two
    single-process backward passes on the same half batches."""
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    from text_segmentation_image_inpainting_b200.engine import TrainStep
    from text_segmentation_image_inpainting_b200.models.image_inpainting import ImageFillOrigin
    from text_segmentation_image_inpainting_b200.synthetic import random_hole_masks
    out = str(tmp_path / "rank0.pt")
    script = tmp_path / "rank.py"
    script.write_text(_RANK_SCRIPT.format(root=ROOT, out=out, graph=graph))
    s = socket.socket(); s.bind(("127.0.0.1", 0)); port = s.getsockname()[1]; s.close()
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr", "127.0.0.1",
                        "--master-port", str(port), str(script)], capture_output=True, text=True, timeout=420)
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-3000:]
    got = torch.load(out)
    dev = torch.device("cuda:0")
    B, HW, world = 2, 256, 2
    xs = det_tensor("ddp.x", (world * B, 3, HW, HW))
    ms = torch.from_numpy(random_hole_masks(world * B, HW, HW, seed=31))
    acc = None
    for rk in range(world):
        net = ImageFillOrigin()
        net.load_state_dict(det_fill_state_dict(net.state_dict()))
        ts = TrainStep(net.to(dev), lr=0.0, momentum=0.0, weight_decay=0.0, nesterov=False, use_graph=False)
        ts.step(xs[rk * B:(rk + 1) * B].to(dev), ms[rk * B:(rk + 1) * B].to(dev))
        torch.cuda.synchronize()
        g = ts.flat.flat_g.clone().cpu()
        acc = g if acc is None else acc + g
    ref = acc / world
    err = float((got["g"] - ref).abs().max() / ref.abs().max())
    assert err <= 2e-3, err                           # wgrad split-K adds are unordered fp32: not bitwise
