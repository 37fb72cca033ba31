"""Inter-stage wire protocol, interoperability with the reference itself (pipeline.py:247-427).

Two gloo processes form a stage boundary; on one side sits this package's ``PipelineCommunication`` + ``DistTransport``, on
the other the REFERENCE's ``PipelineCommunication`` as recorded in tests/golden/wire_protocol.json: every tensor it sent
and received, in order, when it ran unmodified against this package (tests/golden/gen_wire_golden.py).  Here the
recorded side is replayed message for message.  In both directions: the one-off meta handshake (count, then ndims /
dtype id / shape / requires_grad per tensor -- ``DTYPE_TO_ID`` on the wire), two micro-batches of activations ``(hidden
fp32 requiring grad, labels int64)``, and the gradient travelling back.  Whatever the reference sent, this package must
receive bit for bit, with the right dtypes and ``requires_grad`` flags; whatever this package sends must be what the
reference received, tensor for tensor; and the handshake must happen exactly once.
"""
import json
import os
import sys

import numpy as np
import pytest
import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

from test_pipeline_gloo import run_spawn  # noqa: E402

GOLDEN = os.path.join(ROOT, "tests", "golden", "wire_protocol.json")


class StagePipeline:
    """What a ``PipelineCommunication`` reads of its pipeline (pipeline.py:266-268, 331, 389, 392, 404, 420)."""

    def __init__(self):
        self.device = torch.device("cpu")
        self.pipe_buffers = {"inputs": [None, None], "labels": [None, None], "outputs": [None, None]}


def microbatch(i):
    g = torch.Generator().manual_seed(100 + i)
    hidden = torch.randn(2, 8, 16, generator=g).requires_grad_(True)
    labels = torch.randint(0, 211, (2, 8), generator=g, dtype=torch.int64)
    return hidden, labels


def gradient(i):
    return torch.randn(2, 8, 16, generator=torch.Generator().manual_seed(200 + i))


def sender_side(comm, pipeline):
    """The earlier stage: sends activations, receives gradients."""
    assert comm.sent_activation_meta is False and comm.grad_recv_buf is None
    for b in (0, 1):
        pipeline.pipe_buffers["outputs"][b] = microbatch(b)
        comm.send_activations(buffer_id=b)
        assert comm.sent_activation_meta is True
    for b in (0, 1):
        comm.recv_gradients(buffer_id=b)
        assert len(comm.grad_recv_buf) == 1                      # one gradient: the labels produce none
        assert torch.equal(comm.grad_recv_buf[0], gradient(b))
        assert comm.grad_recv_buf[0].dtype == torch.float32 and not comm.grad_recv_buf[0].requires_grad


def receiver_side(comm, pipeline):
    """The later stage: receives activations, sends gradients."""
    assert comm.activation_recv_buf is None
    for b in (0, 1):
        comm.recv_activations(buffer_id=b)
        got = pipeline.pipe_buffers["inputs"][b]
        want = microbatch(b)
        assert isinstance(got, tuple) and len(got) == 2
        assert torch.equal(got[0], want[0]) and torch.equal(got[1], want[1])
        assert got[0].dtype == torch.float32 and got[1].dtype == torch.int64
        assert got[0].requires_grad and not got[1].requires_grad
        assert got[0] is not comm.activation_recv_buf[0]         # cloned out of the reused receive buffer (:386)
    buf_ids = [id(t) for t in comm.activation_recv_buf]
    for b in (0, 1):
        pipeline.pipe_buffers["inputs"][b][0].grad = gradient(b)
        comm.send_gradients(buffer_id=b)
        assert pipeline.pipe_buffers["inputs"][b] is None        # the slot is freed (:404)
    assert [id(t) for t in comm.activation_recv_buf] == buf_ids


def to_tensor(m):
    return torch.from_numpy(np.asarray(m["data"], dtype=m["dtype"]).reshape(m["shape"]))


def replay(messages, peer):
    """The reference's side of the boundary: its recorded sends, and its recorded receives checked bit for bit."""
    for i, m in enumerate(messages):
        want = to_tensor(m)
        if m["op"] == "send":
            dist.send(want, peer)
        else:
            got = torch.empty_like(want)
            dist.recv(got, peer)
            assert torch.equal(got, want), f"message {i} differs from what the reference received: {m}"


def worker(rank, world, port, sender_kind, receiver_kind, q):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world))
    torch.set_num_threads(1)
    try:
        dist.init_process_group("gloo")
        if (sender_kind if rank == 0 else receiver_kind) == "reference":
            with open(GOLDEN) as f:
                replay(json.load(f)[f"{sender_kind}-to-{receiver_kind}"], 1 - rank)
        else:
            from oobleck_b200.execution.pipeline import PipelineCommunication
            pipeline = StagePipeline()
            if rank == 0:
                sender_side(PipelineCommunication(pipeline, None, None, 1), pipeline)
            else:
                receiver_side(PipelineCommunication(pipeline, None, 0, None), pipeline)
        q.put((rank, None, None, None))
        dist.barrier()
    except Exception:  # noqa: BLE001
        import traceback
        q.put((rank, None, None, traceback.format_exc()))
        raise


@pytest.mark.timeout(300)
@pytest.mark.parametrize("sender,receiver", [("reference", "ours"), ("ours", "reference")],
                         ids=["reference-to-this", "this-to-reference"])
def test_stage_boundary_between_the_reference_and_this_package(sender, receiver):
    run_spawn(worker, 2, sender, receiver)
