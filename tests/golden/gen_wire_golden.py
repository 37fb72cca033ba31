#!/usr/bin/env python
"""Record the reference's side of the inter-stage wire protocol -> tests/golden/wire_protocol.json.

Needs the reference's sources (imported unmodified with the stubs of gen_golden.py, ``deepspeed.comm`` delegating to
``torch.distributed``):

    python tests/golden/gen_wire_golden.py REFERENCE_DIR

For each direction of tests/test_wire_protocol_interop.py, two gloo processes form a stage boundary: the reference's
``PipelineCommunication`` on one side, this package's on the other, both driven exactly as that test drives them and
both checked by its assertions.  Every tensor the reference's side sends or receives is recorded in order (dtype,
shape, values); the test replays that record in place of the reference."""
import json
import os
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
sys.path.insert(0, HERE)


def reference_comm(ref_dir, pipeline, prev_rank, next_rank, log):
    import torch.distributed as dist

    import gen_golden
    gen_golden.install_stubs()
    import deepspeed.comm as dc

    def recording(op, fn):
        def call(tensor, peer, *a, **k):
            work = fn(tensor, peer, *a, **k)
            log.append({"op": op, "dtype": str(tensor.dtype).replace("torch.", ""), "shape": list(tensor.shape),
                        "data": tensor.detach().reshape(-1).tolist()})
            return work
        return call

    for name in ("get_rank", "is_initialized"):
        setattr(dc, name, getattr(dist, name))
    dc.send, dc.recv = recording("send", dist.send), recording("recv", dist.recv)
    dc.isend = dc.irecv = None            # the blocking calls are the protocol; an asynchronous one would go unrecorded
    from oobleck.execution.pipeline import PipelineCommunication
    import oobleck.execution.pipeline as ref_mod
    assert ref_mod.__file__.startswith(ref_dir)
    return PipelineCommunication(pipeline, None, prev_rank, next_rank)


def record_worker(rank, world, port, ref_dir, sender_kind, receiver_kind, q):
    import torch
    import torch.distributed as dist

    import test_wire_protocol_interop as T
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world))
    torch.set_num_threads(1)
    try:
        sys.path.insert(0, ref_dir)
        dist.init_process_group("gloo")
        pipeline, log = T.StagePipeline(), []
        prev_rank, next_rank = (None, 1) if rank == 0 else (0, None)
        if (sender_kind if rank == 0 else receiver_kind) == "reference":
            comm = reference_comm(ref_dir, pipeline, prev_rank, next_rank, log)
        else:
            from oobleck_b200.execution.pipeline import PipelineCommunication
            comm = PipelineCommunication(pipeline, None, prev_rank, next_rank)
        (T.sender_side if rank == 0 else T.receiver_side)(comm, pipeline)
        q.put((rank, log, None, None))
        dist.barrier()
    except Exception:  # noqa: BLE001
        import traceback
        q.put((rank, None, None, traceback.format_exc()))
        raise


def main():
    from test_pipeline_gloo import run_spawn
    ref_dir = os.path.abspath(sys.argv[1])
    out = {}
    for sender, receiver in (("reference", "ours"), ("ours", "reference")):
        results = run_spawn(record_worker, 2, ref_dir, sender, receiver)
        out[f"{sender}-to-{receiver}"] = results[0 if sender == "reference" else 1][1]
    path = os.path.join(HERE, "wire_protocol.json")
    with open(path, "w") as f:
        json.dump(out, f, separators=(",", ":"))
    print(f"wrote {path}: " + ", ".join(f"{k} {len(v)} messages" for k, v in out.items()), file=sys.stderr)


if __name__ == "__main__":
    main()
