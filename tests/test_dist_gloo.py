"""World-size-2 `gloo` test of the one-process-per-GPU control plane (no GPU): stage shipment, link-token
exchange order, shared-memory counters / result ring, and the node data loop's host logic with a fake stage."""
import os
import socket
import sys
import time
from pathlib import Path

import numpy as np
import pytest

ROOT = Path(__file__).resolve().parents[1]


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


class FakeRunner:
    """Stands in for StageRunner: records the wiring calls, 'computes' y = x + rank on the host."""

    def __init__(self, rank, world, depth=2):
        self.rank, self.world, self.depth = rank, world, depth
        self.finalized = False
        self.imported = {}
        self.steps = []
        self.out_shape = (1, 4)

    def export_link(self, role):
        return f"tok-r{self.rank}-role{role}".encode()

    def import_link(self, role, token):
        self.imported[role] = bytes(token)

    def finalize(self):
        self.finalized = True

    def step(self, seq):
        self.steps.append(seq)

    def result(self, seq, out):
        out[...] = float(seq) + 0.5
        return out

    def sync(self):
        pass


def _worker(rank, world, port, q):
    sys.path.insert(0, str(ROOT))
    # host-only test: with a GPU visible DistContext would bind rank r to cuda:r, which a one-GPU machine lacks
    os.environ.update(RANK=str(rank), WORLD_SIZE=str(world), LOCAL_RANK=str(rank), MASTER_ADDR="127.0.0.1",
                      MASTER_PORT=str(port), CUDA_VISIBLE_DEVICES="")
    import threading
    from defer_b200.dist import DistContext
    from defer_b200.node import Node
    ctx = DistContext(backend="gloo", ring=8, out_elems=4)
    try:
        runner = FakeRunner(rank, world)
        # --- shipment: rank 0 "dispatcher" scatters one message per stage
        if rank == 0:
            for i in range(world):
                ctx.send_stage(i, {"json": f"stage{i}", "weights": [np.full(3, i, np.float32)], "next_node": str(i + 1)})
            t = threading.Thread(target=ctx.wait_all_ready, daemon=True)
            t.start()
        msg = ctx.recv_stage()
        assert msg["json"] == f"stage{rank}" and msg["weights"][0][0] == rank
        ctx.exchange_links(runner)
        runner.finalize()
        ctx.ack_ready()
        if rank == 0:
            t.join(timeout=30)
            assert not t.is_alive()
        assert ctx.local_runner() is runner
        # neighbours' tokens landed on the right side
        if rank < world - 1:
            assert runner.imported[0] == f"tok-r{rank+1}-role0".encode()
        if rank > 0:
            assert runner.imported[1] == f"tok-r{rank-1}-role1".encode()
        # --- data loop: rank 0 marks microbatches as submitted, the last rank publishes results in order
        node = Node(dist_ctx=ctx, device=rank, poll_s=1e-4)
        th = threading.Thread(target=node._data_loop, args=(runner,), daemon=True)
        th.start()
        n = 20
        if rank == 0:
            got = []
            for s in range(n):
                while s - len(got) >= runner.depth:      # the dispatcher's in-flight throttle
                    got.append(float(ctx.wait_result(len(got), timeout=30)[0]))
                ctx.mark_submitted(s + 1)
            while len(got) < n:
                got.append(float(ctx.wait_result(len(got), timeout=30)[0]))
            assert got == [s + 0.5 for s in range(n)]
            ctx.request_stop()
        th.join(timeout=30)
        assert not th.is_alive()
        if rank == world - 1:
            assert runner.steps == list(range(n))       # every microbatch stepped exactly once, in order
        assert ctx.max_over_ranks(float(rank)) == world - 1
        q.put((rank, "ok"))
    except BaseException as e:  # noqa: BLE001
        import traceback
        q.put((rank, "fail: " + traceback.format_exc()))
    finally:
        ctx.close()


@pytest.mark.timeout(180)
def test_control_plane_world2():
    import torch.multiprocessing as mp
    world, port = 2, _free_port()
    mpctx = mp.get_context("spawn")
    q = mpctx.Queue()
    procs = [mpctx.Process(target=_worker, args=(r, world, port, q)) for r in range(world)]
    for p in procs:
        p.start()
    res = {}
    for _ in range(world):
        r, s = q.get(timeout=150)
        res[r] = s
    for p in procs:
        p.join(timeout=30)
    assert res == {0: "ok", 1: "ok"}, res


# ------------------------------------------------------------------------------------------------------
# The whole one-process-per-GPU path on CPU: Node.run (stage shipment, link exchange, ACK, data loop) on every rank and
# DEFER.run_defer with coalesced ingress on rank 0, with a host-side stand-in for StageRunner.  Checks FIFO order, the
# split of coalesced groups back into per-item results over the shared-memory result ring, and the orderly shutdown.
# ------------------------------------------------------------------------------------------------------
class _HostStage:
    """StageRunner stand-in: no data path (ranks are separate processes); the last stage's result for microbatch `seq`
    is the row vector [seq * batch + i] so the dispatcher-side bookkeeping can be verified end to end."""
    made = []

    def __init__(self, batch, depth, rank, world):
        self.batch, self.depth, self.rank, self.world = batch, depth, rank, world
        self.out_shape = (batch, 4)
        self.links, self.steps, self.items = {}, [], []
        self.finalized = self.closed = self.unlinked = False

    @classmethod
    def from_wire(cls, model_json, weights, device=0, dtype="float32", max_batch=1, depth=1, is_first=True, is_last=True,
                  finalize=True, **kw):
        import os
        r = cls(max_batch, depth, int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]))
        r.json, r.n_weights, r.is_first, r.is_last = model_json, len(weights), is_first, is_last
        cls.made.append(r)
        return r

    def export_link(self, role):
        return f"tok-r{self.rank}-role{role}".encode()

    def import_link(self, role, token):
        self.links[role] = bytes(token)

    def finalize(self):
        self.finalized = True

    def submit_items(self, seq, items):
        self.items.append((seq, len(items)))

    def step(self, seq):
        self.steps.append(seq)

    def result(self, seq, out=None):
        if out is None:
            out = np.empty(self.out_shape, np.float32)
        out[...] = (seq * self.batch + np.arange(self.batch, dtype=np.float32))[:, None]
        return out

    def sync(self):
        pass

    def unlink(self):
        self.unlinked = True

    def close(self):
        self.closed = True


def _worker_defer(rank, world, port, q):
    sys.path.insert(0, str(ROOT))
    # host-only test: with a GPU visible DistContext would bind rank r to cuda:r, which a one-GPU machine lacks
    os.environ.update(RANK=str(rank), WORLD_SIZE=str(world), LOCAL_RANK=str(rank), MASTER_ADDR="127.0.0.1",
                      MASTER_PORT=str(port), CUDA_VISIBLE_DEVICES="")
    import queue as pyqueue
    import threading
    import defer_b200.node as node_mod
    from defer_b200 import applications
    from defer_b200.dispatcher import DEFER
    from defer_b200.dist import DistContext
    node_mod.StageRunner = _HostStage                   # Node.run builds its stage through this name
    G = 4
    ctx = DistContext(backend="gloo", ring=8, out_elems=4, batch=G)
    try:
        node = node_mod.Node(dist_ctx=ctx, device=rank, poll_s=1e-4)
        nt = threading.Thread(target=node.run, daemon=True)
        nt.start()
        if rank == 0:
            model = applications.ResNet50(input_shape=(32, 32, 3))
            cuts = applications.default_cuts(model, world)
            defer = DEFER(list(range(world)), depth=2, coalesce=G, linger_us=200000, dist=ctx)
            in_q, out_q = pyqueue.Queue(), pyqueue.Queue()
            t = threading.Thread(target=defer.run_defer, args=(model, cuts, in_q, out_q), daemon=True)
            t.start()
            assert defer.wait_ready(60), "pipeline did not come up"
            n = 5 * G + 2                                  # the last group is partial (2 items after the linger window)
            for i in range(n):
                in_q.put(np.full((1, 32, 32, 3), float(i), np.float32))
            got = [out_q.get(timeout=60) for _ in range(n)]
            assert all(g.shape == (1, 4) for g in got)
            assert [float(g[0, 0]) for g in got] == [float(i) for i in range(n)]      # FIFO, one result per item
            assert defer.results_delivered == n and defer.items_submitted == n
            defer.close()
            t.join(timeout=30)
            assert not t.is_alive()
        ctx.shutdown(nt)
        stage = _HostStage.made[0]
        assert stage.finalized and stage.unlinked and stage.closed
        assert stage.batch == G and stage.is_first == (rank == 0) and stage.is_last == (rank == world - 1)
        assert stage.steps == list(range(6))               # 5 full groups + the partial one, each stepped once, in order
        if rank == 0:
            assert [c for _, c in stage.items] == [G] * 5 + [2]
        q.put((rank, "ok"))
    except BaseException:  # noqa: BLE001
        import traceback
        q.put((rank, "fail: " + traceback.format_exc()))
        try:
            ctx.close()
        except Exception:
            pass


@pytest.mark.timeout(240)
def test_defer_dist_path_world2_with_coalescing():
    import torch.multiprocessing as mp
    world, port = 2, _free_port()
    mpctx = mp.get_context("spawn")
    q = mpctx.Queue()
    procs = [mpctx.Process(target=_worker_defer, args=(r, world, port, q)) for r in range(world)]
    for p in procs:
        p.start()
    res = {}
    for _ in range(world):
        r, s = q.get(timeout=200)
        res[r] = s
    for p in procs:
        p.join(timeout=30)
    assert res == {0: "ok", 1: "ok"}, res
