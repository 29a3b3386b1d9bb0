"""Which driver owns a plan's buffers (tpdm_sample_*, tpdm_queue_*, tpdm_stream_*): each begin hands the plan to its driver, a
call that needs another owner returns TPDM_ERR_STATE and enqueues nothing (include/tpdm_b200.h, open prompt stream section)."""
import ctypes as C

import pytest
import torch

pytestmark = pytest.mark.gpu

TINY = dict(sample_size=32, patch_size=2, in_channels=16, num_layers=2, attention_head_dim=96, num_attention_heads=4, joint_attention_dim=4096,
            caption_projection_dim=384, pooled_projection_dim=2048, out_channels=16, pos_embed_max_size=96)
P, SLOTS, T_MAX, CAP = 3, 2, 4, 2


@pytest.fixture(scope="module")
def eng():
    from tpdm_b200.modeling_sd3_pnt import SD3PredictNextTimeStepModel

    torch.manual_seed(5)
    model = SD3PredictNextTimeStepModel(transformer_config=TINY, torch_dtype=torch.float32, device="cuda")
    yield model.get_engine()


@pytest.fixture(scope="module")
def inp():
    g = torch.Generator().manual_seed(6)
    mk = lambda *s: torch.randn(*s, generator=g).cuda()
    return dict(lat=mk(P, 16, 32, 32), pe=mk(P, 333, 4096), ne=mk(P, 333, 4096), pp=mk(P, 2048), npp=mk(P, 2048))


@pytest.fixture
def plan(eng):
    from tpdm_b200.engine import Plan

    return Plan(eng, SLOTS, True, 32, 333, T_MAX)      # private: no other test's driver has touched it


class Calls:
    """The ABI calls of one plan, on the current (default) stream; workspaces and outputs stay alive with the object."""

    def __init__(self, plan, inp):
        from tpdm_b200 import _lib as L

        self.L, self.lib, self.h, self.x = L, L.load(), plan.handle, inp
        self.keep = []

    def sample_begin(self):
        x, p = self.x, self.L.ptr
        return self.lib.tpdm_sample_begin(self.h, p(x["lat"][:SLOTS]), p(x["ne"][:SLOTS]), p(x["pe"][:SLOTS]), p(x["npp"][:SLOTS]),
                                          p(x["pp"][:SLOTS]), 7.0, 1, None, 0, None)

    def sample_step(self, step=0):
        return self.lib.tpdm_sample_step(self.h, step, None)

    def queue_begin(self, short_by=0):
        x, p = self.x, self.L.ptr
        nbytes = self.lib.tpdm_queue_workspace_bytes(self.h, P)
        ws, base = self.L.aligned_workspace(nbytes, "cuda")
        outs = (torch.zeros(1, dtype=torch.int32, device="cuda"), torch.zeros(P, 16, 32, 32, device="cuda"),
                torch.zeros(P, dtype=torch.int32, device="cuda"), torch.zeros(P, T_MAX + 1, device="cuda"))
        self.keep.append((ws, outs))
        return self.lib.tpdm_queue_begin(self.h, P, p(x["lat"]), p(x["ne"]), p(x["pe"]), p(x["npp"]), p(x["pp"]), 7.0, base,
                                         nbytes - short_by, *[p(t) for t in outs], None, 0, None, 0, None)

    def queue_step(self):
        return self.lib.tpdm_queue_step(self.h, None)

    def queue_step_graph(self):
        return self.lib.tpdm_queue_step_graph(self.h, None)

    def queue_status(self):
        a, s = self.L.vp(), self.L.vp()
        return self.lib.tpdm_queue_status(self.h, C.byref(a), C.byref(s))

    def set_rollout(self):
        return self.lib.tpdm_queue_set_rollout(self.h, 1, None, None, None, None, None, None)

    def stream_open(self):
        nbytes = self.lib.tpdm_stream_workspace_bytes(self.h, CAP)
        ws, base = self.L.aligned_workspace(nbytes, "cuda")
        self.keep.append(ws)
        return self.lib.tpdm_stream_open(self.h, CAP, 7.0, base, nbytes, None)

    def stream_submit(self):
        x, p = self.x, self.L.ptr
        return self.lib.tpdm_stream_submit(self.h, 1, (C.c_int * 1)(0), p(x["lat"]), p(x["ne"]), p(x["pe"]), p(x["npp"]), p(x["pp"]), None)

    def stream_status(self):
        ptrs = [self.L.vp() for _ in range(5)]
        return self.lib.tpdm_stream_status(self.h, *[C.byref(q) for q in ptrs])

    def stream_close(self):
        return self.lib.tpdm_stream_close(self.h)

    def ok(self, *names):
        for name in names:
            assert getattr(self, name)() == 0, (name, self.lib.tpdm_last_error())
            torch.cuda.synchronize()

    def refused(self, name, code=None, msg=None, **kw):
        """The call fails with `code` (TPDM_ERR_STATE) and launches nothing that the launch counter or the profiler sees."""
        lib = self.lib
        torch.cuda.synchronize()
        lib.tpdm_launch_count(1)
        assert lib.tpdm_profile_start(64) == 0
        st = getattr(self, name)(**kw)
        err = lib.tpdm_last_error()
        ms, flops, count = (C.c_double * 2)(), (C.c_double * 2)(), (C.c_longlong * 2)()
        assert lib.tpdm_profile_stop(ms, flops, count, 2) == 0
        assert st == (self.L.TPDM_ERR_STATE if code is None else code), (name, st, err)
        assert msg is None or msg in err, (name, err)
        assert lib.tpdm_launch_count(0) == 0 and list(count) == [0, 0], name


def test_queue_calls_refused_after_a_later_sample_begin(plan, inp):
    """The sampler overwrites the latents, ctx0 and text rows the queue's slots point into: the queue has lost the plan."""
    c = Calls(plan, inp)
    c.ok("queue_begin", "queue_step", "sample_begin")
    for name in ("queue_step", "queue_step_graph", "queue_status", "set_rollout"):
        c.refused(name, msg=b"call tpdm_queue_begin first")
    c.ok("sample_step")
    c.ok("queue_begin", "queue_step")                   # a new begin hands the plan back to the queue
    c.refused("sample_step", msg=b"call tpdm_sample_begin first")


def test_sample_then_stream_then_queue(plan, inp):
    c = Calls(plan, inp)
    c.ok("sample_begin", "sample_step", "stream_open")
    for name in ("sample_begin", "sample_step", "queue_begin", "set_rollout", "stream_open"):
        c.refused(name, msg=b"open prompt stream")
    c.ok("stream_status", "queue_status", "stream_submit", "queue_step", "queue_step", "stream_close")
    for name in ("stream_submit", "stream_status", "stream_close"):
        c.refused(name, msg=b"no open stream")
    c.refused("sample_step", msg=b"call tpdm_sample_begin first")
    c.refused("queue_step", msg=b"call tpdm_queue_begin first")
    c.ok("queue_begin", "queue_step")
    c.refused("stream_open", msg=b"prompt queue")        # the queue owns the plan now
    c.ok("sample_begin", "stream_open", "stream_close")


def test_fresh_plan_belongs_to_no_driver(plan, inp):
    c = Calls(plan, inp)
    for name in ("sample_step", "queue_step", "queue_step_graph", "queue_status", "set_rollout", "stream_submit", "stream_status",
                 "stream_close"):
        c.refused(name)


def test_queue_workspace_size_is_exact(plan, inp):
    c = Calls(plan, inp)
    c.refused("queue_begin", code=c.L.TPDM_ERR_ARG, msg=b"queue workspace", short_by=1)
    c.refused("queue_step")                              # the refused begin handed the plan to nobody
    c.ok("queue_begin", "queue_step")
