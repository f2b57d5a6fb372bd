"""Plan leasing for the autograd paths (Unet.differentiable, DeepLabV3.forward with x.requires_grad).

A C plan bound to one input shape holds one forward's activations until its backward has run.  Each live autograd graph
therefore leases a plan of its own from a pool keyed by shape, together with the inputs the plan reads; the lease ends when
the graph's backward has been enqueued or when the graph is freed without one.  Plans carry a ``busy`` flag.
"""


def lease_plan(pool, shape, make):
    """A free plan of ``shape`` from ``pool`` (a dict shape -> [plan]), made with ``make()`` when every plan of that shape is
    held by a live graph; marked busy."""
    plans = pool.setdefault(shape, [])
    plan = next((p for p in plans if not p.busy), None)
    if plan is None:
        plan = make()
        plans.append(plan)
    plan.busy = True
    return plan


class Lease:
    """A plan held by one autograd graph, with the forward's inputs (the backward may read them).  Released when the backward
    has been enqueued, or when the graph is freed without one (the Function's ctx, which owns the lease, dies)."""

    def __init__(self, plan, *inputs):
        self.plan, self.inputs = plan, inputs

    def release(self):
        if self.plan is not None:
            self.plan.busy = False
        self.plan, self.inputs = None, None

    def __del__(self):
        self.release()
