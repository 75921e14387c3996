"""Lane scheduler: runs the independent per-scale chains of a multigrid stage on different CUDA streams.

Within one mg stage the chain conv -> BatchNorm -> ReLU of every grid (models/ilsvrc/rnmg.lua:91-159) only
meets the other grids again at the next ResampleConcat, and most of those kernels (14x14, 7x7 ... grids) are
far too small to fill 148 SMs.  Each plan op declares its work as units with the device buffers they read and
write (ops.Op.forward_unit / backward_units); units are assigned a lane by the spatial size they work on, and this
module derives -- once per plan and pass -- the cross-lane event waits that keep every read-after-write, write-after-read and write-after-write
pair ordered.  Execution order on each lane is the plan order, so a single lane reproduces the serial plan.

The schedule is static: (lane switch, event waits, op, event record) tuples replayed through the C ABI
(mg_ctx_lane / mg_ctx_event_wait / mg_ctx_event_record).  Every pass starts with lanes waiting for lane 0 and
ends with lane 0 waiting for all lanes, so nothing outside the pass ever sees a side stream.
"""


class Unit:
    """a schedulable piece of an op's work: buffers (reads, writes) or None, run(E, params), the engine passes it belongs
    to, optional fixed lane ("background"); its spatial size is the op's"""

    def __init__(self, op, io, run, passes, lane=None):
        self.op, self.io, self.run, self.passes, self.lane = op, io, run, passes, lane
        self._size = op.size()

    def size(self):
        return self._size


class Schedule:
    def __init__(self, ops, io_of, run_of, n_lanes, ev_base, background_lane=None):
        """ops in execution order; io_of(op) -> (reads, writes) keys or None; run_of(op) -> callable(E).
        Ops whose `lane` attribute is "background" (work nothing in the pass waits for, e.g. weight gradients) all
        go to `background_lane`; everything else is spread over lanes 0..n_lanes-1 by spatial size."""
        sizes = sorted({op.size() for op in ops}, reverse=True)
        lane_of_size = {h: i % n_lanes for i, h in enumerate(sizes)}
        last_w, readers, synced = {}, {}, {}
        START = (0, -1)                     # pseudo op: everything enqueued on lane 0 before the pass
        record = set()
        self.steps = []                      # (lane, [event ids to wait for], run, seq)
        used = {0}
        for seq, op in enumerate(ops):
            io = io_of(op)
            run = run_of(op)
            if io is None:                   # unknown effects: behind a full join, on lane 0
                self.steps.append((0, "join", run, seq))
                last_w, readers, synced = {}, {}, {}
                START = (0, seq)
                record.add(seq)
                continue
            lane = lane_of_size[op.size()]
            if getattr(op, "lane", None) == "background" and background_lane is not None:
                lane = background_lane
            used.add(lane)
            r, w = io
            deps = set()
            for k in list(r) + list(w):
                deps.add(last_w.get(k, START))
            for k in w:
                deps.update(readers.get(k, ()))
            need = {}
            for dl, ds in deps:
                if dl != lane and synced.get((dl, lane), -2) < ds:
                    need[dl] = max(need.get(dl, -2), ds)
            for dl, ds in need.items():
                synced[(dl, lane)] = ds
                record.add(ds)
            self.steps.append((lane, sorted(need.values()), run, seq))
            for k in w:
                last_w[k] = (lane, seq)
                readers[k] = []
            for k in r:
                readers.setdefault(k, []).append((lane, seq))
        self.record = record
        self.lanes = sorted(used)
        self.ev_base = ev_base               # event ids: ev_base = start, ev_base + 1 + seq, then one per lane for the final join
        self.n_ops = len(ops)

    def n_events(self):
        return 1 + self.n_ops + 8

    def _ev(self, seq):
        return self.ev_base + 1 + seq        # seq = -1 -> the start event

    def _join(self, ctx, cur):
        """lane 0 waits for everything enqueued on the side lanes; returns on lane 0"""
        for l in self.lanes:
            if l:
                if cur != l:
                    ctx.call("mg_ctx_lane", l)
                    cur = l
                ctx.call("mg_ctx_event_record", self.ev_base + 1 + self.n_ops + l)
        if cur != 0:
            ctx.call("mg_ctx_lane", 0)
        for l in self.lanes:
            if l:
                ctx.call("mg_ctx_event_wait", self.ev_base + 1 + self.n_ops + l)
        return 0

    def run(self, E, *args):
        """args: passed on to every op's run after E"""
        ctx = E.ctx
        cur = 0
        try:
            ctx.call("mg_ctx_event_record", self._ev(-1))
            for lane, waits, run, seq in self.steps:
                if waits == "join":
                    cur = self._join(ctx, cur)
                else:
                    if lane != cur:
                        ctx.call("mg_ctx_lane", lane)
                        cur = lane
                    for ds in waits:
                        ctx.call("mg_ctx_event_wait", self._ev(ds))
                run(E, *args)
                if seq in self.record:
                    ctx.call("mg_ctx_event_record", self._ev(seq))
            self._join(ctx, cur)
        finally:
            ctx.call("mg_ctx_lane", 0)
