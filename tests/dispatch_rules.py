"""The kernel choice of csrc/ascent_plan.h (plan_solve), written out independently, and the kernel variants it reaches.

test_gpu_kernel_matrix.py runs every entry of VARIANTS on the GPU against the oracle; test_device_source_on_host.py
checks plan_solve itself against `V.expect` on the CPU, so a change to either side of the rules fails there.
"""


COOP_MAX_BATCH = 6144         # kCoopMaxBatch: AUTO runs the cooperative kernel up to this batch size
COOP_BLOCK = 256              # kCoopBlock


def _gp(S, B, lanes=0):
    """Cooperative kernel: lanes per problem."""
    return lanes if lanes else (32 if B <= 8 * S else 8)


def _bps(S, B, gp):
    """Cooperative kernel: CTAs per SM."""
    return 1 if B <= S * (COOP_BLOCK // gp) else 2


def _coop_window(S, gp, bps, cap=COOP_MAX_BATCH):
    """Batch sizes (lo, hi] for which AUTO picks coop<gp, bps> (lanes chosen by size)."""
    lo, hi = (0, 8 * S) if gp == 32 else (8 * S, cap)
    if gp == 8:
        lo, hi = (lo, min(hi, 32 * S)) if bps == 1 else (max(lo, 32 * S), hi)
    return lo, hi


def _top(window):
    """The largest batch of the window that still leaves a partial last chunk (two short of the top)."""
    lo, hi = window
    return hi - 2 if hi - 2 > lo else None


class V:
    def __init__(self, vid, B, model="elliptical", dcost=1e-5, kernel="auto", coop_lanes=0):
        self.id, self.B, self.model, self.dcost, self.kernel, self.coop_lanes = vid, B, model, dcost, kernel, coop_lanes

    def batch(self, S):
        return self.B(S) if callable(self.B) else self.B

    def expect(self, S, B):
        """(kernel, GP, BPS, MOVE) plan_solve must pick for B on a device with S SMs."""
        coop = (self.model == "circular" and self.dcost > 0) or self.kernel == "coop" or \
               (self.kernel == "auto" and B <= COOP_MAX_BATCH)
        if not coop:
            return ("thread", 8 if self.dcost > 0 else 7)
        gp = _gp(S, B, self.coop_lanes)
        move = 0 if self.dcost == 0 else (2 if self.model == "circular" else 1)
        return ("coop", gp, _bps(S, B, gp), move)


VARIANTS = [
    V("thread-sweeps8", 65536),                                   # the benchmark's configuration (AUTO)
    V("thread-sweeps7", 1000, dcost=0.0, kernel="thread"),
    V("coop-gp32-bps1-move0", lambda S: _top(_coop_window(S, 32, 1)), dcost=0.0),
    V("coop-gp32-bps1-move1", lambda S: _top(_coop_window(S, 32, 1))),
    V("coop-gp8-bps1-move0", lambda S: _top(_coop_window(S, 8, 1)), dcost=0.0),
    V("coop-gp8-bps1-move1", lambda S: _top(_coop_window(S, 8, 1))),
    V("coop-gp8-bps2-move0", lambda S: _top(_coop_window(S, 8, 2)), dcost=0.0),
    V("coop-gp8-bps2-move1", lambda S: _top(_coop_window(S, 8, 2))),
    V("coop-gp32-bps2-move1", lambda S: 8 * S + 62 if 8 * S + 62 <= COOP_MAX_BATCH else None, coop_lanes=32),
    V("circular-coop-gp32-bps1-move2", 1, model="circular"),
    V("circular-coop-gp8-bps1-move2", lambda S: _top(_coop_window(S, 8, 1, cap=32 * S)), model="circular"),
    V("circular-coop-gp8-bps2-move2", lambda S: max(COOP_MAX_BATCH - 2, 32 * S + 30), model="circular"),
    V("circular-thread-sweeps7", 1000, model="circular", dcost=0.0, kernel="thread"),
    V("circular-coop-gp8-bps1-move0", lambda S: _top(_coop_window(S, 8, 1)), model="circular", dcost=0.0),
]
