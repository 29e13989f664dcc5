"""TEST INFRASTRUCTURE: the reference environments the parity tests compare against, on any machine.

With the compiled reference (oracle/_ref) present, the tests drive it live. Without it, each reference environment is
stood in for by the host-sim build of the device source (tests/hostsim, one env each), driven with the reference's
call pattern: make(seed) / reset() / step(a) / caller resets on terminate.

Either way, everything a reference environment returns (observations, rewards, done flags, RNG state, tile maps,
window renders) is folded into one CRC32 chain per environment, and at the end of the test the chains must equal
the ones recorded in tests/golden/reference_tapes.npz under the test's id. The committed tapes were recorded with
`PG2_RECORD_TAPES=<file>.npz pytest ...` from the stand-in at a commit whose engine and host-sim matched the live
reference bit for bit in these same tests; so a change that moves the engine and the host-sim together (they share
their source) still fails here.
"""
import os
import zlib

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
TAPES = os.path.join(HERE, "golden", "reference_tapes.npz")

# Tile map (width, height) of each game by distribution mode (None = the compiled-in mode); the reference's
# tilemap has these sizes (games/<g>/tilemap.cpp), the engine's "tiles" field is padded beyond them.
TILE_DIMS = {
    "maze": {None: (25, 25), 0: (15, 15), 1: (25, 25), 2: (31, 31)},
    "chaser": {None: (11, 11), 0: (11, 11), 1: (13, 13), 2: (19, 19)},
    "jumper": {None: (40, 40), 0: (20, 20), 1: (40, 40), 2: (45, 45)},
    "caveflyer": {None: (40, 40), 0: (20, 20), 1: (40, 40), 2: (45, 45)},
    "climber": {None: (20, 64), 0: (20, 64), 1: (20, 64)},
    "coinrun": {None: (64, 64), 0: (64, 64), 1: (64, 64)},
    "bossfight": {None: (0, 0), 0: (0, 0), 1: (0, 0)},
}


class SimRef:
    """One reference environment played by the host-sim (same constructor and methods as oracle.ref_env.RefEnv)."""

    def __init__(self, game, seed, width=None, height=None, easy_mode=None, mode=None):
        from tests.simlib import HostSim
        if easy_mode is not None:
            mode = 0 if easy_mode else 1
        self.sim = HostSim(game, 1, seed, distribution_mode=-1 if mode is None else int(mode))
        self.dims = TILE_DIMS[game][mode]
        self.width, self.height = width or 512, height or 512   # the reference's default window
        self.obs, self.regenerated = None, False

    def reset(self):
        # the host-sim resets by itself in the step that terminates: the caller's reset() returns that new level
        if not self.regenerated:
            self.obs = self.sim.reset()[0]
        self.regenerated = False
        return self.obs.copy()

    def step(self, action):
        o, r, d = self.sim.step(np.array([action], np.int32))
        self.obs, self.regenerated = o[0], bool(d[0])
        return o[0], float(r[0]), bool(d[0])

    def render(self):
        return self.sim.render_human(0, self.width, self.height)

    def rng_state(self):
        return self.sim.field("mt")[0].view(np.uint32).copy(), int(self.sim.field("mti")[0].view(np.int32)[0])

    def tiles(self):
        w, h = self.dims
        if not w:
            return np.zeros((0, 0), np.int32)
        return (self.sim.field("tiles")[0][:w * h] & 15).reshape(w, h).astype(np.int32)

    def close(self):
        self.sim.close()


class Taped:
    """A reference environment whose results are folded into chain `k` of the tape."""

    def __init__(self, env, tape):
        self.env, self.tape, self.k = env, tape, len(tape)
        tape.append(0)

    def _log(self, *vals):
        for v in vals:
            self.tape[self.k] = zlib.crc32(np.ascontiguousarray(v).tobytes(), self.tape[self.k])

    def reset(self):
        o = self.env.reset()
        self._log(o)
        return o

    def step(self, action):
        o, r, d = self.env.step(action)
        # the observation of a terminating step is replaced by reset()'s, which is logged there
        self._log(np.float32(r), np.bool_(d), b"" if d else o)
        return o, r, d

    def render(self):
        f = self.env.render()
        self._log(f)
        return f

    def rng_state(self):
        st, pos = self.env.rng_state()
        self._log(st, np.int32(pos))
        return st, pos

    def tiles(self):
        t = self.env.tiles()
        self._log(np.int32(t.shape), t.astype(np.int32))
        return t

    def close(self):
        self.env.close()


class Reference:
    """What the `reference` fixture hands a test: `RefEnv(game, seed, ...)` and the tape check at its end."""

    def __init__(self, test_id):
        from oracle import ref_env
        self.test_id, self.tape = test_id, []
        self.live = ref_env.available()
        self._cls = ref_env.RefEnv if self.live else SimRef

    def RefEnv(self, *args, **kw):
        return Taped(self._cls(*args, **kw), self.tape)

    def finish(self):
        got = np.array(self.tape, np.uint32)
        out = os.environ.get("PG2_RECORD_TAPES")
        if out:
            tapes = dict(np.load(out)) if os.path.exists(out) else {}
            tapes[self.test_id] = got
            np.savez(out, **tapes)
            return
        with np.load(TAPES) as tapes:
            assert self.test_id in tapes.files, "no recorded reference tape for %s" % self.test_id
            want = tapes[self.test_id]
        assert len(got) == len(want), "%d reference environments, the tape has %d" % (len(got), len(want))
        bad = np.nonzero(got != want)[0]
        assert not bad.size, "%s reference environments %s returned other results than recorded" % (
            "live" if self.live else "stand-in", bad[:8].tolist())
