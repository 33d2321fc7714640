"""Checkpoints without a GPU: a frame-store buffer saved mid-trajectory and loaded into a fresh buffer continues exactly
like the original (over the NumPy model of the device ring), a reloaded uniform sampler draws the same keys, the
directory protocol ignores interrupted saves and keeps the newest checkpoint_duration checkpoints, and the digest
formula matches a plain-Python restatement."""
import os

import numpy as np
import pytest

from test_frame_store_host import KeysOnly, NumpyFrames


class NumpyFramesIO(NumpyFrames):
    """NumpyFrames with the checkpoint calls of the device frame store (read/write of frames and slots, digest)."""

    @property
    def dtype(self):
        return self.ring.dtype

    @property
    def frame_bytes(self):
        return int(np.prod(self.frame_shape)) * self.dtype.itemsize

    def read_frames(self, lo, hi):
        assert 0 <= hi - lo <= self.n_frames
        return np.asarray([self.ring[f % self.n_frames] for f in range(lo, hi)], self.dtype).reshape(
            (hi - lo,) + self.frame_shape)

    def write_frames(self, lo, frames):
        assert len(frames) <= self.n_frames
        for i, f in enumerate(frames):
            self.ring[(lo + i) % self.n_frames] = f

    def read_slots(self, lo, n):
        sc = self.scalars[lo:lo + n]
        return (self.rows[lo:lo + n].copy(), None, np.asarray([s[0] for s in sc], np.int32),
                np.asarray([s[1] for s in sc], np.float64), np.asarray([s[2] for s in sc], np.uint8),
                np.asarray([s[3] for s in sc], np.uint8))

    def write_slots(self, lo, rows, next_state, a, r, d, e):
        assert next_state is None
        self.rows[lo:lo + len(rows)] = rows
        for i in range(len(rows)):
            self.scalars[lo + i] = (int(a[i]), float(r[i]), bool(d[i]), bool(e[i]))

    def digest(self, n_live, lo, hi):
        from idqn_b200 import checkpoint as ckpt
        s, _, a, r, d, e = self.read_slots(0, n_live)
        return [ckpt.frames_digest(self.read_frames(lo, hi)), ckpt.digest(s)] + [ckpt.digest(x) for x in (a, r, d, e)]


def frame_buffer(stack, n, cap, sampler=None, checkpoint_duration=4):
    from idqn_b200.sample_collection.replay_buffer import ReplayBuffer

    class HostFrameBuffer(ReplayBuffer):
        _frame_store_type = NumpyFramesIO

    return HostFrameBuffer(sampler or KeysOnly(), 8, cap, stack, n, 0.9, checkpoint_duration, compress=False,
                           frame_store=True)


def short_episodes(seed, n):
    from idqn_b200.sample_collection.replay_buffer import TransitionElement
    rng = np.random.default_rng(seed)
    out = []
    for t in range(n):
        end = t % 2 == 1  # two-step episodes ending alternately in a terminal and a truncation: the ring grows
        out.append(TransitionElement(rng.integers(0, 256, (3, 5)).astype(np.uint8), int(rng.integers(0, 6)),
                                     float(rng.integers(-1, 2)), end and t % 4 == 1, end))
    return out


@pytest.mark.parametrize("stack,n", [(4, 1), (1, 3), (2, 2)])
def test_frame_buffer_resumes_exactly(tmp_path, stack, n):
    trs = short_episodes(stack * 10 + n, 160)
    a = frame_buffer(stack, n, 8)
    cut = 70 + 1  # the trajectory holds one transition of an unfinished episode
    for tr in trs[:cut]:
        a.add(tr)
    assert a._store.grows >= 1 and len(a._trajectory) > 0
    a.save(str(tmp_path))
    b = frame_buffer(stack, n, 8)
    b.load(str(tmp_path))
    assert b._store.n_frames == a._store.n_frames
    grows0 = a._store.grows
    for step, tr in enumerate(trs[cut:]):
        a.add(tr)
        b.add(tr)
        sa, sb = a._store, b._store
        assert (b.add_count, b._next_frame_id, list(b._frame_ids), list(b._live_min)) == \
               (a.add_count, a._next_frame_id, list(a._frame_ids), list(a._live_min)), step
        assert sb.n_frames == sa.n_frames and sb.grows == sa.grows - grows0, step
        n_live = min(a.add_count, 8)
        np.testing.assert_array_equal(sb.rows[:n_live], sa.rows[:n_live])
        assert sb.scalars[:n_live] == sa.scalars[:n_live]
        lo = a._lowest_frame_in_use()
        np.testing.assert_array_equal(sb.read_frames(lo, a._next_frame_id), sa.read_frames(lo, a._next_frame_id))


def test_frame_buffer_load_refuses_a_corrupt_or_different_store(tmp_path):
    a = frame_buffer(2, 2, 8)
    for tr in short_episodes(1, 40):
        a.add(tr)
    a.save(str(tmp_path))
    with pytest.raises(ValueError, match="max_capacity"):
        frame_buffer(2, 2, 16).load(str(tmp_path))
    with pytest.raises(ValueError, match="update_horizon"):
        frame_buffer(2, 3, 8).load(str(tmp_path))
    used = frame_buffer(2, 2, 8)
    used.add(short_episodes(1, 1)[0])
    with pytest.raises(ValueError, match="nothing has been added"):
        used.load(str(tmp_path))
    rows = np.load(tmp_path / "rows.npy")
    rows[0, -1] += 1
    np.save(tmp_path / "rows.npy", rows)
    with pytest.raises(ValueError, match="replay digest mismatch in next_state/rows"):
        frame_buffer(2, 2, 8).load(str(tmp_path))


def test_reloaded_uniform_sampler_draws_the_same_keys(tmp_path):
    from idqn_b200.sample_collection.samplers import UniformSamplingDistribution
    s = UniformSamplingDistribution(seed=3)
    for k in range(50):
        s.add(k)
    for k in (0, 7, 3, 49, 20):
        s.remove(k)
    s.sample(32)
    s.save(str(tmp_path))
    t = UniformSamplingDistribution(seed=99)
    t.load(str(tmp_path))
    assert t._key_to_index == s._key_to_index and t._index_to_key == s._index_to_key
    for _ in range(5):
        np.testing.assert_array_equal(t.sample(32), s.sample(32))
    s.remove(11), t.remove(11)
    np.testing.assert_array_equal(t.sample(64), s.sample(64))


def test_directory_protocol(tmp_path):
    from idqn_b200 import checkpoint as ckpt
    root = str(tmp_path)
    assert ckpt.latest_checkpoint(root) is None
    for epoch in range(5):
        tmp = ckpt.begin(root, str(epoch))
        ckpt.write_json(os.path.join(tmp, "loop.json"), {"epoch": epoch})
        os.makedirs(os.path.join(tmp, "agent"))
        np.save(os.path.join(tmp, "agent", "x.npy"), np.arange(epoch))
        ckpt.commit(root, str(epoch), keep=3)
    assert sorted(os.listdir(root)) == ["2", "3", "4"]
    latest = ckpt.latest_checkpoint(root)
    assert latest == os.path.join(root, "4")
    ckpt.verify(latest)
    m = ckpt.read_json(os.path.join(latest, ckpt.MANIFEST))
    assert m["files"] == {"loop.json": os.path.getsize(os.path.join(latest, "loop.json")),
                          os.path.join("agent", "x.npy"): os.path.getsize(os.path.join(latest, "agent", "x.npy"))}
    # an interrupted save (still under its .tmp name, even with a manifest) and a directory without a manifest
    tmp = ckpt.begin(root, "9")
    ckpt.write_json(os.path.join(tmp, ckpt.MANIFEST), {"format": ckpt.FORMAT_VERSION, "serial": 99, "files": {}})
    os.makedirs(os.path.join(root, "10"))
    assert ckpt.latest_checkpoint(root) == latest
    with open(os.path.join(latest, "loop.json"), "a") as f:
        f.write(" ")
    with pytest.raises(ValueError, match="loop.json"):
        ckpt.verify(latest)


def _splitmix64(z):
    M = (1 << 64) - 1
    z ^= z >> 30
    z = (z * 0xBF58476D1CE4E5B9) & M
    z ^= z >> 27
    z = (z * 0x94D049BB133111EB) & M
    return z ^ (z >> 31)


def test_digest_formula():
    from idqn_b200 import checkpoint as ckpt
    # SplitMix64's first output for seed 0 (its state after one step is the golden gamma)
    assert _splitmix64(0x9E3779B97F4A7C15) == 0xE220A8397B1DCDAF
    assert ckpt.digest(bytes(8)) == 0xE220A8397B1DCDAF ^ _splitmix64(8)
    assert ckpt.digest(b"") == 0
    data = bytes(range(1, 20))  # 19 bytes: two whole words and three zero-padded bytes
    words = [int.from_bytes(data[i:i + 8].ljust(8, b"\0"), "little") for i in range(0, 24, 8)]
    want = sum(_splitmix64((w + (i + 1) * 0x9E3779B97F4A7C15) % (1 << 64)) for i, w in enumerate(words)) % (1 << 64)
    assert ckpt.digest(data) == want ^ _splitmix64(19)
    assert ckpt.digest(np.frombuffer(data, np.uint8)) == ckpt.digest(data)
    # frames: each padded to a multiple of 8 bytes, then one stream
    f = np.arange(2 * 5, dtype=np.uint8).reshape(2, 5)
    assert ckpt.frames_digest(f) == ckpt.digest(bytes(f[0]) + bytes(3) + bytes(f[1]) + bytes(3))
