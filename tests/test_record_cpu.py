"""CPU: the Vm recorder's host-side pieces — the crossing rule restated on the host (the reference the GPU tests compare the device
maps with) and the exact merge of per-rank results (slabs.merge_activation / merge_traces)."""
import numpy as np
import pytest

from sph_sm_monodomain_b200 import slabs


def host_crossings(series, vm_up, vm_down, n):
    """The recorder's rule over (step, pre, post) triples: pre = Vm the step started from, post = Vm it produced (float32)."""
    up, down = np.float32(vm_up), np.float32(vm_down)
    out = {k: np.full(n, -1, np.int32) for k in ("first_up", "last_up", "last_down")}
    out["n_up"] = np.zeros(n, np.int32)
    for step, pre, post in series:
        pre, post = np.asarray(pre, np.float32), np.asarray(post, np.float32)
        u = (pre < up) & (post >= up)
        d = (pre >= down) & (post < down)
        out["first_up"][u & (out["first_up"] < 0)] = step
        out["last_up"][u] = step
        out["n_up"][u] += 1
        out["last_down"][d] = step
    return out


def _series(vm):
    """(step, pre, post) of a trajectory vm[0..T] with no change between steps: step t goes from vm[t-1] to vm[t]."""
    return [(t, vm[t - 1], vm[t]) for t in range(1, len(vm))]


def test_rule_on_synthetic_series():
    t = np.arange(0, 201, dtype=np.float32)
    vm = np.stack([np.sin(t * np.float32(2 * np.pi / 50)) * np.float32(2.0),  # period 50, amplitude 2
                   np.full_like(t, 0.5),                                       # never reaches the threshold
                   np.minimum(t, np.float32(10.0))], axis=1).astype(np.float32)  # rises once, never falls
    m = host_crossings(_series(vm), 1.0, 1.0, 3)
    # particle 0: sin(2 pi t / 50) * 2 >= 1 first at t = 5 (2 sin(0.628) = 1.18), crosses again every 50 steps
    assert m["first_up"][0] == 5 and m["n_up"][0] == 4 and m["last_up"][0] == 155
    assert m["last_down"][0] == 171  # 2 sin(2 pi 171/50) = 0.96 < 1 after 2 sin(2 pi 170/50) = 1.18
    assert m["first_up"][1] == m["last_up"][1] == m["last_down"][1] == -1 and m["n_up"][1] == 0
    assert m["first_up"][2] == 1 and m["n_up"][2] == 1 and m["last_down"][2] == -1


def test_rule_hysteresis_and_edges():
    # vm_up = 1.0, vm_down = 0.5: reaching vm_up exactly is an upstroke (post >= vm_up), landing on vm_down exactly is not a
    # downstroke (post < vm_down is needed), and a particle already at / above vm_up makes no upstroke
    series = [(1, [0.0, 1.0, 2.0], [1.0, 0.0, 0.5]), (2, [1.0, 0.0, 0.5], [0.4, 1.0, 2.0])]
    m = host_crossings(series, 1.0, 0.5, 3)
    assert list(m["first_up"]) == [1, 2, 2] and list(m["last_up"]) == [1, 2, 2] and list(m["n_up"]) == [1, 1, 1]
    assert list(m["last_down"]) == [2, 1, -1]


def test_rule_nan_is_no_crossing():
    m = host_crossings([(1, [np.nan, 0.0], [2.0, np.nan])], 1.0, 1.0, 2)
    assert (m["first_up"] == -1).all() and (m["last_down"] == -1).all()


def test_merge_activation_min_max_sum_unset():
    a = {"first_up": np.array([5, -1, 7, -1], np.int32), "last_up": np.array([9, -1, 7, -1], np.int32),
         "last_down": np.array([-1, 3, 8, -1], np.int32), "n_up": np.array([2, 0, 1, 0], np.int32)}
    b = {"first_up": np.array([3, 4, -1, -1], np.int32), "last_up": np.array([4, 6, -1, -1], np.int32),
         "last_down": np.array([6, -1, 2, -1], np.int32), "n_up": np.array([1, 2, 0, 0], np.int32)}
    m = slabs.merge_activation([a, b])
    assert list(m["first_up"]) == [3, 4, 7, -1]
    assert list(m["last_up"]) == [9, 6, 7, -1]
    assert list(m["last_down"]) == [6, 3, 8, -1]
    assert list(m["n_up"]) == [3, 2, 1, 0]
    assert all(v.dtype == np.int32 for v in m.values())
    one = slabs.merge_activation([a])
    assert all(np.array_equal(one[k], a[k]) for k in a)
    with pytest.raises(ValueError):
        slabs.merge_activation([])


def test_merge_of_rank_split_equals_whole():
    """Each step's particles are integrated by exactly one rank (a random owner per step here, like migration): applying the rule
    per rank on its own particles only and merging gives the single-rank maps."""
    rng = np.random.Generator(np.random.PCG64(3))
    n, steps, nranks = 300, 120, 4
    vm = np.cumsum(rng.normal(0.0, 0.6, (steps + 1, n)).astype(np.float32), axis=0).astype(np.float32)
    whole = host_crossings(_series(vm), 0.5, -0.5, n)
    owner = rng.integers(0, nranks, (steps + 1, n))
    parts = []
    for r in range(nranks):
        ser = []
        for t in range(1, steps + 1):
            mine = owner[t] == r
            # a rank only sees the particles it integrated: the others never satisfy either condition (NaN compares false)
            ser.append((t, np.where(mine, vm[t - 1], np.nan), np.where(mine, vm[t], np.nan)))
        parts.append(host_crossings(ser, 0.5, -0.5, n))
    merged = slabs.merge_activation(parts)
    assert whole["n_up"].max() >= 2 and (whole["last_down"] >= 0).any()
    for k in slabs.ACTIVATION_KEYS:
        assert np.array_equal(merged[k], whole[k]), k


def test_merge_traces_owned_masks():
    rows, k = 3, 4
    x0 = np.arange(rows * k * 4, dtype=np.float32).reshape(rows, k, 4)
    o0 = np.array([[1, 0, 1, 0], [1, 1, 0, 0], [0, 0, 0, 0]], bool)
    o1 = np.array([[0, 1, 0, 0], [0, 0, 1, 0], [1, 1, 1, 0]], bool)
    p0 = (11, np.where(o0[..., None], x0, 0).astype(np.float32), o0)
    p1 = (11, np.where(o1[..., None], -x0, 0).astype(np.float32), o1)
    first, x, o = slabs.merge_traces([p0, p1])
    assert first == 11
    assert np.array_equal(o, o0 | o1)
    assert np.array_equal(x[o0], x0[o0]) and np.array_equal(x[o1], -x0[o1])
    assert (x[~(o0 | o1)] == 0).all()
    with pytest.raises(ValueError):
        slabs.merge_traces([p0, p0])  # an entry owned twice
    with pytest.raises(ValueError):
        slabs.merge_traces([p0, (12, p1[1], p1[2])])  # different steps
