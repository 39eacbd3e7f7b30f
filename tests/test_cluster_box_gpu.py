"""GPU parity: lmot_component_cluster / lmot_box_fit vs the reference's componentClustering / boxFitting.

Bar: BIT-EXACT 250x250 label grid and numCluster; boxes bit-exact against the reference sources linked with the
MAR contract (oracle/mar_contract.cpp) in both ruleBasedFilter modes; markers (visualisation only) to 1e-4.
"""
import numpy as np
import pytest

from oracle.recorded import ReferenceDigest

pytestmark = pytest.mark.gpu


def _bit_equal(a, ref):
    """bit-exact equality with a reference result (the large ones are stored as a digest, oracle/recorded.py)"""
    if isinstance(ref, ReferenceDigest):
        return ref.matches(a)
    a = np.ascontiguousarray(a, ref.dtype)
    return a.shape == ref.shape and np.array_equal(a.view(f"u{a.dtype.itemsize}"), np.ascontiguousarray(ref).view(f"u{a.dtype.itemsize}"))


def _elevated(ref, pts):
    e, _ = ref.ground_remove(pts)
    return e


def test_label_grid_bit_exact_hdl64(lm, ref_intended, synth):
    for seed in (1, 2):
        for ts, pts in synth.frames(synth.SceneConfig(seed=seed), 2):
            e = _elevated(ref_intended, pts)
            g_ref, k_ref = ref_intended.component_clustering(e)
            g, k = lm.component_cluster(e)
            assert k == k_ref and k > 10
            assert np.array_equal(g, g_ref)


def test_label_grid_random_clouds(lm, ref_intended):
    rng = np.random.default_rng(0)
    for it in range(12):
        n = int(rng.integers(50, 60000))
        spread = rng.choice([3.0, 10.0, 26.0, 40.0])
        e = np.zeros((n, 3), np.float32)
        centers = rng.uniform(-24, 24, (max(1, n // 200), 2))
        which = rng.integers(0, len(centers), n)
        e[:, :2] = centers[which] + rng.normal(0, spread / 20, (n, 2))
        e[::17, :2] = rng.uniform(-30, 30, (len(e[::17]), 2))          # background + out-of-ROI points
        e[:, 2] = rng.uniform(-1.5, 1.0, n)
        g_ref, k_ref = ref_intended.component_clustering(e)
        g, k = lm.component_cluster(e)
        assert k == k_ref
        assert np.array_equal(g, g_ref)


def test_label_grid_edges(lm, ref_intended):
    # empty cloud; single point (no cell reaches 2); borders and corners of the grid; one giant component
    g, k = lm.component_cluster(np.zeros((0, 3), np.float32))
    assert k == 0 and not g.any()
    one = np.array([[1.0, 1.0, 0.0]], np.float32)
    g, k = lm.component_cluster(one)
    assert k == 0 and not g.any()
    corners = []
    for x in (-24.99, 24.95, 0.0):
        for y in (-24.99, 24.95, 0.0):
            corners += [[x, y, 0.0]] * 2
    corners += [[-25.0, 3.0, 0]] * 2 + [[25.0, 3.0, 0]] * 2 + [[3.0, 24.999998, 0]] * 2
    c = np.array(corners, np.float32)
    g_ref, k_ref = ref_intended.component_clustering(c)
    g, k = lm.component_cluster(c)
    assert k == k_ref and np.array_equal(g, g_ref)
    xs = np.arange(-24.9, 24.9, 0.1, dtype=np.float32)
    dense = np.stack(np.meshgrid(xs, xs), -1).reshape(-1, 2)
    dense = np.concatenate([dense, dense], 0)
    dense = np.concatenate([dense, np.zeros((len(dense), 1), np.float32)], 1).astype(np.float32)
    g_ref, k_ref = ref_intended.component_clustering(dense)
    g, k = lm.component_cluster(dense)
    assert k == k_ref == 1 and np.array_equal(g, g_ref)
    # spiral / comb shapes that need long union-find chains
    comb = []
    for i in range(0, 240, 4):
        for j in range(0, 240):
            comb.append([-24.9 + 0.2 * i, -24.9 + 0.2 * j, 0.0])
    for i in range(0, 240):
        comb.append([-24.9 + 0.2 * i, -24.9 + (0.2 * 239 if (i // 4) % 2 else 0.0), 0.0])
    comb = np.array(comb * 2, np.float32)
    g_ref, k_ref = ref_intended.component_clustering(comb)
    g, k = lm.component_cluster(comb)
    assert k == k_ref and np.array_equal(g, g_ref)


@pytest.mark.parametrize("mode", ["intended", "o2"])
def test_boxes_bit_exact(pkg, synth, mode, ref_intended, ref_o2):
    ref = ref_intended if mode == "intended" else ref_o2
    prm = pkg.default_params()
    prm.rule_filter = pkg.RULE_INTENDED if mode == "intended" else pkg.RULE_GCC13_O2_COMPAT
    ctx = pkg.Lmot(prm)
    try:
        total = 0
        for seed in (1, 4):
            for ts, pts in synth.frames(synth.SceneConfig(seed=seed), 3):
                e = _elevated(ref, pts)
                g_ref, k_ref = ref.component_clustering(e)
                b_ref, m_ref = ref.box_fitting(e, g_ref, k_ref)
                b, m = ctx.box_fit(e, g_ref, k_ref)
                assert b.shape == b_ref.shape, (b.shape, b_ref.shape)
                assert np.array_equal(b.view(np.uint32), b_ref.view(np.uint32))
                np.testing.assert_allclose(m, m_ref, rtol=1e-4, atol=1e-4)
                total += len(b)
        assert total > 50
    finally:
        ctx.close()


def test_boxes_random_blobs(lm, ref_intended):
    """Blobs of every shape: exercises the MAR branch, the L-shape branch (|y| large) and the size filter."""
    rng = np.random.default_rng(3)
    n_l = n_mar = 0
    for it in range(8):
        pts = []
        for c in range(30):
            cx, cy = rng.uniform(-22, 22, 2)
            L, W = rng.uniform(0.3, 5.0), rng.uniform(0.3, 2.5)
            yaw = rng.uniform(-np.pi, np.pi)
            m = int(rng.integers(20, 1500))
            u = rng.uniform(-0.5, 0.5, (m, 2)) * [L, W]
            if rng.random() < 0.5:   # hollow (two visible sides)
                u[: m // 2, 1] = -W / 2
                u[m // 2:, 0] = -L / 2
            x = cx + np.cos(yaw) * u[:, 0] - np.sin(yaw) * u[:, 1]
            y = cy + np.sin(yaw) * u[:, 0] + np.cos(yaw) * u[:, 1]
            z = rng.uniform(-1.7, rng.uniform(-1.2, 0.5), m)
            pts.append(np.stack([x, y, z], 1))
        e = np.concatenate(pts).astype(np.float32)
        e = e[rng.permutation(len(e))]
        g_ref, k_ref = ref_intended.component_clustering(e)
        b_ref, m_ref = ref_intended.box_fitting(e, g_ref, k_ref)
        b, m = lm.box_fit(e, g_ref, k_ref)
        assert b.shape == b_ref.shape
        assert np.array_equal(b.view(np.uint32), b_ref.view(np.uint32))
        np.testing.assert_allclose(m, m_ref, rtol=1e-4, atol=1e-4)
        n_mar += len(b)
    assert n_mar > 20


def test_box_fit_empty(lm):
    b, m = lm.box_fit(np.zeros((0, 3), np.float32), np.zeros((250, 250), np.int32), 0)
    assert b.shape == (0, 8, 3)


def test_cluster_node_side_outputs_bit_exact(lm, ref_intended, synth):
    """SURVEY.md §8(f)3: makeClusteredCloud / setObsMsg / createCostMap (the cluster node's other topics) from the label grid."""
    rng = np.random.default_rng(3)
    for seed in (2, 9):
        for ts, pts in synth.frames(synth.SceneConfig(seed=seed), 2):
            e = _elevated(ref_intended, pts)
            e = np.concatenate([e, rng.uniform(-30, 30, (500, 3)).astype(np.float32) * [1, 1, 0.05]]).astype(np.float32)   # points outside the ROI / near the car
            g_ref, k_ref = ref_intended.component_clustering(e)
            cl_r, ob_r, cm_r = ref_intended.cluster_outputs(e, g_ref)
            g, k = lm.component_cluster(e)
            assert k == k_ref and np.array_equal(g, g_ref)
            cl, ob, cm = lm.cluster_outputs()
            assert cl.shape[0] == cl_r.shape[0] and _bit_equal(cl[:, :3], cl_r)
            assert ob.shape[0] == ob_r.shape[0] and ob.shape[0] > 100
            # [x, y, z, cluster id] in double, as setObsMsg writes them
            assert _bit_equal(np.concatenate([ob[:, :3].astype(np.float64), ob[:, 3:].astype(np.int64).astype(np.float64)], 1), ob_r)
            assert _bit_equal(cm, cm_r) and cm.max() == 100
    # twice in a row: the scratch grid is back at rest
    cl2, ob2, cm2 = lm.cluster_outputs()
    assert np.array_equal(cl2, cl) and np.array_equal(ob2, ob) and np.array_equal(cm2, cm)
