"""GPU parity tests for pc_sample_batch (genSample on the device) and pc_expand_batch (one speculative batch of the
expansion loop with no per-sample host traffic)."""
import numpy as np
import pytest

import oracle
from pointcloudtraj_b200 import PC_QUERY_AUTO, PcError, PcRadiusParams, PcSampler, PointCloudIndex, synth

pytestmark = pytest.mark.gpu

START, END = (0.0, 0.0, 2.0), (40.0, 10.0, 2.0)
BOX = (-50.0, 50.0, -50.0, 50.0, 0.0, 5.0)
PRM = dict(safety_margin=0.6, search_margin=0.25, max_radius=1.5, sample_range=30.0)


def _samplers(inlier, goal, state=1):
    a = (START, END, BOX, PRM["sample_range"], PRM["safety_margin"], inlier, goal)
    return PcSampler.make(*a, engine_state=state), oracle.Sampler.make(*a, engine_state=state)


@pytest.fixture(scope="module")
def ix():
    h = PointCloudIndex(max_points=1 << 18, device=0)
    yield h
    h.close()


@pytest.mark.parametrize("goal,inlier,k", [(0.15, 0.3, 1_000_003), (0.0, 0.5, 70_001), (1.0, 0.0, 50_000), (0.55, 0.45, 300_000),
                                           (0.15, 0.3, 1), (0.15, 0.3, 7), (0.9, 0.05, 8192 * 3)])
def test_sample_stream_vs_oracle(ix, goal, inlier, k):
    """Bit-identical samples and engine state, whatever the share of one-uniform (goal) samples in the stream."""
    ps, os_ = _samplers(inlier, goal)
    got = ix.sample_batch(ps, k)
    want = oracle.gen_samples(os_, k)
    assert (got == want).all()
    assert ps.engine_state == os_.engine_state
    # the stream continues where the batch stopped: a second batch from the returned state
    got2 = ix.sample_batch(ps, 1000)
    want2 = oracle.gen_samples(os_, 1000)
    assert (got2 == want2).all() and ps.engine_state == os_.engine_state


@pytest.mark.skipif(not oracle.have_planner_reference(), reason="needs the upstream pointcloudTraj planner compiled into oracle/_ref (make -C oracle REF=<pointcloudTraj checkout>)")
def test_sample_stream_vs_compiled_reference(ix):
    """Against k calls of the UNMODIFIED genSample (corridor_finder.cpp:333-383) on the planner's own engine (eng(0))."""
    ref = oracle.PlannerReference(**PRM)
    ref.set_pt(START, END, BOX, 30.0, 1000, 0.3, 0.15)
    want = ref.gen_samples(400_000)
    ps, _ = _samplers(0.3, 0.15)
    got = ix.sample_batch(ps, 400_000)
    assert (got == want).all()


def test_sample_bad_arguments(ix):
    ps, _ = _samplers(0.3, 0.15, state=0)
    with pytest.raises(PcError):
        ix.sample_batch(ps, 10)
    ps, _ = _samplers(0.3, 0.15)
    assert ix.sample_batch(ps, 0).shape == (0, 3) and ps.engine_state == 1


def _host_pipeline(ix, nodes, node_coord, node_radius, node_valid, osamp, P, z_l, safety_margin, k):
    """The same batch through the buffer API: host samples, pc_nearest_batch on the node index, steering on the host,
    pc_radius_batch, the loop's filter (corridor_finder.cpp:720-731)."""
    s = oracle.gen_samples(osamp, k)
    nodes.build(node_coord.astype(np.float32))
    nn, _ = nodes.nearest(s.astype(np.float32), flags=PC_QUERY_AUTO)
    ok = (nn >= 0) & (node_valid[np.maximum(nn, 0)] != 0)
    c = oracle.steer(s, node_coord, node_radius, np.maximum(nn, 0))
    r = ix.radius(c.astype(np.float32), P)
    keep = ok & ~((c[:, 2] < z_l) | (r.astype(np.float64) < safety_margin))
    return c[keep], r[keep], nn[keep]


@pytest.mark.parametrize("n_nodes,k", [(1, 5000), (37, 4096), (3000, 20_000), (3000, 200_000), (20_000, 1_000_000), (500, 5_000_000)])
def test_expand_batch_vs_buffer_api(ix, n_nodes, k):
    """(the 5 M-sample case runs as three pipelined chunks; up to 2^26 sample-node pairs the nearest vertex is found by exact
    brute force instead of through the node index: the first three cases)"""
    pts, half = synth.forest_cloud(200_000, seed=6, variant="J", return_half=True)
    ix.build(pts)
    rng = np.random.default_rng(n_nodes)
    # a plausible frozen tree: nodes scattered around the start, float32 radii, a few invalid ones
    node_coord = np.column_stack([rng.uniform(-25, 25, n_nodes), rng.uniform(-25, 25, n_nodes), rng.uniform(0.7, 4.0, n_nodes)])
    node_coord[0] = START
    node_radius = rng.uniform(0.6, 1.25, n_nodes).astype(np.float32)
    node_valid = (rng.uniform(size=n_nodes) > 0.02).astype(np.uint8)
    node_valid[0] = 1
    P = PcRadiusParams.make(PRM["search_margin"], PRM["max_radius"], PRM["sample_range"], START)
    ps, os_ = _samplers(0.3, 0.15, state=12345)
    with PointCloudIndex(max_points=1 << 16, device=0) as nodes, PointCloudIndex(max_points=1 << 16, device=0) as nodes_h:
        cand = ix.expand_batch(nodes, node_coord, node_radius, node_valid, ps, P, BOX[4], PRM["safety_margin"], k)
        c, r, nn = _host_pipeline(ix, nodes_h, node_coord, node_radius, node_valid, os_, P, BOX[4], PRM["safety_margin"], k)
        assert len(cand) == len(c) and 0 < len(c) < k
        assert (cand["center"] == c).all() and (cand["radius"] == r).all() and (cand["nearest"] == nn).all()
        assert ps.engine_state == os_.engine_state
        # capacity overflow: the count is still reported
        with pytest.raises(PcError) as e:
            ix.expand_batch(nodes, node_coord, node_radius, node_valid, ps, P, BOX[4], PRM["safety_margin"], k, cap=3, advance=False)
        assert e.value.code == -4


def test_expand_batch_edge_cases(ix):
    P = PcRadiusParams.make(PRM["search_margin"], PRM["max_radius"], PRM["sample_range"], START)
    node_coord = np.array([START, (3.0, 1.0, 2.0)], np.float64)
    node_radius = np.array([1.0, 0.8], np.float32)
    with PointCloudIndex(max_points=1 << 12, device=0) as nodes:
        # empty cloud: radiusSearch answers max_radius - search_margin everywhere (corridor_finder.cpp:118-120), nothing is dropped
        # for its radius; candidates below the floor still are
        ix.build(np.zeros((0, 3), np.float32))
        ps, os_ = _samplers(0.3, 0.15)
        cand = ix.expand_batch(nodes, node_coord, node_radius, np.ones(2, np.uint8), ps, P, BOX[4], PRM["safety_margin"], 3000)
        s = oracle.gen_samples(os_, 3000)
        d0 = ((s.astype(np.float32).astype(np.float64) - node_coord[0].astype(np.float32)) ** 2).sum(1)
        d1 = ((s.astype(np.float32).astype(np.float64) - node_coord[1].astype(np.float32)) ** 2).sum(1)
        nn = (d1 < d0).astype(np.int32)
        c = oracle.steer(s, node_coord, node_radius, nn)
        keep = ~(c[:, 2] < BOX[4])
        assert len(cand) == int(keep.sum()) and (cand["center"] == c[keep]).all() and (cand["nearest"] == nn[keep]).all()
        assert (cand["radius"] == np.float32(PRM["max_radius"] - PRM["search_margin"])).all()
        # no valid vertex: every sample is dropped, the engine still advances past the k samples
        ps2, os2 = _samplers(0.3, 0.15, state=99)
        cand = ix.expand_batch(nodes, node_coord, node_radius, np.zeros(2, np.uint8), ps2, P, BOX[4], PRM["safety_margin"], 1000)
        oracle.gen_samples(os2, 1000)
        assert len(cand) == 0 and ps2.engine_state == os2.engine_state
        # every sample is the goal (goal_ratio 1): k identical candidates steered from the same vertex
        ps3, _ = _samplers(0.0, 1.0)
        cand = ix.expand_batch(nodes, node_coord, node_radius, np.ones(2, np.uint8), ps3, P, BOX[4], PRM["safety_margin"], 500)
        assert len(cand) == 500 and (cand["center"] == cand["center"][0]).all()
        # k = 0, and bad arguments
        ps4, _ = _samplers(0.3, 0.15)
        assert len(ix.expand_batch(nodes, node_coord, node_radius, np.ones(2, np.uint8), ps4, P, BOX[4], PRM["safety_margin"], 0)) == 0 and ps4.engine_state == 1
        with pytest.raises(PcError):
            ix.expand_batch(ix, node_coord, node_radius, np.ones(2, np.uint8), ps4, P, BOX[4], PRM["safety_margin"], 10)      # nodes == cloud
        with pytest.raises(PcError):
            ix.expand_batch(nodes, node_coord[:0], node_radius[:0], np.ones(0, np.uint8), ps4, P, BOX[4], PRM["safety_margin"], 10)   # empty node set


def test_sample_batch_device_buffer(ix):
    """PC_DEVICE: the samples stay in device memory (a torch tensor), the engine state still comes back to the host."""
    import ctypes as C
    import torch
    from pointcloudtraj_b200 import PC_DEVICE
    ps, os_ = _samplers(0.3, 0.15, state=777)
    k = 123_457
    out = torch.empty((k, 3), dtype=torch.float64, device="cuda:0")
    torch.cuda.synchronize()
    st = C.c_uint32(0)
    rc = ix._L.pc_sample_batch(ix._h, C.byref(ps), k, PC_DEVICE, C.c_void_p(out.data_ptr()), C.byref(st))
    assert rc == 0
    ix.sync()
    want = oracle.gen_samples(os_, k)
    assert (out.cpu().numpy() == want).all() and st.value == os_.engine_state
