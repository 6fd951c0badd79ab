"""The default configuration (floor SOR at k = 50 included) at the benchmark's batch shape: 16 full-size WFOV frames in
flight, 8 frames per launch, so every segment of a batched neighbour-search launch carries a frame.  Two distinct
seeded frames, cycled; every frame must equal the oracle's composition for its input.  Run with the grid and with the
voxel-brick index (KP_KNN_VBI=1) as level 0 of the neighbour searches, which share the candidate buffer code."""

import numpy as np
import pytest

from kinectpy_b200 import synth
from kinectpy_b200.pipeline import FramePipeline, PipelineConfig

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def frames_and_refs(oracle):
    depth, tab, T = synth.render_sequence(synth.WFOV, 2, 3)
    T_fuse = synth.scale_extrinsics(T, 1e-3)
    T_icp = np.stack([synth.perturbed_extrinsic(T_fuse[s], 0.3, (3, -3, 3), unit_scale=1e-3) if s else T_fuse[s] for s in range(3)])
    cfg = PipelineConfig(n_sensors=3, pixels=synth.WFOV.pixels, n_streams=16)
    refs = [oracle.frame_pipeline(cfg, depth[f], tab, T_fuse, T_icp) for f in range(2)]
    return cfg, depth, tab, T_fuse, T_icp, refs


@pytest.mark.parametrize("knn_vbi", ["0", "1"])
def test_bench_batch_shape_matches_oracle(frames_and_refs, knn_vbi, monkeypatch):
    cfg, depth, tab, T_fuse, T_icp, refs = frames_and_refs
    monkeypatch.setenv("KP_KNN_VBI", knn_vbi)
    pipe = FramePipeline(cfg, tab, T_fuse, T_icp)
    assert pipe.frames_in_flight() == (8, 2)
    got = pipe.run(np.ascontiguousarray(depth[np.arange(16) % 2]), want_points=True)
    pipe.close()
    assert len(got) == 16
    for f, g in enumerate(got):
        ref = refs[f % 2]
        assert (g.n_fused, g.n_voxel, g.n_sor, g.n_floor_inliers, g.n_out) == \
            (ref["n_fused"], ref["n_voxel"], ref["n_sor"], ref["n_floor_inliers"], len(ref["points"])), f
        assert np.array_equal(g.points, ref["points"]), f
        for i in range(2):
            assert np.abs(g.icp_T[i] - ref["icp"][i]["T"]).max() < 1e-4, (f, i)
