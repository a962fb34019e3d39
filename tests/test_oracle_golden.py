"""CPU: the oracle (oracle/lift_oracle.py) reproduces the golden vectors that oracle/gen_golden.py recorded from the
REAL reference functions (fiery/models/fiery.py:109-128,193-208,221-273; fiery/utils/geometry.py:39-58,283-314).
This is what pins the oracle on a box where /root/reference does not exist."""
import numpy as np
import pytest
import torch

from oracle import lift_oracle as O
from tests._cases import GOLDEN_CASES, GOLDEN_THREADS, build_case, case_id, golden_str, golden_tag, sha

FAST_CASES = [c for c in GOLDEN_CASES if c[0] in ("cfg1_tiny", "cfg2_static_lss")]


@pytest.fixture(autouse=True, scope="module")
def recorded_thread_count():
    """The oracle's CPU ops run with the thread count the golden vectors were recorded with, whatever the host's core count."""
    before = torch.get_num_threads()
    torch.set_num_threads(GOLDEN_THREADS)
    yield
    torch.set_num_threads(before)


@pytest.mark.parametrize("name", ["singletons", "one_voxel", "long_runs", "first_last_boundaries", "random_runs",
                                  "empty", "single_row"])
def test_cumsum_segment_sum_matches_reference(golden_vs, name):
    feats = torch.from_numpy(golden_vs[f"{name}__feats"]).requires_grad_(True)
    coords = torch.from_numpy(golden_vs[f"{name}__coords"])
    ranks = torch.from_numpy(golden_vs[f"{name}__ranks"])
    sums, kept = O.CumsumSegmentSum.apply(feats, coords, ranks)
    assert torch.equal(sums.detach(), torch.from_numpy(golden_vs[f"{name}__ref_sum"]))      # same torch ops: bit-equal
    assert torch.equal(kept, torch.from_numpy(golden_vs[f"{name}__ref_coords"]))
    if ranks.numel():
        sums.backward(torch.from_numpy(golden_vs[f"{name}__gout"]))
        assert np.array_equal(feats.grad.numpy(), golden_vs[f"{name}__ref_grad"])
        exact = O.direct_segment_sum(feats.detach(), ranks)
        assert torch.allclose(sums.detach().double(), exact, rtol=1e-4, atol=1e-5)


@pytest.mark.parametrize("cname", ["cfg1_tiny", "cfg2_static_lss", "cfg4_pon"])
def test_bev_grid_matches_reference(golden_lift, cname):
    from fiery_b200.synthetic import CONFIGS
    cfg = CONFIGS[cname]
    res, start, dim = O.bev_grid(cfg.x_bound, cfg.y_bound, cfg.z_bound)
    assert np.array_equal(res.numpy(), golden_lift[f"{cname}__resolution"])
    assert np.array_equal(start.numpy(), golden_lift[f"{cname}__start"])
    assert np.array_equal(dim.numpy(), golden_lift[f"{cname}__dimension"])
    assert tuple(dim[:2].tolist()) == cfg.bev_hw


@pytest.mark.parametrize("case", FAST_CASES, ids=case_id)
def test_indices_match_reference(golden_lift, case):
    """Integer voxel indices: bit-exact against the reference, via torch ops and via the explicit fp32 order."""
    cfg, K, E, _, _ = build_case(case)
    tag = golden_tag(case)
    oracle = O.LiftOracle.from_config(cfg)
    comb, trans = O.compose_calibration(K, E)
    assert np.array_equal(trans.numpy(), golden_lift[f"{tag}__translation"])
    if not np.array_equal(comb.numpy(), golden_lift[f"{tag}__combined"]):
        # another LAPACK build may round R @ K^-1 differently (SURVEY.md section 7, hard part 2-iv): pin it
        comb = torch.from_numpy(golden_lift[f"{tag}__combined"])
    idx, keep = oracle.point_indices(K, E, combined=comb)
    assert sha(idx.numpy()) == golden_str(golden_lift[f"{tag}__idx_sha256"])
    assert sha(keep.numpy()) == golden_str(golden_lift[f"{tag}__keep_sha256"])
    assert np.array_equal(keep.sum(1).numpy(), golden_lift[f"{tag}__kept_points"])
    # explicit-order restatement (the arithmetic of the CUDA kernels)
    fr = oracle.frustum
    ego = O.frustum_to_ego_explicit(fr[0, 0, :, 0].numpy(), fr[0, :, 0, 1].numpy(), fr[:, 0, 0, 2].numpy(),
                                    comb.numpy(), trans.numpy())
    idx_e, keep_e = O.voxel_indices_explicit(ego, oracle.start.numpy(), oracle.resolution.numpy(), oracle.dimension.numpy())
    assert np.array_equal(idx_e.reshape(idx.shape), idx.numpy())
    assert np.array_equal(keep_e.reshape(keep.shape), keep.numpy())
    if "cfg1" in case[0]:
        assert np.array_equal(idx.numpy().astype(np.int32), golden_lift[f"{tag}__idx"])


@pytest.mark.parametrize("case", FAST_CASES, ids=case_id)
def test_explicit_calibration_matches_torch(golden_lift, case):
    """R @ inverse(K) written out as LU + solve + ordered matmul equals the reference's torch result for pinhole K."""
    cfg, K, E, _, _ = build_case(case)
    comb, trans = O.compose_calibration_explicit(K.numpy(), E.numpy())
    assert np.array_equal(comb, golden_lift[f"{golden_tag(case)}__combined"])
    assert np.array_equal(trans, golden_lift[f"{golden_tag(case)}__translation"])


@pytest.mark.parametrize("case", FAST_CASES, ids=case_id)
def test_lift_matches_reference(golden_lift, case):
    cfg, K, E, head, gout = build_case(case)
    tag = golden_tag(case)
    oracle = O.LiftOracle.from_config(cfg)
    comb = torch.from_numpy(golden_lift[f"{tag}__combined"])
    head.requires_grad_(True)
    bev = oracle.lift(head, K, E, combined=comb)
    bev.backward(gout)
    pick = golden_lift[f"{tag}__bev_pick"]
    ref = golden_lift[f"{tag}__bev_ref_at_pick"]
    got = bev.detach().flatten()[pick].numpy()
    scale = float(np.abs(ref).max())
    # argsort order (fiery.py:257) may differ between builds, so the cumsum rounding may too: tolerance, not bits
    assert np.abs(got - ref).max() <= 2e-5 * scale
    assert np.allclose(bev.detach().double().sum((1, 2, 3)).numpy(), golden_lift[f"{tag}__bev_sum"], rtol=1e-5)
    assert np.allclose(bev.detach().double().flatten(1).norm(dim=1).numpy(), golden_lift[f"{tag}__bev_norm"], rtol=1e-6)
    gref = golden_lift[f"{tag}__grad_ref_at_pick"]
    ggot = head.grad.reshape(-1)[golden_lift[f"{tag}__grad_pick"]].numpy()
    assert np.abs(ggot - gref).max() <= 2e-5 * float(np.abs(gref).max())
    occupied = bev.detach().abs().sum(1) > 0
    assert np.array_equal(occupied.flatten(1).sum(1).numpy(), golden_lift[f"{tag}__occupied_count"])
    if "cfg1" in case[0]:
        assert O.normwise_error(bev, torch.from_numpy(golden_lift[f"{tag}__bev_ref"])) < 1e-6
        assert O.normwise_error(head.grad, torch.from_numpy(golden_lift[f"{tag}__grad_ref"])) < 1e-6


def test_exact_pooling_is_the_adjudicator(golden_lift):
    """The fp64 direct pooling (oracle variant O3) agrees with the recorded one, and the reference's cumsum path is the
    noisier of the two (SURVEY.md section 7, hard part 1)."""
    case = ("cfg1_tiny", 0.02, 1)
    cfg, K, E, head, _ = build_case(case)
    tag = golden_tag(case)
    oracle = O.LiftOracle.from_config(cfg)
    exact = oracle.lift_exact(head, K, E, combined=torch.from_numpy(golden_lift[f"{tag}__combined"]))
    assert O.normwise_error(exact, torch.from_numpy(golden_lift[f"{tag}__bev_exact"])) < 1e-12
    ref = torch.from_numpy(golden_lift[f"{tag}__bev_ref"])
    assert O.normwise_error(ref, exact) < 1e-4


@pytest.mark.parametrize("case", FAST_CASES, ids=case_id)
def test_c_restatement_agrees(golden_lift, case):
    """oracle/lift_oracle.c (gcc -ffp-contract=off) reproduces the reference's voxel indices bit for bit and its exact
    pooling agrees with the torch fp64 pooling."""
    from oracle import c_oracle
    cfg, K, E, head, _ = build_case(case)
    tag = golden_tag(case)
    oracle = O.LiftOracle.from_config(cfg)
    comb = golden_lift[f"{tag}__combined"]
    trans = golden_lift[f"{tag}__translation"]
    fr = oracle.frustum
    off = (oracle.start - oracle.resolution / 2.0).numpy()
    idx, keep = c_oracle.voxel_indices(fr[0, 0, :, 0].numpy(), fr[0, :, 0, 1].numpy(), fr[:, 0, 0, 2].numpy(), comb, trans, off,
                                       oracle.resolution.numpy(), oracle.dimension.numpy())
    assert sha(idx) == golden_str(golden_lift[f"{tag}__idx_sha256"])
    assert sha(keep) == golden_str(golden_lift[f"{tag}__keep_sha256"])
    D, C = cfg.depth_bins, cfg.out_channels
    prob = head[:, :D].double().softmax(1).numpy()
    X, Y = cfg.bev_hw
    bev = c_oracle.pool_exact(prob, head[:, D:].double().numpy(), idx, keep, cfg.n_cameras, X, Y)
    exact = oracle.lift_exact(head, K, E, combined=torch.from_numpy(comb))
    assert O.normwise_error(torch.from_numpy(bev), exact) < 1e-13


@pytest.mark.parametrize("case", __import__("tests._cases", fromlist=["BENCH_CASES"]).BENCH_CASES, ids=case_id)
def test_indices_at_bench_configs_match_reference(golden_lift, case):
    """The configurations bench.py quotes (8 / 9 / 12 frames): the oracle's voxel indices of every frame -- torch ops and the C
    restatement -- hash to what the reference recorded (fiery.py:236-256)."""
    from oracle import c_oracle
    cfg, K, E, _, _ = build_case(case)
    tag = golden_tag(case)
    oracle = O.LiftOracle.from_config(cfg)
    comb, trans = golden_lift[f"{tag}__combined"], golden_lift[f"{tag}__translation"]
    ce, te = O.compose_calibration_explicit(K.numpy(), E.numpy())
    assert np.array_equal(ce, comb) and np.array_equal(te, trans)
    idx, keep = oracle.point_indices(K, E, combined=torch.from_numpy(comb))
    assert sha(idx.numpy()) == golden_str(golden_lift[f"{tag}__idx_sha256"])
    assert sha(keep.numpy()) == golden_str(golden_lift[f"{tag}__keep_sha256"])
    fr = oracle.frustum
    off = (oracle.start - oracle.resolution / 2.0).numpy()
    idx_c, keep_c = c_oracle.voxel_indices(fr[0, 0, :, 0].numpy(), fr[0, :, 0, 1].numpy(), fr[:, 0, 0, 2].numpy(), comb, trans, off,
                                           oracle.resolution.numpy(), oracle.dimension.numpy())
    assert sha(idx_c) == golden_str(golden_lift[f"{tag}__idx_sha256"])
    assert sha(keep_c) == golden_str(golden_lift[f"{tag}__keep_sha256"])
