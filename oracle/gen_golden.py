"""Generate tests/golden/*.npz from the REAL reference and pin the oracle against it.  Dev container only.

Run from the repo root:   python oracle/gen_golden.py

The reference (wayveai/fiery, mounted read-only at /root/reference) is pure Python; its hot-path functions are
imported here with two stub modules for unused third-party imports (SURVEY.md appendix A) and called unbound on
a namespace carrying the attributes ``Fiery.__init__`` would have built.  This executes the reference's own
bytecode for fiery.py:109-128,193-208,221-273 and geometry.py:39-58,283-314; the encoder tail
(encoder.py:99-102 + fiery.py:216-217) is three lines applied to a synthetic head tensor because
``Encoder.__init__`` needs EfficientNet weights that are not available offline.

Two things happen:
  1. every oracle function is compared with the reference function it restates (bit-exact for integers and for
     float outputs that come from identical torch calls) -- a mismatch aborts;
  2. small golden fixtures are written so the same pin holds on a box without /root/reference.
/root/reference is never read by tests, smoke() or bench.py.
"""
from __future__ import annotations

import hashlib
import os
import sys
import types
from types import SimpleNamespace as NS

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
REFERENCE = "/root/reference"

from fiery_b200.synthetic import CONFIGS, LiftConfig, make_calibration, make_head, make_grad_bev  # noqa: E402
from oracle import lift_oracle as O  # noqa: E402


def import_reference():
    for name, attr in (("pyquaternion", "Quaternion"), ("efficientnet_pytorch", "EfficientNet")):
        if name not in sys.modules:
            m = types.ModuleType(name)
            setattr(m, attr, object)
            sys.modules[name] = m
    sys.path.insert(0, REFERENCE)
    from fiery.models.fiery import Fiery
    from fiery.utils.geometry import VoxelsSumming, calculate_birds_eye_view_parameters
    return Fiery, VoxelsSumming, calculate_birds_eye_view_parameters


def reference_self(Fiery, bev_params, cfg: LiftConfig):
    c = NS(IMAGE=NS(FINAL_DIM=cfg.final_dim),
           LIFT=NS(X_BOUND=list(cfg.x_bound), Y_BOUND=list(cfg.y_bound), Z_BOUND=list(cfg.z_bound),
                   D_BOUND=list(cfg.d_bound)))
    s = NS(cfg=c, encoder_downsample=cfg.downsample, encoder_out_channels=cfg.out_channels)
    s.bev_resolution, s.bev_start_position, s.bev_dimension = bev_params(c.LIFT.X_BOUND, c.LIFT.Y_BOUND, c.LIFT.Z_BOUND)
    s.frustum = Fiery.create_frustum(s)
    return s


def reference_lift(Fiery, s, head, K, E, cfg: LiftConfig):
    B, n = K.shape[:2]
    D, C = cfg.depth_bins, cfg.out_channels
    geom = Fiery.get_geometry(s, K, E)
    if cfg.use_depth_distribution:
        depth = head[:, :D].softmax(dim=1)                                    # encoder.py:99
        x = depth.unsqueeze(1) * head[:, D:D + C].unsqueeze(2)                # encoder.py:100
    else:
        x = head.unsqueeze(2).repeat(1, 1, D, 1, 1)                           # encoder.py:102
    x = x.view(B, n, *x.shape[1:]).permute(0, 1, 3, 4, 5, 2)                  # fiery.py:216-217
    return geom, Fiery.projection_to_birds_eye_view(s, x, geom)


def sha(a: np.ndarray) -> str:
    return hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()


def check(name, cond):
    if not cond:
        raise SystemExit(f"ORACLE != REFERENCE: {name}")
    print(f"  ok  {name}")


def rank_patterns():
    """Hand-made rank patterns for VoxelsSumming (SURVEY.md section 4 fixture 2)."""
    rng = np.random.default_rng(7)
    pats = {
        "singletons": np.arange(17),
        "one_voxel": np.zeros(33, dtype=np.int64) + 5,
        "long_runs": np.repeat(np.array([0, 3, 4, 9]), [40, 1, 300, 7]),
        "first_last_boundaries": np.array([0, 1, 1, 1, 2, 2, 7, 9, 9, 11]),
        "random_runs": np.sort(rng.integers(0, 50, size=500)),
        "empty": np.zeros(0, dtype=np.int64),
        "single_row": np.array([3]),
    }
    return {k: v.astype(np.int64) for k, v in pats.items()}


def main():
    torch.manual_seed(0)
    torch.set_num_threads(8)         # tests/_cases.py GOLDEN_THREADS: the CPU softmax's rounding depends on the thread count
    Fiery, VoxelsSumming, bev_params = import_reference()
    out_dir = os.path.join(ROOT, "tests", "golden")
    os.makedirs(out_dir, exist_ok=True)

    # ---- a6: VoxelsSumming on hand-made patterns -------------------------------------------------------
    print("VoxelsSumming patterns")
    vs = {}
    rng = np.random.default_rng(11)
    for name, ranks_np in rank_patterns().items():
        Nm, C, Y = ranks_np.size, 8, 4
        feats_np = rng.standard_normal((Nm, C), dtype=np.float32)
        coords_np = np.stack([ranks_np // Y, ranks_np % Y, np.zeros_like(ranks_np)], -1).astype(np.int64).reshape(Nm, 3)
        feats = torch.from_numpy(feats_np).requires_grad_(True)
        ranks, coords = torch.from_numpy(ranks_np), torch.from_numpy(coords_np)
        if Nm == 0:
            # reference forward on empty input: mask[:-1] assignment on a 0-length tensor is a no-op
            ref_sum, ref_coords = VoxelsSumming.apply(feats, coords, ranks)
            ref_grad = np.zeros((0, C), np.float32)
            gout_np = np.zeros((0, C), np.float32)
        else:
            ref_sum, ref_coords = VoxelsSumming.apply(feats, coords, ranks)
            gout_np = rng.standard_normal(tuple(ref_sum.shape), dtype=np.float32)
            ref_sum.backward(torch.from_numpy(gout_np))
            ref_grad = feats.grad.numpy().copy()
        f2 = torch.from_numpy(feats_np).requires_grad_(True)
        o_sum, o_coords = O.CumsumSegmentSum.apply(f2, coords, ranks)
        check(f"{name}: sums bit-equal", torch.equal(o_sum, ref_sum))
        check(f"{name}: coords equal", torch.equal(o_coords, ref_coords))
        if Nm:
            o_sum.backward(torch.from_numpy(gout_np))
            check(f"{name}: grad bit-equal", np.array_equal(f2.grad.numpy(), ref_grad))
        vs[f"{name}__feats"] = feats_np
        vs[f"{name}__coords"] = coords_np
        vs[f"{name}__ranks"] = ranks_np
        vs[f"{name}__gout"] = gout_np
        vs[f"{name}__ref_sum"] = ref_sum.detach().numpy()
        vs[f"{name}__ref_coords"] = ref_coords.numpy()
        vs[f"{name}__ref_grad"] = ref_grad
    np.savez_compressed(os.path.join(out_dir, "voxels_summing.npz"), **vs)

    # ---- a7: BEV parameters ------------------------------------------------------------------------------
    print("BEV parameters")
    params = {}
    for cname in ("cfg1_tiny", "cfg2_static_lss", "cfg4_pon", "cfg6_res_0p4_0p3"):
        cfg = CONFIGS[cname]
        r, s0, d = bev_params(list(cfg.x_bound), list(cfg.y_bound), list(cfg.z_bound))
        ro, so, do = O.bev_grid(cfg.x_bound, cfg.y_bound, cfg.z_bound)
        check(f"{cname}: bev params", torch.equal(r, ro) and torch.equal(s0, so) and torch.equal(d, do))
        params[f"{cname}__resolution"], params[f"{cname}__start"], params[f"{cname}__dimension"] = r.numpy(), s0.numpy(), d.numpy()

    # ---- full path, per config -----------------------------------------------------------------------------
    lift = dict(params)
    cases = [("cfg1_tiny", 0.02, 1), ("cfg1_tiny", 0.0, 1), ("cfg2_static_lss", 0.02, 1), ("cfg2_static_lss", 0.0, 1),
             ("cfg4_pon", 0.02, 1), ("cfg3_baseline", 0.02, 2), ("cfg6_res_0p4_0p3", 0.02, 2), ("cfg6_res_0p4_0p3", 0.0, 2)]
    # the configurations bench.py quotes, at their full batch (BASELINE.json configs[1..3]): tag carries the frame count
    bench_cases = [("cfg2_static_lss_b8", 0.02, 8), ("cfg3_baseline", 0.02, 9), ("cfg4_pon", 0.02, 12)]
    for cname, jitter, frames in cases + bench_cases:
        base = CONFIGS[cname]
        cfg = LiftConfig(**{**base.__dict__, "frames": frames})
        tag = f"{cname}__j{int(jitter * 1000):03d}"
        if (cname, jitter, frames) in bench_cases:
            tag += f"__f{frames}"
        print(f"lift {tag}")
        Knp, Enp = make_calibration(cfg, seed=3, jitter_rad=jitter)
        head_np = make_head(cfg, seed=3)
        gout_np = make_grad_bev(cfg, seed=3)
        K, E = torch.from_numpy(Knp), torch.from_numpy(Enp)
        s = reference_self(Fiery, bev_params, cfg)
        oracle = O.LiftOracle.from_config(cfg)
        check("frustum bit-equal", torch.equal(oracle.frustum, s.frustum.data))

        head = torch.from_numpy(head_np).requires_grad_(True)
        geom, bev_ref = reference_lift(Fiery, s, head, K, E, cfg)
        bev_ref.backward(torch.from_numpy(gout_np))
        grad_ref = head.grad.numpy().copy()

        head_o = torch.from_numpy(head_np).requires_grad_(True)
        geom_o = oracle.geometry(K, E)
        check("get_geometry bit-equal", torch.equal(geom_o, geom))
        comb, trans = O.compose_calibration(K, E)
        fr = s.frustum.data
        explicit = O.frustum_to_ego_explicit(fr[0, 0, :, 0].numpy(), fr[0, :, 0, 1].numpy(), fr[:, 0, 0, 2].numpy(),
                                             comb.numpy(), trans.numpy())
        n_float_mismatch = int((explicit != geom.numpy()).sum())
        print(f"      explicit no-FMA order vs torch matmul: {n_float_mismatch} / {explicit.size} floats differ")
        bev_o = oracle.lift(head_o, K, E)
        bev_o.backward(torch.from_numpy(gout_np))
        # argsort is unstable but deterministic on one build/thread count; the oracle calls the same ops, so
        # values agree to the last bit here.  Tests on other boxes use the tolerance, not bit equality.
        check("BEV oracle == reference (allclose 1e-6 normwise)", O.normwise_error(bev_o, bev_ref) < 1e-6)
        check("grad oracle == reference", O.normwise_error(head_o.grad, torch.from_numpy(grad_ref)) < 1e-6)

        idx_o, keep_o = oracle.point_indices(K, E)
        # the reference never exposes idx directly; recompute with its own expression (fiery.py:236-237)
        idx_r = ((geom - (s.bev_start_position - s.bev_resolution / 2.0)) / s.bev_resolution).view(frames, -1, 3).long()
        check("voxel idx bit-equal", torch.equal(idx_o, idx_r))
        idx_e, keep_e = O.voxel_indices_explicit(explicit, s.bev_start_position.numpy(), s.bev_resolution.numpy(),
                                                 s.bev_dimension.numpy())
        idx_e = idx_e.reshape(frames, -1, 3)
        keep_e = keep_e.reshape(frames, -1)
        n_idx_mismatch = int((idx_e != idx_o.numpy()).any(-1).sum())
        print(f"      explicit-order voxel idx vs reference: {n_idx_mismatch} / {idx_e.shape[0] * idx_e.shape[1]} points differ")
        check("explicit-order idx == reference idx", n_idx_mismatch == 0)
        check("explicit-order keep == reference keep", np.array_equal(keep_e, keep_o.numpy()))

        exact = oracle.lift_exact(torch.from_numpy(head_np), K, E)
        print(f"      reference vs fp64 truth: normwise {O.normwise_error(bev_ref, exact):.3e}  "
              f"max-abs-scaled {O.max_abs_scaled_error(bev_ref, exact):.3e}")

        X, Y = cfg.bev_hw
        occupied = (bev_ref.detach().abs().sum(1) > 0)
        lift[f"{tag}__combined"] = comb.numpy()
        lift[f"{tag}__translation"] = trans.numpy()
        lift[f"{tag}__idx_sha256"] = np.frombuffer(sha(idx_r.numpy()).encode(), dtype=np.uint8)
        lift[f"{tag}__keep_sha256"] = np.frombuffer(sha(keep_o.numpy()).encode(), dtype=np.uint8)
        lift[f"{tag}__kept_points"] = keep_o.sum(1).numpy()
        lift[f"{tag}__occupied_sha256"] = np.frombuffer(sha(occupied.numpy()).encode(), dtype=np.uint8)
        lift[f"{tag}__occupied_count"] = occupied.flatten(1).sum(1).numpy()
        lift[f"{tag}__bev_sum"] = bev_ref.detach().double().sum((1, 2, 3)).numpy()
        lift[f"{tag}__bev_norm"] = bev_ref.detach().double().flatten(1).norm(dim=1).numpy()
        lift[f"{tag}__exact_norm"] = exact.flatten(1).norm(dim=1).numpy()
        lift[f"{tag}__grad_norm"] = np.array([np.linalg.norm(grad_ref.astype(np.float64))])
        # sample indices in ascending order: they compress far better, which keeps lift.npz under 1 MB
        pick = np.sort(np.random.default_rng(5).integers(0, bev_ref.numel(), size=4096))
        lift[f"{tag}__bev_pick"] = pick
        lift[f"{tag}__bev_ref_at_pick"] = bev_ref.detach().flatten()[pick].numpy()
        gpick = np.sort(np.random.default_rng(6).integers(0, grad_ref.size, size=4096))
        lift[f"{tag}__grad_pick"] = gpick
        lift[f"{tag}__grad_ref_at_pick"] = grad_ref.reshape(-1)[gpick]
        if cname == "cfg1_tiny":                     # small enough to keep whole
            lift[f"{tag}__idx"] = idx_r.numpy().astype(np.int32)
            lift[f"{tag}__bev_ref"] = bev_ref.detach().numpy()
            lift[f"{tag}__grad_ref"] = grad_ref
            if jitter:                               # the fp64 pooling of one case pins the oracle's exact path
                lift[f"{tag}__bev_exact"] = exact.numpy()
    np.savez_compressed(os.path.join(out_dir, "lift.npz"), **lift)
    for f in sorted(os.listdir(out_dir)):
        print(f, os.path.getsize(os.path.join(out_dir, f)), "bytes")


if __name__ == "__main__":
    main()
