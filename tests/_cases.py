"""Shared helpers for the parity tests: the cases oracle/gen_golden.py recorded, rebuilt from the same seeds."""
import hashlib

import numpy as np
import torch

from fiery_b200.synthetic import CONFIGS, LiftConfig, make_calibration, make_grad_bev, make_head

# (config name, calibration jitter in rad, frames) -- must match oracle/gen_golden.py:main
GOLDEN_CASES = [("cfg1_tiny", 0.02, 1), ("cfg1_tiny", 0.0, 1), ("cfg2_static_lss", 0.02, 1), ("cfg2_static_lss", 0.0, 1),
                ("cfg4_pon", 0.02, 1), ("cfg3_baseline", 0.02, 2), ("cfg6_res_0p4_0p3", 0.02, 2), ("cfg6_res_0p4_0p3", 0.0, 2)]


# torch intra-op threads the golden vectors were recorded with -- must match oracle/gen_golden.py:main.  The CPU softmax splits
# its work by thread count, and a split that does not fall on the vector width rounds some elements differently (e.g. 6 or 16
# threads on the tiny config); the reference's cumsum pooling then amplifies that past the tight golden comparisons.
GOLDEN_THREADS = 8


# the configurations bench.py quotes, at their full batch; golden tags carry the frame count
BENCH_CASES = [("cfg2_static_lss_b8", 0.02, 8), ("cfg3_baseline", 0.02, 9), ("cfg4_pon", 0.02, 12)]


def case_id(case):
    return f"{case[0]}-j{int(case[1] * 1000):03d}-f{case[2]}"


def golden_tag(case):
    tag = f"{case[0]}__j{int(case[1] * 1000):03d}"
    return tag + f"__f{case[2]}" if tuple(case) in BENCH_CASES else tag


def build_case(case, seed=3):
    name, jitter, frames = case
    cfg = LiftConfig(**{**CONFIGS[name].__dict__, "frames": frames})
    K, E = make_calibration(cfg, seed=seed, jitter_rad=jitter)
    return cfg, torch.from_numpy(K), torch.from_numpy(E), torch.from_numpy(make_head(cfg, seed=seed)), \
        torch.from_numpy(make_grad_bev(cfg, seed=seed))


def sha(a) -> str:
    return hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()


def golden_str(arr) -> str:
    return bytes(arr.tolist()).decode()
