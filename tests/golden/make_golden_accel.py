"""Records the flows that tests/test_accel.py hands to ``zuko_b200.accelerate``, built by the constructors
of the UNMODIFIED reference, as module trees (tests/module_tree.py): class names, constructor attributes,
parameters and buffers.  The test rebuilds them from tests/golden/accel_reference_flows.npz, so it runs
on the reference's own module layout where the reference is not installed.

    PYTHONDONTWRITEBYTECODE=1 python tests/golden/make_golden_accel.py <directory containing the reference's zuko/>
"""

from __future__ import annotations

import sys
from functools import partial
from pathlib import Path

import numpy as np
import torch

sys.dont_write_bytecode = True
HERE = Path(__file__).resolve().parent
sys.path.insert(0, str(HERE.parent))

from module_tree import record  # noqa: E402


def reference_flows(zuko) -> dict:  # noqa: ANN001
    torch.manual_seed(0)
    F, T, D = zuko.flows, zuko.transforms, zuko.distributions
    base = lambda n: F.UnconditionalDistribution(D.DiagNormal, torch.zeros(n), torch.ones(n), buffer=True)  # noqa: E731
    adjacency = torch.tensor([[1, 0, 0], [1, 1, 0], [0, 1, 1]], dtype=bool)
    return {
        "nsf": F.NSF(5, 3, transforms=2, bins=4, hidden_features=[32, 32]),
        "maf": F.MAF(4, 0, transforms=2, hidden_features=[16]),
        "maf_randperm": F.MAF(6, 2, transforms=3, randperm=True),
        "nice": F.NICE(5, 2, transforms=3),
        "nsf_passes2": F.NSF(6, 0, transforms=2, passes=2),
        "nsf_single_feature": F.NSF(1, 2, transforms=2),
        "ncsf": F.NCSF(3, 2, transforms=2, bins=4, hidden_features=[16]),
        "maf_elu": F.MAF(4, 2, transforms=2, hidden_features=[32, 32], activation=torch.nn.ELU),
        "nsf_residual": F.NSF(4, 2, transforms=2, hidden_features=[16, 32, 32], residual=True),
        "adjacency": F.Flow([F.MaskedAutoregressiveTransform(3, 1, adjacency=adjacency)], base(3)),
        "composed": F.Flow(
            [
                F.UnconditionalTransform(T.SoftclipTransform, bound=6.0),
                F.MaskedAutoregressiveTransform(4, 2, univariate=partial(T.MonotonicRQSTransform, slope=1e-2), shapes=[(8,), (8,), (7,)]),
                F.UnconditionalTransform(T.PermutationTransform, torch.randperm(4), buffer=True),
                F.UnconditionalTransform(T.RotationTransform, torch.randn(4, 4)),
                F.GeneralCouplingTransform(4, 2).inv,
            ],
            base(4),
        ),
        # what the engine does not implement: accelerate() must refuse these
        "maf_prelu": F.MAF(3, 0, activation=torch.nn.PReLU),
        "naf": F.NAF(3, 0),
        "gf": F.GF(3, 0),
        "maf_float64": F.MAF(3, 0).double(),
    }  # fmt: skip


def main() -> None:
    sys.path.insert(0, str(Path(sys.argv[1]).resolve()))
    import zuko

    np.savez_compressed(HERE / "accel_reference_flows.npz", **record(reference_flows(zuko)))


if __name__ == "__main__":
    main()
