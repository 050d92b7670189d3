"""plonk-prototype_b200 — B200-native MSM / NTT backend behind the dusk-plonk / dusk-bls12_381 API
surface that Manta-Network/Plonk-Prototype's circuits prove through.  See DESIGN.md."""
from ._native import Context, Pb200Error, LIB_PATH, EXPORTS, verify, verify_batch, opening_key_from_tau  # noqa: F401
from .domain import EvaluationDomain, Polynomial, Evaluations, InvalidEvalDomainSize, default_context  # noqa: F401
from .msm import msm_variable_base, pippenger, CommitKey, g1_to_bytes  # noqa: F401
from .dist_ntt import DistributedDomain, ShardSpec, GpuBackend, PeerBuffers  # noqa: F401
from .prover import StandardComposer, Prover, PublicParameters, ShardedParameters, torch_allgather, torch_device_collectives, scalars_to_mont  # noqa: F401
from . import gadgets, jubjub, poseidon, serial  # noqa: F401
