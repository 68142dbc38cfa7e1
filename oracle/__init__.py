"""CPU oracle of the Asyrp hot path (UNet forward + DDIM reverse loop).

TEST INFRASTRUCTURE.  A plain-PyTorch fp32 restatement of the reference's algorithm, each function citing the
reference file:line it follows.  Only tests/, __graft_entry__.smoke() and bench.py (cpu_baseline /
--impl reference) may import it; the product package asyrp_official_b200 never does.

Parity pinning: tests/golden/make_golden.py imports the reference's own modules from the reference checkout
(stage_reference.reference_dir()), loads the same synthetic state dicts (oracle/synth.py) and writes golden outputs
to tests/golden/; tests/test_oracle.py checks this restatement against them (bit-level on CPU fp32).
"""
from . import adm, ddpm, sampler, synth  # noqa: F401
