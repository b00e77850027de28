"""TEST INFRASTRUCTURE ONLY.

CPU restatement of the DiffSinger reverse-diffusion hot path (DiffNet + DDPM / PLMS
samplers).  Nothing under ``oracle/`` is part of the shipped product: only ``tests/``,
``__graft_entry__.smoke()`` and the ``cpu_baseline`` / ``--impl reference`` legs of
``bench.py`` may import it, and only as the checker / the timed CPU baseline.

Parity pinning: the reference has no tests or golden vectors for this path
(SURVEY.md §4), so the oracle is pinned against the live reference PyTorch modules
imported from /root/reference in the build container (``oracle/ref_bridge.py`` +
``oracle/gen_golden.py``); the vectors it produced are committed in ``tests/golden``.
"""

# ATen's CPU convolutions split their float32 sums by the number of intra-op threads: the golden vectors are recorded, and
# must be compared bit for bit, at this count
FIXTURE_THREADS = 8
