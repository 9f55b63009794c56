"""CPU oracles for the mfrec SGD hot path -- TEST INFRASTRUCTURE ONLY.

Only ``tests/``, ``__graft_entry__.smoke()`` and ``bench.py``'s ``cpu_baseline`` /
``--impl reference`` legs may import this package; the product (``mfrec_b200``) never
does and fails loudly when its CUDA library is missing.

``oracle.cpu``  our plain-C restatement (``mfrec_oracle.c``), ctypes-bound.
``oracle.ref``  the reference's own Cython kernels built unmodified into ``oracle/_ref``.
``oracle.als_systems``  the normal equations of one ALS-WRMF half-pass in float64 NumPy, and a
                checker of a device's solutions against them.
"""
