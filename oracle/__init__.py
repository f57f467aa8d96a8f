"""oracle/ -- TEST INFRASTRUCTURE ONLY.

A CPU restatement (numpy + a plain-C triple loop) of the PCMF CAVI iteration of the
reference (AntoinePassemiers/Oriana, `oriana/models/zigap.py:79-158`, `gap.py:67-129`,
`nodes/probabilistic/gamma.py:37-61`, `bernoulli.py:41-48`, `utils.py:9-51`).

Only `tests/`, `__graft_entry__.smoke()` and the `cpu_baseline` / `--impl reference`
legs of `bench.py` may import or execute anything under this directory, and there only
as the checker (or the timed CPU baseline) -- never as the product path.  The product
(`oriana_b200/`) never imports it and raises when its CUDA library is missing.

Pinning status
--------------
* CAVI step (Z-kernel, Gamma/Bernoulli updates, M-step): PINNED against the unmodified
  reference (`oracle/make_golden.py` imports a checkout of it, `oracle/refshim.py`
  CHECKOUT, under the `np.float/np.int` alias shim, copies the state out of a
  constructed reference model, steps it and stores the trajectories under
  `tests/golden/`).  `tests/test_oracle.py` replays those fixtures through this port.
* Special functions (sigmoid/logit/digamma/inverse digamma, Gamma mean/meanlog,
  Bernoulli mean): pinned by the reference's own known-answer tests
  (`test/test.py:13-41,60-79`), restated in `tests/test_oracle.py::test_special_functions_against_reference_kats` and `tests/test_special_gpu.py`.
* ELBO: the reference has NO ELBO function.  The float64 formula in `cavi_numpy.elbo`
  is derived from the model definition (`zigap.py:21-53`); for it: PARITY UNPINNED
  (the float64 oracle is the only pin; it is checked for monotonicity on the de-quirked
  update in `tests/test_oracle.py`).
* Third-party arithmetic on the path: `scipy.special.digamma` / `polygamma(1, .)`
  (reference pins scipy==1.1.0, `requirements.txt:2`; here scipy 1.18.1) and
  `sklearn.decomposition.NMF` (init only; side-stepped by copying state).
"""
