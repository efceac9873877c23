"""Precision knob (the only setting the reference does not have).

precision = "auto": float32 inputs run the fp32 path (bf16x2-split tensor-core contractions, fp32
sweeps, fp64 scalar reductions); anything else runs the fp64 path, which reproduces the reference's
float64 results to ~1e-10.  "fp32" / "fp64" force a mode regardless of the input dtype.

precision = "fp32x3" (opt-in): results are float32 whatever the input dtype.  NMF with "hals", or "mu" with beta = 1 or 2,
at rank <= 64 on one GPU keeps X and both factors as THREE bf16 planes (hi + mid + lo: the fp32 values exactly) and forms
every tensor-core product from the six terms down to order 2^-16 with fp32 accumulation -- 24-bit operands instead of the
17 bits of "fp32", at 6 instead of 4 bytes per element and orientation of X.  Everything else (other ranks, one_nmf_step,
NTF, NTD, PARAFAC2, the update rules called directly) computes in float64 and returns float32; the sharded entry point
refuses it.  It costs time: measured at 65536 x 8192, rank 64, on one B200, MU runs at 0.6-0.7x the "fp32" rate and HALS at
about 1/6 of it (its solves run on the fp32 CUDA-core sweep, see DESIGN.md section 1).
"""
precision = "auto"

# "auto" only: float32 problems of at most this many data elements run their arithmetic in float64 (inputs promoted on
# upload, results returned as float32).  Such problems are bound by launch latency on a B200, not by bandwidth or FLOPs, so
# the reference's own float64 arithmetic costs nothing there -- and near-exact small data (BASELINE configs[0]: 1000 x 500,
# relative residual 2e-3) needs it: bf16 hi/lo planes carry 17 bits, and after 100 iterations the fp32 trajectory is 5e-4
# away from the float64 one.  Larger problems use the tensor-core path (see DESIGN.md, "precision").
small_problem_elements = 1 << 22


def set_precision(mode):
    global precision
    if mode not in ("auto", "fp32", "fp64", "fp32x3"):
        raise ValueError(f"precision must be 'auto', 'fp32', 'fp64' or 'fp32x3', got {mode!r}")
    precision = mode
