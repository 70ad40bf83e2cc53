"""Known-answer vectors of TensorFlow r1.9's own unit test for `GRUCell`.

Provenance: tensorflow/python/kernel_tests/rnn_cell_test.py (class RNNCellTest, `testGRUCell`) at branch r1.9 -- the
core RNN cell test, since `tf.contrib.rnn.GRUCell` is `rnn_cell_impl.GRUCell`.  The kernels are built under a
constant 0.5 initialiser; the biases keep GRUCell's own defaults (gates/bias 1.0, candidate/bias 0.0); 2 units,
state h = [[0.1, 0.1]].  TensorFlow is not vendored in the reference and cannot run here, so inputs AND expected
outputs below were restated from the public test source rather than copied from a file on this machine; the GRU
equations of tests/gru_oracle.py -- written from GRUCell's semantics, not from these numbers -- reproduce both to 6
digits (tests/test_gru_host.py).
"""
import numpy as np

UNITS = 2
KERNEL_INIT = 0.5
GATES_BIAS, CANDIDATE_BIAS = 1.0, 0.0
H = np.array([[0.1, 0.1]], np.float32)

CASES = [
    # (x, expected new h)
    (np.array([[1.0, 1.0]], np.float32), np.array([[0.175991, 0.175991]], np.float32)),
    (np.array([[1.0, 1.0, 1.0]], np.float32), np.array([[0.156736, 0.156736]], np.float32)),
]
