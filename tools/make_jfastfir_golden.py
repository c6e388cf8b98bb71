"""Write tests/golden/jfastfir_golden.npz from the reference's own JFastFir test vectors (JAERO/tests/jfastfir_data_*.cpp,
compiled into oracle/_ref by oracle/Makefile). The data files print 6 significant digits, which float32 holds exactly:
the test restores each value with "%.6g". The input is kept whole (the filter needs every sample), the expected output
every STEP-th sample. Needs oracle/_ref."""
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from oracle import ref  # noqa: E402

STEP = 5

if __name__ == "__main__":
    L = ref.lib()
    n = L.jref_golden_jfastfir_len()
    gi = np.zeros((n, 2)); go = np.zeros((n, 2))
    L.jref_golden_jfastfir(gi.ctypes.data, go.ctypes.data)
    six = lambda a: np.array([float("%.6g" % v) for v in a.ravel()]).reshape(a.shape)
    i32, o32 = gi.astype(np.float32), go[::STEP].astype(np.float32)
    assert np.array_equal(six(i32), gi) and np.array_equal(six(o32), go[::STEP])
    np.savez_compressed(os.path.join(ROOT, "tests", "golden", "jfastfir_golden.npz"), input=i32, expected_output=o32, step=STEP,
                        Fs=L.jref_golden_jfastfir_Fs(), fb=L.jref_golden_jfastfir_fb())
