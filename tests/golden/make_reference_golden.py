"""Regenerate tests/golden/reference.json: what the reference's own parser and colour kernels (oracle/_ref) give on the
inputs of the tests that compare the oracle with them, so that those tests keep their comparison where oracle/_ref cannot
be built (it needs the reference's sources).

  python tests/golden/make_reference_golden.py

Each value is what the comparing test asserts the reference gives: the oracle's parse fields, its verdicts under the
rules of the tests (a stream accepted here only as a widened stream is one the reference rejects) and the SHA-256 of its
outputs. Where oracle/_ref is present every value is checked against the reference itself before it is written, and
"checked_against_reference" is true. The committed file was written without oracle/_ref, from oracle/ and tests/ as of
commit cc8507e, where every one of these comparisons ran live against oracle/_ref and passed (the CPU suite ran without
a skip); neither oracle/ nor these tests' inputs have changed since.

  parser        per golden case: test_oracle_parser_matches_reference_parser
  accept_reject per mutation: test_oracle_parser_accept_reject_matches_reference
  kernels       per picture, format and crop: test_oracle_output_matches_reference_kernels
  kernels_411   per picture and format: test_oracle_411_pinned
  widened       per stream, the reference's accept (0 for all): test_oracle_widened_streams_pinned
  header_fuzz   per mutation, "1" / "0" / "-" (verdict undefined): test_parser_header_fuzz_matches_oracle_and_reference
"""
import json
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

import oracle  # noqa: E402
from rocjpeg_b200 import api, datagen  # noqa: E402
import test_host_library as thl  # noqa: E402
import test_oracle_pinning as top  # noqa: E402


def main():
    orc = oracle.Oracle()
    have_ref = oracle.ref_available()
    rp = oracle.RefParser() if have_ref else None
    rk = oracle.RefKernels() if have_ref else None
    if have_ref:
        from ref_assembly import reference_output
    out = {"parser": {}, "accept_reject": {}, "kernels": {}, "kernels_411": {}, "widened": {}, "header_fuzz": ""}

    for name in top.CASES:
        data = top.load(name)
        rc, o = orc.parse(data)
        assert rc == 0, name
        out["parser"][name] = top.parser_fields(o, o.num_mcus_ref, o)
        if rp is not None:
            r = rp.parse(data)
            assert r.ok == 1 and top.parser_fields(r, r.num_mcus, o) == out["parser"][name], name

    for name, data in top._mutations(top.load("synth_420_123x77")).items():
        rc, o = orc.parse(data)
        ok = int(rc == 0 and not o.features)
        out["accept_reject"][name] = {"ok": ok, "dims": [o.width, o.height, o.css] if ok else None}
        if rp is not None:
            assert top.ref_verdict(rp.parse(data)) == out["accept_reject"][name], name

    for css in [c for c in datagen.CSS_NAMES if c != "411"]:
        for key, data, fmt, crop in top.kernel_cases(css):
            rc, info = orc.parse(data)
            _, dst = orc.decode(data, fmt, crop)
            valid = [d[:rows, :rb] for d, (rows, rb) in zip(dst, oracle.output_shapes(info, fmt, crop, orc))]
            out["kernels"][key] = top.sha(valid)
            if rk is not None:
                ref = reference_output(rk, info, orc.planes(data, info), fmt, crop)
                assert all(np.array_equal(d, r) for d, r in zip(valid, ref)), key

    for (w, h, rows) in ((200, 120, 0), (131, 67, 1), (33, 9, 0)):
        data = datagen.make_jpeg(w, h, "411", seed=70 + w, restart_rows=rows)
        rc, info = orc.parse(data)
        planes = orc.planes(data, info)
        for fmt in ("rgb", "rgb_planar"):
            _, dst = orc.decode(data, fmt)
            valid = [d[:r_, :rb] for d, (r_, rb) in zip(dst, oracle.output_shapes(info, fmt))]
            out["kernels_411"][f"{w}x{h}|{fmt}"] = top.sha(valid)
            if rk is not None:
                rc, info444 = orc.parse(datagen.make_jpeg(w, h, "444", seed=1))
                ph, pw = info444.blocks_h[0] * 8, info444.blocks_w[0] * 8
                fake = [np.ascontiguousarray(planes[0][:ph, :pw])] + [
                    np.ascontiguousarray(np.repeat(planes[c], 4, axis=1)[:ph, :pw]) for c in (1, 2)]
                ref = reference_output(rk, info444, fake, fmt, (0, 0, 0, 0))
                assert all(np.array_equal(d, r) for d, r in zip(valid, ref)), (w, h, fmt)

    for name, data in top.widened_streams(orc).items():
        out["widened"][name] = 0
        if rp is not None:
            assert not rp.parse(data).ok, name

    s = api.JpegStream()
    verdicts = []
    for name, kind, hdr_end, data in thl.header_fuzz():
        st = s.parse(data)
        widened = thl.fuzz_widened(s, st)
        v = "-" if widened is None else "0" if widened or st != api.SUCCESS else "1"
        if rp is not None and v != "-":
            assert str(int(rp.parse(data).ok)) == v, (name, kind)
        verdicts.append(v)
    out["header_fuzz"] = "".join(verdicts)

    out["meta"] = {"checked_against_reference": have_ref}
    with open(os.path.join(HERE, "reference.json"), "w") as f:
        json.dump(out, f, indent=1, sort_keys=True)
    print("wrote reference.json; checked against the reference:", have_ref)


if __name__ == "__main__":
    main()
