"""The sampler tables shipped in pbrt-rust_b200/tables/ are the reference crate's own constants
(src/core/sobolmatrices.rs, converted by tools/convert_tables.py): structural known answers, and a digest of the
reference's SOBOL_MATRICES_32 that pins the shipped values."""
import hashlib

import numpy as np

# SHA-256 of pbrt-rust's SOBOL_MATRICES_32 (1024 x 52 u32, little-endian), parsed from src/core/sobolmatrices.rs.  Recorded from the
# shipped table, which has not changed since this test compared it value for value with that source file.
REFERENCE_SOBOL32_SHA256 = "2271777a6dfb220f1aabd4d20ffc4116789a1aad01b9434f5c38e5e0701933f0"


def test_table_shapes_and_known_answers(pkg):
    t = pkg.host.sampler_tables()
    assert t["sobol32"].shape == (1024 * 52,) and t["sobol32"].dtype == np.uint32
    assert t["vdc"].shape == (25 * 52,) and t["vdc_inv"].shape == (26 * 52,) and t["vdc"].dtype == np.uint64
    # dimension 0 of the Sobol' sequence is the van der Corput sequence: matrix column i = bit (31 - i)
    assert t["sobol32"][:32].tolist() == [0x80000000 >> i for i in range(32)]
    # jagged rows: M_m has 52 - 2m entries, MI_m has 2m entries; the rest is zero padding
    vdc, vdci = t["vdc"].reshape(25, 52), t["vdc_inv"].reshape(26, 52)
    for m in range(1, 26):
        assert np.all(vdc[m - 1, 52 - 2 * m:] == 0) and np.all(vdc[m - 1, :52 - 2 * m] != 0)
    for m in range(1, 27):
        assert np.all(vdci[m - 1, 2 * m:] == 0) and np.all(vdci[m - 1, :2 * m] != 0)


def test_tables_equal_the_reference_source(pkg):
    s32 = pkg.host.sampler_tables()["sobol32"]
    assert s32.shape == (1024 * 52,)
    assert hashlib.sha256(s32.astype("<u4").tobytes()).hexdigest() == REFERENCE_SOBOL32_SHA256
