import numpy as np

from carma_pack_b200 import io as cio


def test_clean_and_pack(tmp_path):
    t = np.array([3.0, 1.0, 2.0, 2.0, np.nan, 5.0])
    y = np.array([30.0, 10.0, 20.0, 21.0, 0.0, np.inf])
    e = np.ones(6)
    tc, yc, ec = cio.clean_light_curve(t, y, e)
    assert list(tc) == [1.0, 2.0, 3.0] and list(yc) == [10.0, 20.0, 30.0]  # first of the duplicated time kept
    p = tmp_path / "lc.dat"
    np.savetxt(p, np.column_stack([t[:4], y[:4], e[:4]]), fmt="%10.5f")
    tr, yr, er = cio.read_ascii(str(p))
    assert list(tr) == [1.0, 2.0, 3.0]
    tt, yy, ee, off, kept = cio.pack_ragged([(t, y, e), (np.array([1.0]), np.array([1.0]), np.array([1.0])),
                                             (np.arange(4.0), np.arange(4.0), np.ones(4))])
    assert list(off) == [0, 3, 7] and list(kept) == [0, 2] and tt.size == 7
    assert np.all(np.diff(tt[:3]) > 0) and np.all(np.diff(tt[3:]) > 0)


def _card(key, value, comment=""):
    if isinstance(value, bool):
        v = "%20s" % ("T" if value else "F")
    elif isinstance(value, str):
        v = "%-20s" % ("'%-8s'" % value)
    else:
        v = "%20s" % value
    return ("%-8s= %s / %s" % (key, v, comment))[:80].ljust(80)


def _write_fits_bintable(path, cols):
    """Minimal FITS file: empty primary HDU + one BINTABLE extension (what Kepler light-curve files look like)."""
    codes = {"f8": "D", "f4": "E", "i4": "J", "i2": "I"}
    dt = np.dtype([(n, ">" + a.dtype.str[1:]) for n, a in cols])
    nrow = len(cols[0][1])
    tab = np.zeros(nrow, dtype=dt)
    for n, a in cols:
        tab[n] = a
    primary = "".join([_card("SIMPLE", True), _card("BITPIX", 8), _card("NAXIS", 0), _card("EXTEND", True), "END".ljust(80)])
    ext = [_card("XTENSION", "BINTABLE"), _card("BITPIX", 8), _card("NAXIS", 2), _card("NAXIS1", dt.itemsize),
           _card("NAXIS2", nrow), _card("PCOUNT", 0), _card("GCOUNT", 1), _card("TFIELDS", len(cols))]
    for k, (n, a) in enumerate(cols, 1):
        ext += [_card("TTYPE%d" % k, n, "column title"), _card("TFORM%d" % k, codes[a.dtype.str[1:]])]
    ext.append("END".ljust(80))
    with open(path, "wb") as f:
        for hdr in (primary, "".join(ext)):
            b = hdr.encode("ascii")
            f.write(b + b" " * (-len(b) % 2880))
        raw = tab.tobytes()
        f.write(raw + b"\0" * (-len(raw) % 2880))


def test_fits_binary_table_light_curve(tmp_path):
    """FITS ingestion (the Kepler file of src/paper/data is read this way at carma_paper.py:522-531): a binary-table
    extension with TIME (D), CADENCENO (J), SAP_FLUX / SAP_FLUX_ERR (E) columns, NaN gaps included."""
    rng = np.random.default_rng(0)
    n = 500
    time = 2455462.5 + np.cumsum(rng.uniform(0.01, 0.03, n))
    flux = (1000.0 + rng.standard_normal(n)).astype(np.float32)
    ferr = np.full(n, 0.5, dtype=np.float32)
    time[17] = np.nan
    flux[40:43] = np.nan
    p = str(tmp_path / "lc.fits")
    _write_fits_bintable(p, [("TIME", time), ("CADENCENO", np.arange(n, dtype=np.int32)), ("SAP_FLUX", flux), ("SAP_FLUX_ERR", ferr)])
    cols = cio.read_fits_table(p)
    assert set(cols) == {"TIME", "CADENCENO", "SAP_FLUX", "SAP_FLUX_ERR"} and cols["CADENCENO"][7] == 7
    assert np.array_equal(cols["TIME"], time, equal_nan=True) and cols["SAP_FLUX"].dtype == np.float32
    t, y, e = cio.read_fits(p)
    assert t.size == n - 4 and t[0] == 0.0 and np.all(np.diff(t) > 0) and np.all(np.isfinite(y))
    good = np.isfinite(time) & np.isfinite(flux)
    assert np.allclose(y, flux[good].astype(float)) and np.allclose(t, time[good] - time[good].min())
    # and it packs into the ragged batch layout next to an ASCII curve
    tt, yy, ee, off, kept = cio.pack_ragged([(t, y, e), (np.arange(5.0), np.arange(5.0), np.ones(5))])
    assert list(off) == [0, n - 4, n + 1]
