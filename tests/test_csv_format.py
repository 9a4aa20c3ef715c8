"""CPU: the CSV formatting code of dc_table_csv (csrc/csv.cu), through its host-compiled test entry points -- every value
as Python's repr / pandas' to_csv writes it, whole tables as the per-image DataFrame + insert + to_csv, and the
all_droplets.csv assembly as pd.concat(...).to_csv."""
import ctypes as C
import sys
from pathlib import Path

import numpy as np
import pandas as pd
import pytest

REPO = Path(__file__).resolve().parent.parent


def fmt(values) -> list[str]:
    from unet_dc_segmentation_b200 import _lib
    v = np.ascontiguousarray(values)
    is_double = v.dtype == np.float64
    assert is_double or v.dtype == np.int64
    out = np.empty(24 * v.size + 1, dtype=np.uint8)
    off = np.empty(v.size + 1, dtype=np.int64)
    _lib.check(_lib.load().dc_debug_format_values(v.ctypes.data, int(is_double), v.size, out.ctypes.data, out.size,
                                                  off.ctypes.data))
    text = out[:off[-1]].tobytes().decode("ascii")
    return [text[off[i]:off[i + 1]] for i in range(v.size)]


def check_repr(values):
    v = np.asarray(values, dtype=np.float64)
    v = v[~np.isnan(v)]
    got = fmt(v)
    want = [repr(x) for x in v.tolist()]
    bad = [(w, g) for w, g in zip(want, got) if w != g]
    assert not bad, f"{len(bad)} of {v.size} differ, e.g. (repr, ours) {bad[:5]}"


def neighbours(x, k=1):
    x = np.asarray(x, dtype=np.float64)
    out = [x]
    lo, hi = x.copy(), x.copy()
    for _ in range(k):
        lo, hi = np.nextafter(lo, -np.inf), np.nextafter(hi, np.inf)
        out += [lo, hi]
    return np.concatenate(out)


def test_random_bit_patterns():
    rs = np.random.default_rng(0)
    for _ in range(10):                                     # 10^7 doubles, every exponent equally likely
        check_repr(rs.integers(0, 2**64, 1_000_000, dtype=np.uint64, endpoint=False).view(np.float64))


def test_random_values_equal_pandas_to_csv():
    rs = np.random.default_rng(1)
    v = np.concatenate([rs.integers(0, 2**64, 200_000, dtype=np.uint64).view(np.float64),
                        rs.random(200_000) * 10.0 ** rs.integers(-8, 20, 200_000), [np.inf, -np.inf, -0.0, 0.0]])
    v = v[~np.isnan(v)]
    want = pd.DataFrame({"x": v}).to_csv(index=False, header=False).split("\n")[:-1]
    assert fmt(v) == want


def test_powers_of_ten_and_neighbours():
    p = np.array([float(f"1e{k}") for k in range(-324, 309)])
    check_repr(neighbours(p[p > 0], 3))
    check_repr(-neighbours(p[p > 0], 1))


def test_powers_of_two_and_subnormals():
    check_repr(neighbours(np.ldexp(1.0, np.arange(-1074, 1024)), 2))
    check_repr(np.arange(0, 100_000, dtype=np.uint64).view(np.float64))                  # smallest subnormals
    sub = np.random.default_rng(2).integers(0, 2**52, 200_000, dtype=np.uint64)
    check_repr(sub.view(np.float64))
    check_repr(neighbours(np.array([np.finfo(np.float64).tiny, np.finfo(np.float64).max, 5e-324]), 2))


def test_two_to_the_53_region():
    base = np.float64(2.0 ** 53)
    check_repr(base + np.arange(-5000, 5000, dtype=np.float64))
    check_repr(neighbours(np.array([2.0 ** 53, 2.0 ** 54, 2.0 ** 52, 9007199254740993.0]), 50))


def test_layout_switches():
    """Positional from 1e-4 up to (not including) 1e16, exponent form outside, on both sides of each switch."""
    check_repr(neighbours(np.array([1e-4, 1e16, 9999999999999998.0, 1e-5, 1e15, 0.0001, 1e17]), 200))
    assert fmt(np.array([12.0, 9999999999999998.0, 1e-4, -0.0, 1e-5, 1e16, 1.2345678901234568e17, 5e-324, np.inf,
                         -np.inf, 0.0, 1.5, 123456789.125])) == \
        ["12.0", "9999999999999998.0", "0.0001", "-0.0", "1e-05", "1e+16", "1.2345678901234568e+17", "5e-324", "inf",
         "-inf", "0.0", "1.5", "123456789.125"]
    assert fmt(np.array([np.nan])) == [""]                  # pandas' na_rep


def test_table_value_families():
    """What dc_label_stats writes: centroids k/n, diameters sqrt(4a/pi), micron columns a/3.45^2 and a/px^2 for many
    px -- down to px whose square underflows, so that the area in square microns overflows to inf."""
    rs = np.random.default_rng(3)
    n = rs.integers(1, 20_000, 300_000)
    k = rs.integers(0, 4096, 300_000) * n + rs.integers(0, n)
    check_repr(k / n)
    a = np.arange(1, 1_000_001, dtype=np.float64)
    check_repr(np.sqrt(4.0 * a / np.pi))
    check_repr(a / (3.45 ** 2))
    check_repr(np.sqrt(4.0 * a / np.pi) / 3.45)
    px = np.concatenate([10.0 ** rs.uniform(-200, 200, 2000), [1e-160, 1e-170, 3.45, 0.1, 7.0]])
    aa = rs.integers(1, 100_000, px.size).astype(np.float64)
    with np.errstate(over="ignore"):
        check_repr(aa / (px * px))
        check_repr(np.sqrt(4.0 * aa / np.pi) / px)
    assert fmt(aa[:1] / (1e-160 * 1e-160)) == ["inf"]


def test_int64():
    i64 = np.iinfo(np.int64)
    p = 10 ** np.arange(19, dtype=object)
    vals = [0, 1, -1, i64.max, i64.min, i64.max - 1, i64.min + 1] + [int(x) + d for x in p for d in (-1, 0, 1)]
    vals += [-v for v in vals if v > i64.min]
    vals += np.random.default_rng(4).integers(i64.min, i64.max, 100_000).tolist()
    v = np.array([x for x in vals if i64.min <= x <= i64.max], dtype=np.int64)
    assert fmt(v) == [str(x) for x in v.tolist()]


# ------------------------------------------------------------------ whole tables
def host_table_csv(tables, names, capacity, micron):
    """dc_debug_table_csv_host on a host table; returns (per-frame text bytes, area sums)."""
    from unet_dc_segmentation_b200 import _lib
    from unet_dc_segmentation_b200.quantify import csv_field, pack_fields, table_csv_bounds
    B = len(tables)
    counts = np.array([t["n"] for t in tables], dtype=np.int32)
    cols = {}
    for c, dt in (("area", np.int64), ("equivalent_diameter", np.float64), ("centroid-0", np.float64),
                  ("centroid-1", np.float64), ("area_sqmicron", np.float64), ("eq_diam_micron", np.float64)):
        a = np.zeros((B, capacity), dtype=dt)
        for b, t in enumerate(tables):
            a[b, :min(t["n"], capacity)] = t[c][:capacity]
        cols[c] = a
    buf, offs = pack_fields([csv_field(n) for n in names])
    nbytes, _ = table_csv_bounds(B, capacity, micron, int(offs[-1]))
    out = np.zeros(nbytes, dtype=np.uint8)
    foff = np.zeros(B + 1, dtype=np.int64)
    asum = np.zeros(B, dtype=np.int64)
    p = lambda a: a.ctypes.data                      # noqa: E731
    args = _lib.TableCsvArgs(B, capacity, p(counts), p(cols["area"]), p(cols["equivalent_diameter"]),
                             p(cols["centroid-0"]), p(cols["centroid-1"]),
                             p(cols["area_sqmicron"]) if micron else None, p(cols["eq_diam_micron"]) if micron else None,
                             p(buf), p(offs), int(offs[-1]), p(out), out.size, p(foff), p(asum), None, 0)
    _lib.check(_lib.load().dc_debug_table_csv_host(C.byref(args)))
    return [out[foff[b]:foff[b + 1]].tobytes() for b in range(B)], asum


def pandas_csv(t, name, micron):
    """The parent's per-image path: the column-contract DataFrame (empty and column-less without droplets), the filename
    inserted in front, to_csv -- encoded as Path.write_text writes it."""
    from unet_dc_segmentation_b200.quantify import COLUMNS, MICRON_COLUMNS, text_encoding
    n = t["n"]
    if n == 0:
        df = pd.DataFrame()
    else:
        cols = {"label": np.arange(1, n + 1, dtype=np.int64), **{k: t[k][:n] for k in COLUMNS[1:] + MICRON_COLUMNS}}
        df = pd.DataFrame({k: cols[k] for k in COLUMNS + (MICRON_COLUMNS if micron else [])})
    df.insert(0, "filename", name)
    return df, df.to_csv(index=False).encode(text_encoding())


def random_table(rs, n, px):
    a = rs.integers(1, 5000, n).astype(np.int64)
    area = a.astype(np.float64)
    with np.errstate(over="ignore"):
        return {"n": n, "area": a, "equivalent_diameter": np.sqrt(4.0 * area / np.pi),
                "centroid-0": rs.integers(0, 2048 * 64, n) / a, "centroid-1": rs.random(n) * 2048,
                "area_sqmicron": area / (px * px), "eq_diam_micron": np.sqrt(4.0 * area / np.pi) / px}


NAMES = ["f0.png", "a,b.png", 'q"u.png', "é ü 漢.tif", "new\nline.png", "plain name.jpeg", "c,\"d\",e.png", "x.png"]


@pytest.mark.parametrize("micron", [False, True])
def test_host_tables_equal_pandas(micron):
    rs = np.random.default_rng(5 + micron)
    px = 3.45 if micron else 1.0
    ns = [0, 1, 37, 0, 500, 3, 2, 64]
    tables = [random_table(rs, n, px) for n in ns]
    tables[2]["centroid-1"][:5] = [0.0, 1e-5, 1e16, 123456789012345678.0, 0.1]
    if micron:
        tables[4]["area_sqmicron"][:3] = np.inf                        # an extreme px_per_micron
    texts, asum = host_table_csv(tables, NAMES, 512, micron)
    for b, (t, name) in enumerate(zip(tables, NAMES)):
        _, want = pandas_csv(t, name, micron)
        assert texts[b] == want, (b, texts[b][:200], want[:200])
        assert asum[b] == (t["area"].sum() if t["n"] else 0)


def test_host_table_capacity_overflow_yields_no_text():
    rs = np.random.default_rng(7)
    tables = [random_table(rs, n, 1.0) for n in (3, 9, 0)]
    texts, asum = host_table_csv(tables, ["a.png", "b.png", "c.png"], 8, False)
    assert texts[1] == b"" and asum[1] == -1
    assert texts[0] == pandas_csv(tables[0], "a.png", False)[1] and texts[2] == b"filename\n"


def test_bounds_and_argument_checks():
    from unet_dc_segmentation_b200 import _lib
    from unet_dc_segmentation_b200.quantify import table_csv_bounds
    nb, ws = table_csv_bounds(2, 10, True, 20)
    head = len("filename,label,area,equivalent_diameter,centroid-0,centroid-1,area_sqmicron,eq_diam_micron\n")
    assert nb == 2 * head + 10 * (20 + 2 * (10 + 20 + 5 * 24 + 7 + 1)) and ws >= 2 * 10 * 8
    with pytest.raises(_lib.DcError):
        table_csv_bounds(0, 10, False, 0)
    args = _lib.TableCsvArgs()
    assert _lib.load().dc_debug_table_csv_host(C.byref(args)) == _lib.DC_EINVAL


def test_csv_tables_include_is_current(tmp_path):
    """csrc/csv_tables.inc is generated (tools/gen_csv_tables.py); the committed copy must be what the generator writes."""
    import subprocess
    out = tmp_path / "csv_tables.inc"
    subprocess.run([sys.executable, str(REPO / "tools" / "gen_csv_tables.py"), str(out)], check=True)
    assert out.read_text() == (REPO / "unet_dc_segmentation_b200" / "csrc" / "csv_tables.inc").read_text()


# ------------------------------------------------------------------ all_droplets.csv
@pytest.mark.parametrize("pattern", ["all", "mixed", "leading_empty", "none"])
def test_combined_csv_equals_pandas_concat(pattern):
    """cli.combined_csv_bytes from the per-image files == pd.concat(per-image frames, ignore_index=True).to_csv of the
    installed pandas, which turns label / area into float64 when empty frames take part (pandas 3)."""
    from unet_dc_segmentation_b200 import cli
    from unet_dc_segmentation_b200.quantify import csv_field, text_encoding
    rs = np.random.default_rng(8)
    ns = {"all": [3, 5, 1, 7], "mixed": [3, 0, 5, 0, 2], "leading_empty": [0, 4, 2, 0], "none": [0, 0, 0]}[pattern]
    frames, texts, fields = [], [], []
    for b, n in enumerate(ns):
        name = NAMES[b % len(NAMES)]
        df, text = pandas_csv(random_table(rs, n, 3.45), name, True)
        frames.append(df)
        texts.append(text)
        fields.append(csv_field(name))
    want = pd.concat(frames, ignore_index=True).to_csv(index=False).encode(text_encoding())
    assert cli.combined_csv_bytes(texts, fields) == want
