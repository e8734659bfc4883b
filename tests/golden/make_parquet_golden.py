"""Generates tests/golden/parquet_testing.json from the Apache parquet-testing corpus that the
reference vendors under thirdparty/parquet-testing/data (the fixtures its own
integration_tests/src/main/python/parquet_testing_test.py reads):

    python tests/golden/make_parquet_golden.py <spark-rapids source checkout>

The tests read only the committed JSON, never the checkout.

Each entry: file bytes (base64), the flat columns we decode, and the expected values as decoded by
pyarrow (the independent reader), normalised to python values: decimals -> unscaled ints,
dates -> days, timestamps -> microseconds, binary/strings -> latin-1 text.
"""
import base64
import decimal
import json
import os

import pyarrow as pa
import pyarrow.parquet as pq

SRC = os.path.join("thirdparty", "parquet-testing", "data")
FILES = {
    "alltypes_plain.parquet": ["id", "bool_col", "tinyint_col", "smallint_col", "int_col", "bigint_col", "float_col", "double_col", "date_string_col", "string_col"],
    "alltypes_plain.snappy.parquet": ["id", "bool_col", "int_col", "bigint_col", "float_col", "double_col", "string_col"],
    "alltypes_dictionary.parquet": ["id", "bool_col", "tinyint_col", "int_col", "bigint_col", "float_col", "double_col", "date_string_col", "string_col"],
    "int32_decimal.parquet": ["value"],
    "int64_decimal.parquet": ["value"],
    "fixed_length_decimal.parquet": ["value"],
    "fixed_length_decimal_legacy.parquet": ["value"],
    "datapage_v1-snappy-compressed-checksum.parquet": ["a", "b"],
    "plain-dict-uncompressed-checksum.parquet": ["long_field", "binary_field"],
    "rle-dict-snappy-checksum.parquet": ["long_field", "binary_field"],
    "datapage_v2.snappy.parquet": ["a", "c"],
    "binary.parquet": ["foo"],
    "int32_with_null_pages.parquet": ["int32_field"],
    "dict-page-offset-zero.parquet": ["l_partkey"],
    "single_nan.parquet": ["mycol"],
    "nan_in_stats.parquet": ["x"],
}
# the reference's own Scala/pytest fixtures (tests/src/test/resources): Spark-written decimals as INT32/INT64 and as legacy
# FIXED_LEN_BYTE_ARRAY, timestamp/date columns, a 10-row-group file its split tests read, an unsigned 64-bit column
SRC2 = os.path.join("tests", "src", "test", "resources")
FILES2 = {
    "decimal-test.parquet": ["c_0", "c_1", "c_2", "c_3", "c_4", "c_5"],
    "decimal-test-legacy.parquet": ["c_0", "c_1", "c_2", "c_3", "c_4", "c_5"],
    "timestamp-date-test.parquet": ["time", "date"],
    "file-splits.parquet": ["loan_id", "orig_channel", "orig_interest_rate", "orig_upb", "orig_date", "dti", "zip", "seller_id"],
    "test_unsigned64.parquet": ["simple_uint64"],
}
# DELTA_BINARY_PACKED: the integer columns of the corpus' delta files (selected by their encoding); these files come
# with the corpus' own *_expect.csv goldens, which the generator checks pyarrow against before trusting it
DELTA_FILES = ["delta_binary_packed.parquet", "delta_encoding_required_column.parquet", "delta_encoding_optional_column.parquet"]


def delta_int_columns(path):
    md = pq.ParquetFile(path).metadata
    rg = md.row_group(0)
    cols = []
    for c in range(rg.num_columns):
        cc = rg.column(c)
        if cc.physical_type in ("INT32", "INT64") and set(cc.encodings) <= {"DELTA_BINARY_PACKED", "RLE"}:
            cols.append(cc.path_in_schema)
    return cols


def check_against_expect_csv(path, tbl, cols):
    import csv
    rows = list(csv.reader(open(path.replace(".parquet", "_expect.csv"))))
    hdr = [h.strip() for h in rows[0]]
    for c in cols:
        j = hdr.index(c.strip().rstrip(":"))
        exp = [None if r[j] in ("", "NULL", "null") else int(r[j]) for r in rows[1:]]
        got = tbl.column(c).to_pylist()
        assert got == exp, (path, c)


def norm(v, typ):
    if v is None:
        return None
    if pa.types.is_decimal(typ):
        return int(decimal.Decimal(v).scaleb(typ.scale))
    if pa.types.is_binary(typ) or pa.types.is_string(typ) or pa.types.is_large_string(typ):
        return (v if isinstance(v, bytes) else v.encode()).decode("latin-1")
    if pa.types.is_floating(typ):
        return "nan" if v != v else float(v)
    if pa.types.is_boolean(typ):
        return bool(v)
    return int(v)


def main(checkout):
    out = {}
    files = dict(FILES)
    for name in DELTA_FILES:
        files[name] = delta_int_columns(os.path.join(checkout, SRC, name))
    srcdir = {name: os.path.join(checkout, SRC) for name in files}
    for name, cols in FILES2.items():
        files["spark_rapids_tests/" + name] = cols
        srcdir["spark_rapids_tests/" + name] = os.path.join(checkout, SRC2)
    for name, cols in files.items():
        path = os.path.join(srcdir[name], os.path.basename(name))
        raw = open(path, "rb").read()
        tbl = pq.read_table(path, columns=cols)
        if name in DELTA_FILES:
            check_against_expect_csv(path, tbl, cols)
        expect = {}
        for c in cols:
            col = tbl.column(c)
            typ = col.type
            if pa.types.is_date32(typ):
                vals = [None if v is None else int(v) for v in col.cast(pa.int32()).to_pylist()]
            elif pa.types.is_timestamp(typ):
                vals = [None if v is None else int(v) for v in col.cast(pa.timestamp("us")).cast(pa.int64()).to_pylist()]
            elif pa.types.is_uint64(typ):   # cudf UINT64 is delivered as the same 64 bits; the library's INT64 view is two's complement
                vals = [None if v is None else (int(v) - (1 << 64) if int(v) >= (1 << 63) else int(v)) for v in col.to_pylist()]
            else:
                vals = [norm(v, typ) for v in col.to_pylist()]
            expect[c] = {"type": str(typ), "values": vals}
        out[name] = {"b64": base64.b64encode(raw).decode(), "columns": cols, "expect": expect}
    dst = os.path.join(os.path.dirname(os.path.abspath(__file__)), "parquet_testing.json")
    with open(dst, "w") as fh:
        json.dump(out, fh)
    print("wrote", dst, os.path.getsize(dst), "bytes")


if __name__ == "__main__":
    import sys
    main(sys.argv[1])
