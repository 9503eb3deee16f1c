"""Metadata loaders (reference file formats) and the synthetic recipe."""
import numpy as np
import pytest

from mplan2vdl_b200 import meta, synth
from oracle.oracle import gen_column
from util import FIXTURES, needs_reference


def test_loaders_on_a_tiny_directory(tmp_path):
    (tmp_path / "bounds.csv").write_text("fact,f_val,100,5000,10,2\nfact,f_date,727564,730089,10,0\nfact,fact_dim,0,4,10,0\n"
                                         "dim,d_key,1,5,5,0\ndim,dim_d_key_pkey,-9223372036854775808,-9223372036854775808,5,63\n")
    (tmp_path / "storage.csv").write_text("sys,fact,f_val,decimal,06/1,10,8,80,0,0,0,false\nsys,fact,f_date,date,06/2,10,4,40,0,0,0,true\n"
                                          "sys,fact,fact_dim,oid,06/3,10,8,80,0,0,0,false\nsys,dim,d_key,int,06/4,5,4,20,0,0,0,true\n")
    (tmp_path / "dictionary.csv").write_text('dim,d_name,"ASIA",64\n')
    (tmp_path / "schema.msqldump").write_text(
        'SET SCHEMA "sys";\nCREATE TABLE "sys"."dim" (\n\t"d_key" INTEGER NOT NULL,\n\tCONSTRAINT "dim_d_key_pkey" PRIMARY KEY ("d_key")\n);\n'
        'CREATE TABLE "sys"."fact" (\n\t"f_val" DECIMAL(15,2),\n\tCONSTRAINT "fact_dim" FOREIGN KEY ("f_key") REFERENCES "sys"."dim" ("d_key")\n);\n')
    cat = meta.load_metadata(str(tmp_path))
    assert cat.column("fact.f_val").width == 8 and cat.column("fact.f_date").width == 4
    assert cat.column("fact.f_date").is_sorted and cat.column("fact.f_val").trailing_zeros == 2
    assert cat.tables["fact"].rows == 10 and cat.tables["dim"].pkey == ["d_key"]
    fk = cat.tables["fact"].fkeys[0]
    assert (fk.name, fk.ref_table, fk.ref_columns) == ("fact_dim", "dim", ["d_key"])
    assert cat.decode("dim.d_name", 64) == "ASIA"
    rt = meta.Catalog.from_json(cat.to_json())
    assert rt.to_json() == cat.to_json()


def test_bad_record_width_is_rejected(tmp_path):
    (tmp_path / "bounds.csv").write_text("t,c,0,1,5\n")       # the stale 5-column format (SURVEY.md section 2.1)
    with pytest.raises(ValueError):
        meta.read_bounds(str(tmp_path / "bounds.csv"))


@needs_reference
def test_builtin_catalog_is_the_reference_metadata():
    assert meta.load_metadata(FIXTURES).to_json() == meta.builtin_catalog().to_json()


def test_builtin_catalog_facts(catalog):
    li = catalog.tables["lineitem"]
    assert li.rows == 59_986_052 and catalog.tables["orders"].rows == 15_000_000       # bounds.csv:48,59
    assert [catalog.column("lineitem." + c).width for c in ("l_quantity", "l_extendedprice", "l_discount", "l_shipdate")] == [8, 8, 8, 4]
    assert catalog.column("lineitem.l_returnflag").width == 8      # char -> SInt64 (Types.hs:134)
    assert catalog.dictionary["customer.c_mktsegment"]["BUILDING"] == 16
    assert {f.name: f.ref_table for f in li.fkeys}["lineitem_orders"] == "orders"


def test_columns_respect_bounds_and_trailing_zeros(catalog):
    for name in ("l_quantity", "l_extendedprice", "l_discount", "l_tax", "l_shipdate"):
        spec = synth.column_spec(catalog, "lineitem." + name, 1)
        col = catalog.column("lineitem." + name)
        a = gen_column(spec, 200_000, 0, synth.seed_for(1))
        assert a.min() >= col.vmin and a.max() <= col.vmax
        assert not np.any(a & ((1 << col.trailing_zeros) - 1))
        assert a.dtype.itemsize == col.width
    rf = gen_column(synth.column_spec(catalog, "lineitem.l_returnflag", 1), 10_000, 0, 1)
    assert set(np.unique(rf)) == {16, 40, 64}


def test_generation_is_counter_based(catalog):
    spec = synth.column_spec(catalog, "lineitem.l_extendedprice", 1)
    whole = gen_column(spec, 10_000, 0, 42)
    parts = np.concatenate([gen_column(spec, 3_000, 0, 42), gen_column(spec, 7_000, 3_000, 42)])
    np.testing.assert_array_equal(whole, parts)
    assert not np.array_equal(whole, gen_column(spec, 10_000, 0, 43))


def test_fk_columns_are_consistent(catalog):
    sf = 0.01
    n_li, n_o = synth.table_rows(catalog, "lineitem", sf), synth.table_rows(catalog, "orders", sf)
    fk = gen_column(synth.column_spec(catalog, "lineitem.lineitem_orders", sf), n_li, 0, 1)
    ok = gen_column(synth.column_spec(catalog, "lineitem.l_orderkey", sf), n_li, 0, 1)
    okeys = gen_column(synth.column_spec(catalog, "orders.o_orderkey", sf), n_o, 0, 1)
    assert fk.min() == 0 and fk.max() == n_o - 1 and np.all(np.diff(fk) >= 0)      # clustered, every order hit
    np.testing.assert_array_equal(okeys[fk], ok)
    oc = gen_column(synth.column_spec(catalog, "orders.orders_customer", sf), n_o, 0, 1)
    ck = gen_column(synth.column_spec(catalog, "orders.o_custkey", sf), n_o, 0, 1)
    np.testing.assert_array_equal(oc + 1, ck)
    assert oc.max() < synth.table_rows(catalog, "customer", sf)
