"""The C header, the ctypes binding and DuckDB's own enums agree.

* include/duckdb_b200.h is plain C: it compiles with `gcc -std=c99 -pedantic`, and the struct layouts /
  enum values a C program sees are the ones duckdb_b200/capi.py declares to ctypes.
* b200_type / b200_vector_type / b200_expr_op / b200_join_type reuse the numeric values of DuckDB's
  PhysicalType / VectorType / ExpressionType / JoinType (INTEGRATION.md: the shim passes them through without a
  mapping table).  Checked against the values read from the reference's headers (tests/golden/reference_answers.json).
"""
import ctypes as C
import os
import subprocess

import pytest

from conftest import reference_answers
from duckdb_b200 import capi

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

PROBE = r"""
#include <stddef.h>
#include <stdio.h>
#include "duckdb_b200.h"
#define SZ(T) printf("sizeof %s %zu\n", #T, sizeof(T))
#define OFF(T, F) printf("offsetof %s.%s %zu\n", #T, #F, offsetof(T, F))
#define VAL(E) printf("enum %s %d\n", #E, (int)(E))
int main(void) {
	SZ(b200_vector); OFF(b200_vector, type); OFF(b200_vector, vector_type); OFF(b200_vector, data);
	OFF(b200_vector, sel); OFF(b200_vector, validity); OFF(b200_vector, dict_size);
	SZ(b200_expr_node); OFF(b200_expr_node, op); OFF(b200_expr_node, type); OFF(b200_expr_node, left);
	OFF(b200_expr_node, right); OFF(b200_expr_node, col); OFF(b200_expr_node, is_null); OFF(b200_expr_node, value);
	SZ(b200_agg_desc); OFF(b200_agg_desc, func); OFF(b200_agg_desc, input_type); OFF(b200_agg_desc, input);
	OFF(b200_agg_desc, reserved);
	VAL(B200_OK); VAL(B200_ERR_INVALID); VAL(B200_ERR_NO_DEVICE); VAL(B200_ERR_CUDA); VAL(B200_ERR_OOM);
	VAL(B200_ERR_OVERFLOW); VAL(B200_ERR_CAPACITY);
	VAL(B200_BOOL); VAL(B200_UINT8); VAL(B200_INT8); VAL(B200_UINT16); VAL(B200_INT16); VAL(B200_UINT32);
	VAL(B200_INT32); VAL(B200_UINT64); VAL(B200_INT64); VAL(B200_FLOAT); VAL(B200_DOUBLE); VAL(B200_INT128);
	VAL(B200_FLAT_VECTOR); VAL(B200_CONSTANT_VECTOR); VAL(B200_DICTIONARY_VECTOR);
	VAL(B200_EXPR_COLREF); VAL(B200_EXPR_CONST); VAL(B200_EXPR_NOT); VAL(B200_EXPR_IS_NULL);
	VAL(B200_EXPR_IS_NOT_NULL); VAL(B200_EXPR_EQ); VAL(B200_EXPR_NE); VAL(B200_EXPR_LT); VAL(B200_EXPR_GT);
	VAL(B200_EXPR_LE); VAL(B200_EXPR_GE); VAL(B200_EXPR_DISTINCT); VAL(B200_EXPR_NOT_DISTINCT); VAL(B200_EXPR_AND);
	VAL(B200_EXPR_OR); VAL(B200_EXPR_ADD); VAL(B200_EXPR_SUB); VAL(B200_EXPR_MUL); VAL(B200_EXPR_CAST);
	VAL(B200_AGG_COUNT_STAR); VAL(B200_AGG_COUNT); VAL(B200_AGG_SUM); VAL(B200_AGG_SUM_NO_OVERFLOW);
	VAL(B200_AGG_MIN); VAL(B200_AGG_MAX); VAL(B200_AGG_AVG);
	VAL(B200_JOIN_LEFT); VAL(B200_JOIN_INNER); VAL(B200_JOIN_SEMI); VAL(B200_JOIN_ANTI); VAL(B200_JOIN_MARK);
	return 0;
}
"""


@pytest.fixture(scope="module")
def c_view(tmp_path_factory):
    """What a C99 compiler sees in the header: {('sizeof', T): n, ('offsetof', 'T.f'): n, ('enum', NAME): v}."""
    d = tmp_path_factory.mktemp("abi")
    src, exe = d / "probe.c", d / "probe"
    src.write_text(PROBE)
    subprocess.check_call(["gcc", "-std=c99", "-pedantic", "-Wall", "-Werror", "-I", os.path.join(ROOT, "include"),
                           str(src), "-o", str(exe)])
    out = subprocess.check_output([str(exe)], text=True)
    view = {}
    for line in out.splitlines():
        kind, name, value = line.split()
        view[(kind, name)] = int(value)
    return view


@pytest.mark.parametrize("cname,ctype", [("b200_vector", capi.Vector), ("b200_expr_node", capi.ExprNode),
                                         ("b200_agg_desc", capi.AggDesc)])
def test_struct_layouts_match_ctypes(c_view, cname, ctype):
    assert c_view[("sizeof", cname)] == C.sizeof(ctype)
    for field, _ in ctype._fields_:
        assert c_view[("offsetof", f"{cname}.{field}")] == getattr(ctype, field).offset, field


def test_enum_values_match_ctypes_constants(c_view):
    pairs = {
        "B200_OK": capi.OK, "B200_ERR_INVALID": capi.ERR_INVALID, "B200_ERR_NO_DEVICE": capi.ERR_NO_DEVICE,
        "B200_ERR_CUDA": capi.ERR_CUDA, "B200_ERR_OOM": capi.ERR_OOM, "B200_ERR_OVERFLOW": capi.ERR_OVERFLOW,
        "B200_ERR_CAPACITY": capi.ERR_CAPACITY,
        "B200_BOOL": capi.BOOL, "B200_UINT8": capi.UINT8, "B200_INT8": capi.INT8, "B200_UINT16": capi.UINT16,
        "B200_INT16": capi.INT16, "B200_UINT32": capi.UINT32, "B200_INT32": capi.INT32, "B200_UINT64": capi.UINT64,
        "B200_INT64": capi.INT64, "B200_FLOAT": capi.FLOAT, "B200_DOUBLE": capi.DOUBLE, "B200_INT128": capi.INT128,
        "B200_FLAT_VECTOR": capi.FLAT_VECTOR, "B200_CONSTANT_VECTOR": capi.CONSTANT_VECTOR,
        "B200_DICTIONARY_VECTOR": capi.DICTIONARY_VECTOR,
        "B200_EXPR_COLREF": capi.EXPR_COLREF, "B200_EXPR_CONST": capi.EXPR_CONST, "B200_EXPR_NOT": capi.EXPR_NOT,
        "B200_EXPR_IS_NULL": capi.EXPR_IS_NULL, "B200_EXPR_IS_NOT_NULL": capi.EXPR_IS_NOT_NULL,
        "B200_EXPR_EQ": capi.EXPR_EQ, "B200_EXPR_NE": capi.EXPR_NE, "B200_EXPR_LT": capi.EXPR_LT,
        "B200_EXPR_GT": capi.EXPR_GT, "B200_EXPR_LE": capi.EXPR_LE, "B200_EXPR_GE": capi.EXPR_GE,
        "B200_EXPR_DISTINCT": capi.EXPR_DISTINCT, "B200_EXPR_NOT_DISTINCT": capi.EXPR_NOT_DISTINCT,
        "B200_EXPR_AND": capi.EXPR_AND, "B200_EXPR_OR": capi.EXPR_OR, "B200_EXPR_ADD": capi.EXPR_ADD,
        "B200_EXPR_SUB": capi.EXPR_SUB, "B200_EXPR_MUL": capi.EXPR_MUL, "B200_EXPR_CAST": capi.EXPR_CAST,
        "B200_AGG_COUNT_STAR": capi.AGG_COUNT_STAR, "B200_AGG_COUNT": capi.AGG_COUNT, "B200_AGG_SUM": capi.AGG_SUM,
        "B200_AGG_SUM_NO_OVERFLOW": capi.AGG_SUM_NO_OVERFLOW, "B200_AGG_MIN": capi.AGG_MIN,
        "B200_AGG_MAX": capi.AGG_MAX, "B200_AGG_AVG": capi.AGG_AVG,
        "B200_JOIN_LEFT": capi.JOIN_LEFT, "B200_JOIN_INNER": capi.JOIN_INNER, "B200_JOIN_SEMI": capi.JOIN_SEMI,
        "B200_JOIN_ANTI": capi.JOIN_ANTI, "B200_JOIN_MARK": capi.JOIN_MARK,
    }
    for name, value in pairs.items():
        assert c_view[("enum", name)] == value, name
    for t, size in capi.TYPE_SIZE.items():
        if t in capi.DTYPE_OF_TYPE:
            assert capi.DTYPE_OF_TYPE[t].itemsize == size


def test_enum_values_are_duckdbs(c_view):
    duckdb = reference_answers("enums")
    physical = duckdb["PhysicalType"]
    for ours, theirs in [("B200_BOOL", "BOOL"), ("B200_UINT8", "UINT8"), ("B200_INT8", "INT8"),
                         ("B200_UINT16", "UINT16"), ("B200_INT16", "INT16"), ("B200_UINT32", "UINT32"),
                         ("B200_INT32", "INT32"), ("B200_UINT64", "UINT64"), ("B200_INT64", "INT64"),
                         ("B200_FLOAT", "FLOAT"), ("B200_DOUBLE", "DOUBLE"), ("B200_INT128", "INT128")]:
        assert c_view[("enum", ours)] == physical[theirs], ours
    expr = duckdb["ExpressionType"]
    for ours, theirs in [("B200_EXPR_COLREF", "BOUND_REF"), ("B200_EXPR_CONST", "VALUE_CONSTANT"),
                         ("B200_EXPR_NOT", "OPERATOR_NOT"), ("B200_EXPR_IS_NULL", "OPERATOR_IS_NULL"),
                         ("B200_EXPR_IS_NOT_NULL", "OPERATOR_IS_NOT_NULL"), ("B200_EXPR_EQ", "COMPARE_EQUAL"),
                         ("B200_EXPR_NE", "COMPARE_NOTEQUAL"), ("B200_EXPR_LT", "COMPARE_LESSTHAN"),
                         ("B200_EXPR_GT", "COMPARE_GREATERTHAN"), ("B200_EXPR_LE", "COMPARE_LESSTHANOREQUALTO"),
                         ("B200_EXPR_GE", "COMPARE_GREATERTHANOREQUALTO"), ("B200_EXPR_DISTINCT", "COMPARE_DISTINCT_FROM"),
                         ("B200_EXPR_NOT_DISTINCT", "COMPARE_NOT_DISTINCT_FROM"), ("B200_EXPR_AND", "CONJUNCTION_AND"),
                         ("B200_EXPR_OR", "CONJUNCTION_OR")]:
        assert c_view[("enum", ours)] == expr[theirs], ours
    join = duckdb["JoinType"]
    for ours, theirs in [("B200_JOIN_LEFT", "LEFT"), ("B200_JOIN_INNER", "INNER"), ("B200_JOIN_SEMI", "SEMI"),
                         ("B200_JOIN_ANTI", "ANTI"), ("B200_JOIN_MARK", "MARK")]:
        assert c_view[("enum", ours)] == join[theirs], ours
    vec = duckdb["VectorType"]
    for ours, theirs in [("B200_FLAT_VECTOR", "FLAT_VECTOR"), ("B200_CONSTANT_VECTOR", "CONSTANT_VECTOR"),
                         ("B200_DICTIONARY_VECTOR", "DICTIONARY_VECTOR")]:
        assert c_view[("enum", ours)] == vec[theirs], ours


def test_expression_programs_list_children_before_parents():
    """operators.Expr emits post-order programs: every child index is smaller than its parent's (the kernel
    evaluates nodes by index and the shim's TranslateExpression emits the same order)."""
    from duckdb_b200 import operators as ops

    e = ops.Expr()
    a = e.col(0, capi.INT32)
    b = e.const(8766, capi.INT32)
    lt = e.cmp(capi.EXPR_LT, a, b)
    c = e.col(1, capi.INT64)
    ge = e.cmp(capi.EXPR_GE, c, e.const(5, capi.INT64))
    root = e.and_(lt, e.not_(e.is_null(ge)))
    nodes = e.array()
    assert root == len(e.nodes) - 1
    for i, n in enumerate(e.nodes):
        assert n.left < i and n.right < i
    assert nodes[b].value.i == 8766 and nodes[b].is_null == 0
    assert nodes[lt].op == capi.EXPR_LT and nodes[lt].type == capi.BOOL
    null_const = e.const(None, capi.DOUBLE, is_null=True)
    assert e.nodes[null_const].is_null == 1
