"""The ctypes mirrors of the per-group image descriptors of the C ABI
(include/mdpp_b200.h) have the header's fields, in order, and its size."""
import ctypes as C
import os
import re

import pytest

from mdp_playground_b200 import _lib

HEADER = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))),
                      "include", "mdpp_b200.h")


def header_fields(name):
    """Field names of `typedef struct name { ... } name;`, in order."""
    text = open(HEADER).read()
    body = re.search(r"typedef struct %s \{(.*?)\} %s;" % (name, name), text, re.S)
    assert body, name
    body = re.sub(r"/\*.*?\*/", "", body.group(1), flags=re.S)
    names = []
    for decl in body.split(";"):
        decl = decl.strip()
        if decl:
            # "int64_t env_begin, env_count" -> env_begin, env_count
            first, *rest = decl.split(",")
            names.append(first.split()[-1])
            names += [r.strip() for r in rest]
    return names


@pytest.mark.parametrize("name,cls,first,size", [
    ("mdpp_image_discrete_group", _lib.ImageDiscreteGroup,
     _lib.ImageDiscreteTables, C.sizeof(_lib.ImageDiscreteTables) + 3 * 8),
    ("mdpp_image_continuous_group", _lib.ImageContinuousGroup,
     _lib.ImageContinuousConfig, C.sizeof(_lib.ImageContinuousConfig) + 2 * 8),
])
def test_image_group_structs_match_the_header(name, cls, first, size):
    assert [f[0] for f in cls._fields_] == header_fields(name)
    assert cls._fields_[0][1] is first
    assert all(f[1] is C.c_int64 for f in cls._fields_[1:])
    # (the embedded struct's size is a multiple of 8: no padding in between)
    assert C.sizeof(first) % 8 == 0 and C.sizeof(cls) == size
    assert C.sizeof(_lib.ImageDiscreteGroup) == 128  # one 4-byte word per lane


def test_new_entry_points_are_exported_symbols():
    for sym in ("mdpp_set_image_discrete_groups", "mdpp_render_discrete_groups",
                "mdpp_set_image_continuous_groups", "mdpp_render_continuous_groups"):
        assert sym in _lib.EXPORTED_SYMBOLS
        assert re.search(r"\b%s\(" % sym, open(HEADER).read()), sym
