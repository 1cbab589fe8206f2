"""CPU-only checks of the remove entry points: a NULL handle, or n > 0 with NULL labels, is refused with DAWN_ERR_INVALID
before the handle is used or the GPU is touched, so the refusal holds on a host without a GPU."""
import ctypes as C

DAWN_ERR_INVALID = -1


def test_index_remove_refuses_a_null_handle(dawn):
    lib = dawn.load_library()
    labels = (C.c_uint64 * 2)(5, 6)
    removed = C.c_size_t(7)
    assert lib.dawn_index_remove(None, 5, C.byref(removed)) == DAWN_ERR_INVALID
    assert removed.value == 0
    assert b"null index handle" in lib.dawn_last_error()
    removed.value = 7
    assert lib.dawn_index_remove_batch(None, labels, 2, C.byref(removed)) == DAWN_ERR_INVALID
    assert removed.value == 0
    assert lib.dawn_index_remove_batch(None, None, 0, None) == DAWN_ERR_INVALID


def test_index_remove_refuses_null_labels_before_using_the_handle(dawn):
    lib = dawn.load_library()
    # stands in for a handle: the NULL-labels check comes first, so it is never dereferenced
    not_a_handle = C.create_string_buffer(64)
    removed = C.c_size_t(7)
    assert lib.dawn_index_remove_batch(C.cast(not_a_handle, C.c_void_p), None, 3, C.byref(removed)) == DAWN_ERR_INVALID
    assert removed.value == 0
    assert b"labels is null" in lib.dawn_last_error()


def test_multi_remove_validates_its_arguments(dawn):
    lib = dawn.load_library()
    labels = (C.c_uint64 * 1)(9)
    removed = C.c_size_t(7)
    assert lib.dawn_multi_remove(None, 9, C.byref(removed)) == DAWN_ERR_INVALID
    assert removed.value == 0
    assert lib.dawn_multi_remove_batch(None, labels, 1, None) == DAWN_ERR_INVALID
    assert b"null multi handle" in lib.dawn_multi_last_error()
    not_a_handle = C.create_string_buffer(64)
    removed.value = 7
    assert lib.dawn_multi_remove_batch(C.cast(not_a_handle, C.c_void_p), None, 1, C.byref(removed)) == DAWN_ERR_INVALID
    assert removed.value == 0
    assert b"labels is null" in lib.dawn_multi_last_error()


def test_python_bindings_expose_remove(dawn):
    for cls in (dawn.Index, dawn.MultiIndex):
        assert callable(getattr(cls, "remove")) and callable(getattr(cls, "remove_batch"))
