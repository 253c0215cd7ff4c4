/* TEST DOUBLE -- the C ABI double of tests/_double/afesp_gpu_double.c, unchanged except that afesp_gpu_open loads the
 * bridge of tests/_frozen_core.py, whose engine honours the option "frozen_core".  Built into a temporary directory by
 * tests/test_frozen_core.py and LD_PRELOADed in front of libafesp_gpu.so; never part of the product.
 */
#include <Python.h>

static PyObject* import_frozen_core_bridge(const char* name) {
  (void)name;   /* "tests._double.bridge" in the included file */
  return PyImport_ImportModule("tests._frozen_core");
}
#define PyImport_ImportModule import_frozen_core_bridge
#include "_double/afesp_gpu_double.c"
