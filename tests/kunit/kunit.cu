// tests/kunit/kunit.cu -- TEST INFRASTRUCTURE, NOT PRODUCT CODE.
// GPU build of the single-case runners (kunit_cases.cuh): the product's device functions compiled by nvcc for sm_100a,
// run one warp per case.  Built by tests/kunit/kunit_py.py into libkunit.so, and with -DURMB_BIG into libkunit_big.so
// (the capacities of the build that maps reads over a capacity again: kRunCap 192).
#include "kunit_cases.cuh"
