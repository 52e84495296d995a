# tests/cpp/sparse.mk — builds the compiled SparsifiedGP drop-in test (the reference's own limbo::model::SparsifiedGP and
# MultiGP next to limbo_b200::model::SparsifiedGP).  Needs the reference's sources; the binary goes to oracle/_ref/
# (git-ignored) and is run by tests/test_gpu_sparse_dropin_cpp.py.
CXX ?= g++
REF ?= /root/reference/src
ROOT := ../..
OUT := $(ROOT)/oracle/_ref/sparse_dropin_test
all: $(OUT)
$(OUT): sparse_dropin_test.cpp $(ROOT)/include/limbo_b200/model/sparsified_gp.hpp $(ROOT)/include/limbo_b200/model/gp.hpp $(ROOT)/include/limbo_b200.h $(ROOT)/oracle/ref_sparse/Eigen/Core
	mkdir -p $(ROOT)/oracle/_ref
	$(CXX) -O2 -std=c++17 -w -DNDEBUG -ffp-contract=off -I$(ROOT)/oracle/ref_sparse -I$(ROOT)/oracle/ref_shim -I$(REF) -I$(ROOT)/include sparse_dropin_test.cpp -o $@ \
	  -L$(ROOT)/limbo_b200/lib -llimbo_b200 -Wl,-rpath,'$$ORIGIN/../../limbo_b200/lib'
