# Builds libadt_b200.so (sm_100a) in-tree.  `python -c "import __graft_entry__ as g; g.build()"` calls this.
NVCC ?= /usr/local/cuda/bin/nvcc
NVFLAGS = -gencode arch=compute_100a,code=sm_100a -lineinfo -O3 -std=c++17 --expt-extended-lambda --expt-relaxed-constexpr \
          -Xcompiler -fPIC -shared
SRC = adt_b200/csrc/api.cu adt_b200/csrc/score.cu adt_b200/csrc/score_tc.cu adt_b200/csrc/sampler.cu adt_b200/csrc/gemm_tc.cu adt_b200/csrc/flash_tc.cu
HDR = $(wildcard adt_b200/csrc/*.cuh) include/adt_b200.h
LIB = adt_b200/lib/libadt_b200.so

all: $(LIB)

$(LIB): $(SRC) $(HDR)
	mkdir -p adt_b200/lib
	$(NVCC) $(NVFLAGS) -o $@ $(SRC)

clean:
	rm -f $(LIB)
.PHONY: all clean
