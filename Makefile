# Builds libsqeazy.so (the drop-in C-ABI library: hand-written sm_100a kernels + C++17 host code)
# and the test-only oracle libraries. `python -c "import __graft_entry__ as g; g.build()"` runs this.
NVCC      ?= /usr/local/cuda/bin/nvcc
CXX       ?= g++
ARCH      := -gencode arch=compute_100a,code=sm_100a
NVFLAGS   := $(ARCH) -O3 -std=c++17 -lineinfo -Xcompiler -fPIC,-fvisibility=default,-ffp-contract=off -Xptxas -v
CSRC      := sqeazy_b200/csrc
OBJDIR    := build/obj
LIB       := sqeazy_b200/libsqeazy.so

CU_SRCS   := $(CSRC)/api.cu $(CSRC)/staging.cu $(CSRC)/device/bitswap.cu $(CSRC)/device/bitshuffle.cu $(CSRC)/device/diff.cu $(CSRC)/device/quantise.cu $(CSRC)/device/lz4_encode.cu $(CSRC)/device/lz4_decode.cu $(CSRC)/device/roi.cu
CPP_SRCS  := $(CSRC)/host/text.cpp $(CSRC)/host/numerics.cpp $(CSRC)/host/pipeline.cpp $(CSRC)/host/h5_filter.cpp
CU_OBJS   := $(patsubst $(CSRC)/%.cu,$(OBJDIR)/%.o,$(CU_SRCS))
CPP_OBJS  := $(patsubst $(CSRC)/%.cpp,$(OBJDIR)/%.o,$(CPP_SRCS))
HDRS      := $(wildcard $(CSRC)/*.hpp $(CSRC)/*.inl $(CSRC)/device/*.h $(CSRC)/device/*.cuh $(CSRC)/host/*.hpp include/*.h)

REF       := /root/reference/src/cpp/src
LZ4SO     := /usr/lib/x86_64-linux-gnu/liblz4.so.1

SQY       := sqeazy_b200/bin/sqy

all: $(LIB) $(SQY) oracle

$(OBJDIR)/%.o: $(CSRC)/%.cu $(HDRS)
	@mkdir -p $(dir $@)
	$(NVCC) $(NVFLAGS) -c $< -o $@ 2> $@.ptxas.log || (cat $@.ptxas.log; exit 1)

$(OBJDIR)/%.o: $(CSRC)/%.cpp $(HDRS)
	@mkdir -p $(dir $@)
	$(CXX) -O2 -std=c++17 -fPIC -ffp-contract=off -Wall -c $< -o $@

$(LIB): $(CU_OBJS) $(CPP_OBJS)
	$(NVCC) $(ARCH) -shared -o $@ $^ -cudart static -ldl

# ---- sqy command line tool: a plain C++ client of the C ABI (no CUDA in this translation unit)
$(SQY): $(CSRC)/cli/sqy.cpp $(CSRC)/cli/tiff_min.hpp include/sqeazy.h include/sqeazy_b200.h $(LIB)
	@mkdir -p $(dir $@)
	$(CXX) -O2 -std=c++17 -Wall -o $@ $(CSRC)/cli/sqy.cpp -Lsqeazy_b200 -lsqeazy -Wl,-rpath,'$$ORIGIN/..'

# ---- test-only oracle: C restatement (always) and the compiled reference stages (when /root/reference exists)
oracle: oracle/_build/libsqyoracle.so oracle/_build/libdiff_sim.so oracle_ref

oracle/_build/libsqyoracle.so: oracle/sqy_oracle.c
	@mkdir -p oracle/_build
	gcc -O2 -std=c11 -fPIC -shared -ffp-contract=off -Wall -o $@ $<

# CPU replay of the diff3x3x1 kernels' thread program (tests/test_diff_cpu.py)
oracle/_build/libdiff_sim.so: tests/helpers/diff_sim.cpp $(CSRC)/device/diff_thread.h
	@mkdir -p oracle/_build
	g++ -O2 -std=c++17 -fPIC -shared -I$(CSRC)/device -o $@ $<

oracle_ref:
	@if [ -d $(REF) ]; then $(MAKE) oracle/_ref/libsqyref.so; else echo "no /root/reference: using prebuilt oracle/_ref if present"; fi

oracle/_ref/libsqyref.so: oracle/ref_harness.cpp $(wildcard oracle/refshim/*.hpp oracle/refshim/lz4inc/*.h)
	@mkdir -p oracle/_ref
	g++ -std=c++14 -O3 -march=x86-64 -msse4.2 -ftree-vectorize -fopenmp -DNDEBUG -D_SQY_X_=0 -include cmath -fPIC -shared \
	    -Ioracle/refshim -Ioracle/refshim/lz4inc -I$(REF) -I$(REF)/encoders oracle/ref_harness.cpp $(LZ4SO) -o $@

clean:
	rm -rf build $(LIB) sqeazy_b200/bin oracle/_build oracle/_ref/libsqyref.so

.PHONY: all oracle oracle_ref clean
