# Top-level build: product library (CUDA, sm_100a), data generator, CPU checker.
NVCC   ?= /usr/local/cuda/bin/nvcc
CC     ?= gcc
CXX    ?= g++
PKG    := streamly_lz4_b200
CSRC   := $(PKG)/csrc
ARCH   := -gencode arch=compute_100a,code=sm_100a
EXTRA  ?=
NVFLAGS := $(EXTRA) $(ARCH) -O3 -lineinfo -std=c++17 -Xcompiler -fPIC,-Wall,-Wno-unused-function -Xptxas -v -Iinclude -I$(CSRC)

LIB    := $(PKG)/libb200lz4.so
BOUNDS := $(PKG)/libb200lz4_bounds.so
GEN    := $(PKG)/datagen/libb200gen.so

CU_SRCS  := $(wildcard $(CSRC)/*.cu)
CU_HDRS  := $(wildcard $(CSRC)/*.cuh) $(wildcard $(CSRC)/*.h) $(wildcard $(CSRC)/*.hpp) include/b200lz4.h

all: $(LIB) $(BOUNDS) $(GEN) oracle

$(LIB): $(CU_SRCS) $(CU_HDRS)
	$(NVCC) $(NVFLAGS) -shared -o $@ $(CU_SRCS) 2> $(CSRC)/ptxas.log || (cat $(CSRC)/ptxas.log; false)
	@grep -E "registers|spill|error|warning" $(CSRC)/ptxas.log | sort | uniq -c | sort -rn | head -40 || true

$(GEN): $(PKG)/datagen/datagen.c
	$(CC) -O2 -fPIC -shared -o $@ $<

oracle:
	$(MAKE) -s -C oracle

# debug build of the same library with destination-bounds checks in the decoder kernels (tests/test_gpu_modes.py)
bounds: $(BOUNDS)
$(BOUNDS): $(CU_SRCS) $(CU_HDRS)
	$(NVCC) $(NVFLAGS) -DB200LZ4_BOUNDS_CHECK -shared -o $@ $(CU_SRCS) 2> /dev/null

# development build with cycle accounting in the wide decoder (load it with B200LZ4_LIB=build/libb200lz4_stats.so)
stats: $(CU_SRCS) $(CU_HDRS)
	mkdir -p build
	$(NVCC) $(NVFLAGS) -DB200LZ4_WIDE_STATS -shared -o build/libb200lz4_stats$(SUFFIX).so $(CU_SRCS) 2> build/ptxas_stats.log || (cat build/ptxas_stats.log; false)

clean:
	rm -f $(LIB) $(BOUNDS) $(GEN) $(CSRC)/ptxas.log
	$(MAKE) -C oracle clean

.PHONY: all oracle clean stats bounds

# plain-C example over the C ABI (needs a B200 to run)
examples: $(LIB)
	mkdir -p build
	$(CC) -O2 -Wall -Iinclude examples/c_roundtrip.c -L$(PKG) -lb200lz4 -Wl,-rpath,$(CURDIR)/$(PKG) -o build/c_roundtrip

.PHONY: examples
