# otezip-b200 — gcc for the plain-C host library, nvcc (sm_100a only) for the kernels.
NVCC ?= /usr/local/cuda/bin/nvcc
CC ?= gcc
ARCH := -gencode arch=compute_100a,code=sm_100a
NVFLAGS := $(ARCH) -O3 -lineinfo -std=c++17 -Xcompiler -fPIC -Xptxas -v
CSRC := otezip_b200/csrc
LIB := otezip_b200/libotezip_b200.so
CUH := $(wildcard $(CSRC)/*.cuh) include/otz_gpu.h
HOST_C := $(wildcard $(CSRC)/host/*.c)
HOST_O := $(HOST_C:.c=.o)

all: $(LIB) oracle debug d64enc

$(CSRC)/otz_shim.o: $(CSRC)/otz_shim.cu $(CUH)
	$(NVCC) $(NVFLAGS) -c -o $@ $< 2> $(CSRC)/ptxas.log || (cat $(CSRC)/ptxas.log; false)

$(CSRC)/host/%.o: $(CSRC)/host/%.c $(wildcard include/otezip/*.h) include/otz_gpu.h
	$(CC) -O2 -Wall -Wextra -std=c99 -D_GNU_SOURCE -fPIC -Iinclude -c -o $@ $<

$(LIB): $(CSRC)/otz_shim.o $(HOST_O)
	$(NVCC) $(ARCH) -shared -o $@ $^ -lcudart_static -lpthread -ldl -lrt

# the same library with the kernels' software bounds checks compiled in (otz_common.cuh: OTZ_CHK; tests/test_gpu_bounds.py)
DBGLIB := otezip_b200/libotezip_b200_dbg.so
$(CSRC)/otz_shim_dbg.o: $(CSRC)/otz_shim.cu $(CUH)
	$(NVCC) $(NVFLAGS) -DOTZ_BOUNDS_CHECK -c -o $@ $< 2> $(CSRC)/ptxas_dbg.log || (cat $(CSRC)/ptxas_dbg.log; false)
$(DBGLIB): $(CSRC)/otz_shim_dbg.o $(HOST_O)
	$(NVCC) $(ARCH) -shared -o $@ $^ -lcudart_static -lpthread -ldl -lrt
debug: $(DBGLIB)

# Deflate64 / DEFLATE encoder of the tests and tools/deflate64_bench.py (tests/deflate64.py loads it with ctypes)
D64ENC := tools/libd64enc.so
$(D64ENC): tools/d64enc.c
	$(CC) -O2 -Wall -Wextra -std=c99 -fPIC -shared -o $@ $<

oracle: $(LIB)
	$(MAKE) -C oracle

clean:
	rm -f $(CSRC)/*.o $(CSRC)/host/*.o $(LIB) $(DBGLIB) $(D64ENC) $(CSRC)/ptxas.log $(CSRC)/ptxas_dbg.log
d64enc: $(D64ENC)
.PHONY: all oracle clean debug d64enc
