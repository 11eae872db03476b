# Build of the product library (host C + sm_100a CUDA), the test tools and the oracle.
NVCC ?= /usr/local/cuda/bin/nvcc
CC ?= gcc
CSRC := edge264_b200/csrc
NVFLAGS := -gencode arch=compute_100a,code=sm_100a -lineinfo -O3 -std=c++17 -Xcompiler -fPIC -Xcompiler -Wno-unused-function
CFLAGS := -std=gnu11 -O3 -march=x86-64-v3 -fPIC -Wall -Wno-unused-function -Wno-unused-variable -Wno-unused-but-set-variable
LIB := edge264_b200/libedge264_b200.so

all: $(LIB) tools/gen264 tools/b200_decode tools/libe264bench.so oracle

$(CSRC)/recon.o: $(CSRC)/recon.cu $(wildcard $(CSRC)/*.cuh) $(wildcard $(CSRC)/*.h) include/e264b_recon.h
	$(NVCC) $(NVFLAGS) -Xptxas -v -c $< -o $@ 2> $(CSRC)/recon.ptxas.log || (cat $(CSRC)/recon.ptxas.log; false)
$(CSRC)/decoder.o: $(CSRC)/decoder.c $(wildcard $(CSRC)/*.h)
	$(CC) $(CFLAGS) -c $< -o $@
$(CSRC)/slice_dec.o: $(CSRC)/slice_dec.c $(wildcard $(CSRC)/*.h)
	$(CC) $(CFLAGS) -c $< -o $@
$(LIB): $(CSRC)/recon.o $(CSRC)/decoder.o $(CSRC)/slice_dec.o
	$(NVCC) -shared -o $@ $^ -cudart shared
# experiment builds of the runtime with other block geometries of the inter kernel (tools/gpu_variants.sh; not part of `all`)
VARIANTS := w4 w8 timing itiming iw4 iw8
variants: $(foreach v,$(VARIANTS),edge264_b200/variants/$(v)/libedge264_b200.so)
edge264_b200/variants/w8/libedge264_b200.so: VFLAGS := -DINTER_WARPS=8
edge264_b200/variants/w4/libedge264_b200.so: VFLAGS := -DINTER_WARPS=4
edge264_b200/variants/timing/libedge264_b200.so: VFLAGS := -DE264_ROWS_TIMING
edge264_b200/variants/itiming/libedge264_b200.so: VFLAGS := -DE264_INTER_TIMING
edge264_b200/variants/iw4/libedge264_b200.so: VFLAGS := -DINTRA_WARPS=4
edge264_b200/variants/iw8/libedge264_b200.so: VFLAGS := -DINTRA_WARPS=8
edge264_b200/variants/%/libedge264_b200.so: $(CSRC)/recon.cu $(wildcard $(CSRC)/*.cuh) $(wildcard $(CSRC)/*.h) $(CSRC)/decoder.o $(CSRC)/slice_dec.o
	mkdir -p $(dir $@)
	$(NVCC) $(NVFLAGS) $(VFLAGS) -c $(CSRC)/recon.cu -o $(dir $@)recon.o
	$(NVCC) -shared -o $@ $(dir $@)recon.o $(CSRC)/decoder.o $(CSRC)/slice_dec.o -cudart shared
tools/gen264: tools/gen264.c $(wildcard $(CSRC)/*.h)
	$(CC) $(CFLAGS) -O2 -o $@ $<
tools/b200_decode: tools/e264_decode.c $(LIB)
	$(CC) -O2 -std=gnu11 -Iinclude $< -o $@ -Wl,-rpath,'$$ORIGIN/../edge264_b200' -Ledge264_b200 -ledge264_b200
tools/libe264bench.so: tools/e264_bench.c $(LIB)
	$(CC) -O2 -std=gnu11 -fPIC -shared -Iinclude $< -o $@ -Wl,-rpath,'$$ORIGIN/../edge264_b200' -Ledge264_b200 -ledge264_b200 -pthread
oracle:
	$(MAKE) -C oracle all
clean:
	rm -f $(CSRC)/*.o $(LIB) tools/gen264 tools/b200_decode tools/libe264bench.so
.PHONY: all oracle clean variants
