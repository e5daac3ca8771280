# Builds bbs_sign_b200/libbbs_b200.so: hand-written CUDA for sm_100a behind the C ABI of include/bbs_b200.h.
# One object per (kernel group, curve) so `make -j` compiles them in parallel.
NVCC      ?= nvcc
ARCH      := -gencode arch=compute_100a,code=sm_100a
NVCCFLAGS := $(ARCH) -O3 -std=c++17 -lineinfo -Xcompiler -fPIC $(EXTRA_NVCCFLAGS)
SRC       := bbs_sign_b200/csrc
BUILD     ?= build/obj
OUT       ?= bbs_sign_b200/libbbs_b200.so
GROUPS    := ctx h2s verify pairing sign signitem proof proofitem rlc selftest
HDRS      := $(wildcard $(SRC)/*.cuh) $(wildcard $(SRC)/*.inc) include/bbs_b200.h
OBJS      := $(BUILD)/capi.o $(foreach g,$(GROUPS),$(BUILD)/tu_$(g)_bls.o $(BUILD)/tu_$(g)_bn.o)

all: $(OUT)

$(BUILD)/capi.o: $(SRC)/capi.cu $(HDRS)
	@mkdir -p $(BUILD)
	$(NVCC) $(NVCCFLAGS) -c -o $@ $<

$(BUILD)/tu_%_bls.o: $(SRC)/tu_%.cu $(HDRS)
	@mkdir -p $(BUILD)
	$(NVCC) $(NVCCFLAGS) -DBBS_TU_BLS -Xptxas -v -c -o $@ $< 2> $(BUILD)/tu_$*_bls.ptxas.log || (cat $(BUILD)/tu_$*_bls.ptxas.log; false)

$(BUILD)/tu_%_bn.o: $(SRC)/tu_%.cu $(HDRS)
	@mkdir -p $(BUILD)
	$(NVCC) $(NVCCFLAGS) -DBBS_TU_BN -Xptxas -v -c -o $@ $< 2> $(BUILD)/tu_$*_bn.ptxas.log || (cat $(BUILD)/tu_$*_bn.ptxas.log; false)

$(OUT): $(OBJS)
	$(NVCC) $(ARCH) -shared -o $@ $(OBJS)

clean:
	rm -rf $(BUILD) $(OUT)

.PHONY: all clean
