# Builds gp_emulator_b200/libgpemu.so (sm_100a only) in-tree.  `make -j` compiles one object per padded input
# dimension in parallel.  The oracle is pure numpy, so there is nothing to compile under oracle/.
NVCC      ?= nvcc
ARCH      := -gencode arch=compute_100a,code=sm_100a
NVFLAGS   := $(ARCH) -O3 -std=c++17 -lineinfo -Xcompiler -fPIC -Xcompiler -Wall -Iinclude
CSRC      := gp_emulator_b200/csrc
BUILD     := build/obj
DPS       := 2 4 6 8 10 12 16 24 32
LIB       := gp_emulator_b200/libgpemu.so

OBJS := $(BUILD)/gpemu.o $(BUILD)/project.o $(BUILD)/invert.o $(BUILD)/search.o $(BUILD)/peaks.o $(BUILD)/var_large.o $(BUILD)/tf32.o $(BUILD)/train.o $(foreach d,$(DPS),$(BUILD)/inst_dp$(d).o)
HDRS := $(wildcard $(CSRC)/*.cuh) $(wildcard $(CSRC)/*.h) include/gpemu.h

all: $(LIB)

$(BUILD):
	mkdir -p $(BUILD)

$(BUILD)/gpemu.o: $(CSRC)/gpemu.cu $(HDRS) | $(BUILD)
	$(NVCC) $(NVFLAGS) -c $< -o $@

$(BUILD)/peaks.o: $(CSRC)/peaks.cu $(HDRS) | $(BUILD)
	$(NVCC) $(NVFLAGS) -c $< -o $@

$(BUILD)/project.o: $(CSRC)/project.cu $(HDRS) | $(BUILD)
	$(NVCC) $(NVFLAGS) -Xptxas -v -c $< -o $@ 2> $(BUILD)/project.ptxas.log || (cat $(BUILD)/project.ptxas.log; exit 1)

$(BUILD)/invert.o: $(CSRC)/invert.cu $(HDRS) | $(BUILD)
	$(NVCC) $(NVFLAGS) -Xptxas -v -c $< -o $@ 2> $(BUILD)/invert.ptxas.log || (cat $(BUILD)/invert.ptxas.log; exit 1)

$(BUILD)/search.o: $(CSRC)/search.cu $(HDRS) | $(BUILD)
	$(NVCC) $(NVFLAGS) -Xptxas -v -c $< -o $@ 2> $(BUILD)/search.ptxas.log || (cat $(BUILD)/search.ptxas.log; exit 1)

$(BUILD)/var_large.o: $(CSRC)/predict_var_large.cu $(HDRS) | $(BUILD)
	$(NVCC) $(NVFLAGS) -Xptxas -v -c $< -o $@ 2> $(BUILD)/var_large.ptxas.log || (cat $(BUILD)/var_large.ptxas.log; exit 1)

$(BUILD)/train.o: $(CSRC)/train.cu $(HDRS) | $(BUILD)
	$(NVCC) $(NVFLAGS) -Xptxas -v -c $< -o $@ 2> $(BUILD)/train.ptxas.log || (cat $(BUILD)/train.ptxas.log; exit 1)

$(BUILD)/tf32.o: $(CSRC)/predict_tf32_inst.cu $(HDRS) | $(BUILD)
	$(NVCC) $(NVFLAGS) -Xptxas -v -c $< -o $@ 2> $(BUILD)/tf32.ptxas.log || (cat $(BUILD)/tf32.ptxas.log; exit 1)

$(BUILD)/inst_dp%.o: $(CSRC)/predict_full_inst.cu $(HDRS) | $(BUILD)
	$(NVCC) $(NVFLAGS) -Xptxas -v -DGPE_DP=$* -c $< -o $@ 2> $(BUILD)/inst_dp$*.ptxas.log || (cat $(BUILD)/inst_dp$*.ptxas.log; exit 1)

$(LIB): $(OBJS)
	$(NVCC) $(ARCH) -shared -o $@ $(OBJS) -lcudart -ldl

build/fp64_peaks: $(CSRC)/peaks.cu $(HDRS)
	mkdir -p build
	$(NVCC) $(NVFLAGS) -DGPE_PEAKS_MAIN -o $@ $<

clean:
	rm -rf build/obj $(LIB)

.PHONY: all clean
