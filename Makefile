# Builds libasep.so (sm_100a only) and the oracle's compiled helpers in-tree.
NVCC      ?= /usr/local/cuda/bin/nvcc
ARCH      := -gencode arch=compute_100a,code=sm_100a
NVCCFLAGS := -O3 -std=c++17 -lineinfo $(ARCH) -Xcompiler -fPIC -Xcompiler -Wall -Iinclude --expt-relaxed-constexpr
CSRC      := audiosourcesep_b200/csrc
SRCS      := $(CSRC)/api.cu $(CSRC)/flow_kernels.cu $(CSRC)/langevin.cu $(CSRC)/nn_fp32.cu $(CSRC)/nn_tc.cu $(CSRC)/nn_tcx.cu $(CSRC)/glow_model.cu $(CSRC)/conv_tc.cu $(CSRC)/ncsn_kernels.cu $(CSRC)/ncsn_model.cu $(CSRC)/train_kernels.cu $(CSRC)/glow_train.cu $(CSRC)/wgrad_tc.cu $(CSRC)/ncsn_train_kernels.cu $(CSRC)/conv_wgrad_tc.cu $(CSRC)/ncsn_train.cu $(CSRC)/bsseval.cu $(CSRC)/mel_kernels.cu $(CSRC)/resample_kernels.cu $(CSRC)/mwf_kernels.cu
OBJS      := $(SRCS:.cu=.o)
LIB       := audiosourcesep_b200/libasep.so

all: $(LIB)

# k_mwf needs every product rounded before it is added (see the head of mwf_kernels.cu)
$(CSRC)/mwf_kernels.o: NVCCFLAGS += -fmad=false

$(CSRC)/%.o: $(CSRC)/%.cu $(wildcard $(CSRC)/*.h) $(wildcard $(CSRC)/*.cuh) include/asep.h include/asep_dlpack.h
	$(NVCC) $(NVCCFLAGS) -Xptxas -v -c $< -o $@ 2> $@.ptxas.log || (cat $@.ptxas.log; exit 1)

$(LIB): $(OBJS)
	$(NVCC) -shared $(ARCH) -o $@ $(OBJS) -lcudart

clean:
	rm -f $(OBJS) $(LIB) $(CSRC)/*.ptxas.log

.PHONY: all clean
