# Build of the B200-native Eesen CTC hot path (in-tree; artefacts are git-ignored but travel with gpurun).
#   eesen_b200/lib/libeesen_b200.so   CUDA kernels (sm_100a) + C ABI (include/eesen_b200.h) + C++ host mirror
#   eesen_b200/bin/train-ctc-parallel the training driver (host logic of reference src/netbin/train-ctc-parallel.cc)
#   eesen_b200/bin/net-output-extract the forward-only tool (src/netbin/net-output-extract.cc), batched
#   eesen_b200/bin/format-to-nonparallel  <BiLstmParallel> -> <BiLstm> marker rewrite (src/netbin/format-to-nonparallel.cc)
# `make oracle` builds the CPU checker (test infrastructure, oracle/).
CUDA    ?= /usr/local/cuda
NVCC    := $(CUDA)/bin/nvcc
CXX     := g++
ARCH    := -gencode arch=compute_100a,code=sm_100a
NVFLAGS := $(ARCH) -lineinfo -O3 -std=c++17 -Xcompiler -fPIC -Xcompiler -Wall $(if $(TIMING),-DEB_LSTM_TIMING,)
CXXFLAGS:= -O2 -std=c++17 -fPIC -Wall -I$(CUDA)/include
OBJDIR  ?= build
LIBDIR  ?= eesen_b200/lib
BINDIR  := eesen_b200/bin

CU_SRCS := gemm gemm_tc lstm lstm_tc ctc ce optim decode
CC_SRCS := base net abi_ops abi_net abi_decode
CU_OBJS := $(patsubst %,$(OBJDIR)/%.cu.o,$(CU_SRCS))
CC_OBJS := $(patsubst %,$(OBJDIR)/%.cc.o,$(CC_SRCS))

BINS    := train-ctc-parallel net-output-extract format-to-nonparallel net-change-model

all: $(LIBDIR)/libeesen_b200.so $(patsubst %,$(BINDIR)/%,$(BINS))

$(OBJDIR)/%.cu.o: eesen_b200/csrc/%.cu eesen_b200/csrc/common.cuh eesen_b200/csrc/kernels.h eesen_b200/csrc/tc_common.cuh
	@mkdir -p $(OBJDIR)
	$(NVCC) $(NVFLAGS) -c $< -o $@

$(OBJDIR)/%.cc.o: eesen_b200/host/%.cc eesen_b200/host/base.h eesen_b200/host/net.h eesen_b200/host/context.h eesen_b200/csrc/kernels.h include/eesen_b200.h
	@mkdir -p $(OBJDIR)
	$(CXX) $(CXXFLAGS) -c $< -o $@

$(LIBDIR)/libeesen_b200.so: $(CU_OBJS) $(CC_OBJS)
	@mkdir -p $(LIBDIR)
	$(NVCC) $(ARCH) -shared -o $@ $^ -cudart shared -ldl

$(BINDIR)/%: eesen_b200/host/%.cc eesen_b200/host/options.h eesen_b200/host/minibatch.h $(LIBDIR)/libeesen_b200.so
	@mkdir -p $(BINDIR)
	$(CXX) $(CXXFLAGS) $< -o $@ -L$(LIBDIR) -leesen_b200 -Wl,-rpath,'$$ORIGIN/../lib' -L$(CUDA)/lib64 -lcudart -Wl,-rpath,$(CUDA)/lib64

oracle:
	$(MAKE) -C oracle all

clean:
	rm -rf $(OBJDIR) $(LIBDIR) $(BINDIR)

.PHONY: all oracle clean
