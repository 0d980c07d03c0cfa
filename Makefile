# Build of the B200-native KOMB hot path (sm_100a only).
#   make            -> komb_b200/libkombgpu.so  (CUDA kernels + C ABI), bin/komb2 (drop-in host)
#   make oracle     -> oracle/libkomb_oracle.so (+ oracle/_ref when /root/reference exists): checkers only
NVCC      := nvcc
CXX       := g++
ARCH      := -gencode arch=compute_100a,code=sm_100a
NVCCFLAGS := -O3 -std=c++17 -lineinfo $(ARCH) -Xcompiler -fPIC,-Wall,-Wno-unused-function -Iinclude -Ikomb_b200/csrc
CSRC      := komb_b200/csrc
OBJDIR    := build/obj
CU        := $(CSRC)/capi.cu $(CSRC)/build.cu $(CSRC)/sort.cu $(CSRC)/peel.cu $(CSRC)/corea.cu $(CSRC)/dist.cu $(CSRC)/densest.cu $(CSRC)/comm.cu $(CSRC)/pbuild.cu $(CSRC)/ppeel.cu $(CSRC)/apeel.cu $(CSRC)/rpeel.cu $(CSRC)/pcore.cu $(CSRC)/pcapi.cu $(CSRC)/truss.cu $(CSRC)/sam.cu $(CSRC)/format.cu $(CSRC)/fasta.cu $(CSRC)/psam.cu $(CSRC)/pfasta.cu
OBJ       := $(patsubst $(CSRC)/%.cu,$(OBJDIR)/%.o,$(CU))
HDR       := include/kombgpu.h $(wildcard $(CSRC)/*.cuh)

all: komb_b200/libkombgpu.so bin/komb2 bin/komb2_tokenize

$(OBJDIR)/%.o: $(CSRC)/%.cu $(HDR)
	@mkdir -p $(OBJDIR)
	$(NVCC) $(NVCCFLAGS) $(PTXAS_V) -c $< -o $@

komb_b200/libkombgpu.so: $(OBJ)
	$(NVCC) $(ARCH) -shared -o $@ $(OBJ) -cudart static

bin/komb2: host/komb2.cpp host/kgraph.hpp host/sam_tokenizer.hpp host/cli.hpp include/kombgpu.h komb_b200/libkombgpu.so
	@mkdir -p bin
	$(CXX) -O2 -std=c++17 -fopenmp -Wall -Iinclude -Ihost host/komb2.cpp -o $@ -Lkomb_b200 -lkombgpu -Wl,-rpath,'$$ORIGIN/../komb_b200'

bin/komb2_tokenize: host/tokenize_main.cpp host/sam_tokenizer.hpp
	@mkdir -p bin
	$(CXX) -O2 -std=c++17 -fopenmp -Wall -Ihost host/tokenize_main.cpp -o $@

oracle:
	$(MAKE) -C oracle all
	@if [ -f /root/reference/src/graph.cpp ]; then $(MAKE) -C oracle ref; fi

clean:
	rm -rf build komb_b200/libkombgpu.so bin

.PHONY: all oracle clean
