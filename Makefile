# Build of the product library and the tools around it.
#
#   make lib      -> sunvolumerender_b200/libsvr_b200.so   (hand-written CUDA, sm_100a only)
#   make oracle   -> oracle/libsvr_oracle.so + oracle/_ref/*.so   (checkers; see oracle/Makefile)
#   make tools    -> tools/svr_headless                     (headless C++ driver)
#   make all
#
# -use_fast_math puts logf/expf/powf/sinf/cosf, division and FTZ in the same arithmetic class as
# the reference build (CMakeLists.txt:9).  No -maxrregcount: the reference's cap of 32 spills.

NVCC     ?= /usr/local/cuda/bin/nvcc
HOSTCXX  ?= /usr/bin/g++
ARCH     := -gencode arch=compute_100a,code=sm_100a
NVFLAGS  := -std=c++17 -O3 -use_fast_math -lineinfo $(ARCH) -Xcompiler -fPIC -Xptxas -v -cudart shared
CSRC     := sunvolumerender_b200/csrc
OBJDIR   := build/obj
SRCS     := $(CSRC)/svr_api.cu $(CSRC)/svr_macrocell.cu $(CSRC)/svr_raycast.cu $(CSRC)/svr_pathtrace.cu $(CSRC)/svr_volume_io.cu $(CSRC)/svr_tf_io.cu $(CSRC)/svr_env_io.cu $(CSRC)/svr_canvas.cu $(CSRC)/svr_denoise.cu $(CSRC)/svr_project.cu
OBJS     := $(patsubst $(CSRC)/%.cu,$(OBJDIR)/%.o,$(SRCS))
HDRS     := $(wildcard $(CSRC)/*.cuh $(CSRC)/*.h include/*.h)
LIB      := sunvolumerender_b200/libsvr_b200.so

.PHONY: all lib oracle tools clean
all: lib oracle tools

lib: $(LIB)

$(OBJDIR)/%.o: $(CSRC)/%.cu $(HDRS)
	@mkdir -p $(OBJDIR)
	$(NVCC) $(NVFLAGS) -c $< -o $@ 2> $(OBJDIR)/$*.ptxas.log || (cat $(OBJDIR)/$*.ptxas.log; exit 1)

$(LIB): $(OBJS)
	$(NVCC) $(ARCH) -shared -cudart shared -o $@ $(OBJS) -lz

oracle:
	$(MAKE) -C oracle all

tools: tools/svr_headless

tools/svr_headless: tools/svr_headless.cpp $(LIB) include/svr_canvas.h include/svr_render.h include/svr_types.h include/svr_volume_io.h include/svr_tf_io.h
	$(HOSTCXX) -O2 -std=c++17 -Iinclude -I/usr/local/cuda/include tools/svr_headless.cpp -o $@ \
	    -Lsunvolumerender_b200 -lsvr_b200 -L/usr/local/cuda/lib64 -lcudart -ldl \
	    -Wl,-rpath,'$$ORIGIN/../sunvolumerender_b200' -Wl,-rpath,/usr/local/cuda/lib64

clean:
	rm -rf build $(LIB) tools/svr_headless
	$(MAKE) -C oracle clean
