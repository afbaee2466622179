# Builds the B200 BGZF codec in-tree (sm_100a only).  `make` = product; `make testlibs` = test infrastructure.
NVCC      ?= nvcc
CC        ?= gcc
CXX       ?= g++
ARCH      := -gencode arch=compute_100a,code=sm_100a
NVFLAGS   := $(ARCH) -O3 -lineinfo -std=c++17 -Xcompiler -fPIC -Xptxas -v $(NVEXTRA)
CFLAGS    := -O2 -Wall -fPIC -std=gnu99
PKG       := 7bgzf_b200
CSRC      := $(PKG)/csrc
HOST      := $(PKG)/host
OBJ       := build/obj

CU_SRCS   := $(CSRC)/bgzf_compress.cu $(CSRC)/bgzf_inflate.cu $(CSRC)/bgzf_ranges.cu $(CSRC)/bgzf_gzip.cu $(CSRC)/b200bgzf_api.cu
CU_OBJS   := $(patsubst $(CSRC)/%.cu,$(OBJ)/%.o,$(CU_SRCS))
HDRS      := $(wildcard $(CSRC)/*.h) include/b200bgzf.h

PERSONAS  := $(PKG)/7migz $(PKG)/7gzip $(PKG)/7gzinga $(PKG)/7dictzip $(PKG)/7razf
all: $(PKG)/lib7bgzf_b200.so $(PKG)/7bgzf.so $(PKG)/7bgzf $(PERSONAS)

$(OBJ)/%.o: $(CSRC)/%.cu $(HDRS)
	@mkdir -p $(OBJ)
	$(NVCC) $(NVFLAGS) -c $< -o $@ 2> $(OBJ)/$*.ptxas.log || (cat $(OBJ)/$*.ptxas.log; false)

$(OBJ)/%.o: $(HOST)/%.c include/b200bgzf.h $(CSRC)/bgzf_gzip_route.h
	@mkdir -p $(OBJ)
	$(CC) $(CFLAGS) -c $< -o $@

# the codec library: kernels + C ABI (+ the BGZF_METHOD parser)
$(PKG)/lib7bgzf_b200.so: $(CU_OBJS) $(OBJ)/method.o $(OBJ)/multi.o $(OBJ)/containers.o
	$(NVCC) $(ARCH) -shared -o $@ $^ -Xlinker --version-script=$(HOST)/exports.map -lpthread

# the LD_PRELOAD object: the same plus htslib's bgzf_compress
$(PKG)/7bgzf.so: $(CU_OBJS) $(OBJ)/method.o $(OBJ)/multi.o $(OBJ)/containers.o $(OBJ)/hook.o
	$(NVCC) $(ARCH) -shared -o $@ $^ -Xlinker --version-script=$(HOST)/exports.map -lpthread

# the applet
$(PKG)/7bgzf: $(OBJ)/applet_7bgzf.o $(OBJ)/applet_containers.o $(PKG)/lib7bgzf_b200.so
	$(CC) -o $@ $(OBJ)/applet_7bgzf.o $(OBJ)/applet_containers.o -L$(PKG) -l7bgzf_b200 -lpthread -Wl,-rpath,'$$ORIGIN'

# the same applet under its other names (the reference is a multi-call binary too: cielbox.c:215-223)
$(PERSONAS): $(PKG)/7bgzf
	ln -sf 7bgzf $@

# the same library with the bounds asserts compiled in (BG_ASSERT, csrc/bgzf_block.h): point the GPU tests at it with
#   B200BGZF_LIB_PATH=build/checked/lib7bgzf_b200.so python -m pytest tests -m gpu
checked: build/checked/lib7bgzf_b200.so
build/checked/lib7bgzf_b200.so: $(CU_SRCS) $(HDRS) $(OBJ)/method.o $(OBJ)/multi.o $(OBJ)/containers.o
	@mkdir -p build/checked
	$(NVCC) $(ARCH) -O3 -lineinfo -std=c++17 -Xcompiler -fPIC -DBG_CHECK -shared -o $@ $(CU_SRCS) $(OBJ)/method.o $(OBJ)/multi.o $(OBJ)/containers.o -Xlinker --version-script=$(HOST)/exports.map -lpthread

# ---- test / bench infrastructure (never linked into the product) ----
testlibs: build/libdatagen.so build/libemul.so build/datagen build/hook_mt oracle/liboracle.so

build/libdatagen.so: tools/datagen.c
	@mkdir -p build
	$(CC) -O2 -fPIC -shared -o $@ $<
build/datagen: tools/datagen.c
	$(CC) -O2 -DDATAGEN_MAIN -o $@ $<
build/hook_mt: tools/hook_mt.c
	@mkdir -p build
	$(CC) -O2 -o $@ $< -ldl -lpthread
build/libemul.so: tests/model/emul.cpp $(CSRC)/bgzf_block.h $(CSRC)/bgzf_tables.h
	@mkdir -p build
	$(CXX) -O2 -fPIC -shared -o $@ tests/model/emul.cpp
oracle/liboracle.so: $(wildcard oracle/*.c)
	$(CC) -O2 -fPIC -shared -pthread -o $@ $(wildcard oracle/*.c) -ldl

clean:
	rm -rf build $(PKG)/*.so $(PKG)/7bgzf $(PERSONAS) oracle/liboracle.so

.PHONY: all testlibs clean checked
