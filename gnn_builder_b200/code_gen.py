"""``Project`` -- the drop-in seam of ``gnnbuilder/code_gen.py:62-395`` for the GPU backend.

Same constructor arguments, method names and return values, so the call sequence of the
reference's demos (``demos/demo.py:102-129``) works unchanged:

    proj = Project(name, model, "regression", vitis_hls_path, build_dir, dataset=ds,
                   max_nodes=600, max_edges=600, float_or_fixed="float")
    proj.gen_hw_model(); proj.gen_testbench(); proj.gen_makefile()
    data = proj.build_and_run_testbench()   # {"model_output_mae": ..., "model_runtime": ...}

What changes is what happens underneath: instead of rendering HLS C++ and shelling out to
``make`` + ``./result`` (code_gen.py:201-213, 355-381), ``gen_hw_model`` binds the model to a
B200 through the C-ABI handle and ``build_and_run_testbench`` runs every graph of ``tb_data/``
on the GPU, one graph per call with host buffers -- the same region the reference testbench
times (model_tb.cpp.jinja:200-204).  FPGA-only arguments (``vitis_hls_path``, ``fpga_part``,
``clock_speed``, ``*_guess``, ``n_jobs``) are accepted and ignored; the Vitis methods raise.
"""
from __future__ import annotations

import json
import os
import subprocess
import time
from functools import cached_property
from pathlib import Path
from typing import Optional

import numpy as np
import torch

from .data import GraphBatch, read_tb_data, write_tb_data
from .engine import Engine
from .models import GNNModel
from .utils import iter_graphs


class FPX:
    """code_gen.py:39-52 (kept for signature compatibility; fixed-point mode is not offered)"""

    def __init__(self, W: int = 32, I: int = 16, Q: str = "AP_TRN", O: str = "AP_WRAP"):  # noqa: E741
        self.W, self.I, self.Q, self.O = W, I, Q, O
        if I > 33:
            raise Exception("I must be <= 33")
        if W - I > 32:
            raise Exception("W-I must be <= 32")

    def __str__(self):
        return f"ap_fixed<{self.W},{self.I},{self.Q},{self.O}>"


SUPPORTED_FPGA_PARTS = ["xcu50-fsvh2104-2-e", "xcu280-fsvh2892-2L-e"]


class Project:
    def __init__(self, name: str, model: GNNModel, pyg_output_encoding: str,
                 vitis_hls_path: Optional[Path], build_dir: Path, dataset=None,
                 max_nodes: int = 500, max_edges: int = 500,
                 num_nodes_guess: Optional[int] = None, num_edges_guess: Optional[int] = None,
                 degree_guess: Optional[int] = None, float_or_fixed: str = "float",
                 fpx: FPX = FPX(W=32, I=16), clock_speed: float = 3.33,
                 fpga_part: str = "xcu50-fsvh2104-2-e", n_jobs: int = 1,
                 cosim_wave_debug: bool = False, device: int = -1):
        self.model = model
        self.dataset = dataset
        self.name = name
        self.max_nodes = max_nodes
        self.max_edges = max_edges
        self.num_nodes_guess = num_nodes_guess if num_nodes_guess is not None else max_nodes
        self.num_edges_guess = num_edges_guess if num_edges_guess is not None else max_edges
        self.degree_guess = degree_guess if degree_guess is not None else max_nodes
        self.pyg_output_encoding = pyg_output_encoding
        valid = ["regression", "classification_integer", "classification_onehot"]
        if self.pyg_output_encoding not in valid:
            raise ValueError(f"pyg_output_encoding must be one of {valid}")
        self.vitis_hls_path = vitis_hls_path
        self.build_dir = Path(build_dir)
        self.float_or_fixed = float_or_fixed
        self.fpx = fpx
        if float_or_fixed not in ["float", "fixed"]:
            raise ValueError("float_or_fixed must be one of ['float', 'fixed']")
        self.clock_speed = clock_speed
        if self.clock_speed <= 0:
            raise ValueError("clock_speed must be > 0")
        self.fpga_part = fpga_part
        if self.fpga_part not in SUPPORTED_FPGA_PARTS:
            raise ValueError(f"fpga_part must be one of {SUPPORTED_FPGA_PARTS}")
        self.n_jobs = n_jobs
        if self.n_jobs <= 0:
            raise ValueError("n_jobs must be > 0")
        self.cosim_wave_debug = cosim_wave_debug
        self.device = device
        self.engine: Optional[Engine] = None

    def validate_project(self):
        if self.name is None:
            raise Exception("No name is set.")
        if self.dataset is None:
            raise Exception("No dataset is set.")
        if self.model is None:
            raise Exception("No model is set.")

    @cached_property
    def model_dir(self) -> Path:
        return self.build_dir / self.name

    # ------------------------------------------------------------------ generation
    def gen_hw_model(self):
        """Bind the model to the GPU (the analogue of rendering model.h/model.cpp)."""
        self._check_top_renderable("gen_hw_model")
        if self.float_or_fixed == "fixed":
            raise NotImplementedError(
                "ap_fixed mode needs Xilinx's ap_fixed.h/hls_math.h to pin results against; "
                "the B200 backend implements the float model only")
        os.makedirs(self.model_dir, exist_ok=True)
        if self.engine is not None:
            self.engine.close()
        self.engine = Engine(self.model, max_nodes=self.max_nodes, max_edges=self.max_edges,
                             device=self.device)
        manifest = dict(name=self.name, desc=self.model.describe(), max_nodes=self.max_nodes,
                        max_edges=self.max_edges,
                        param_names=self.model.layer_parameter_names_flat,
                        param_shapes=self.model.layer_parameter_shapes_flat)
        (self.model_dir / "model_desc.json").write_text(json.dumps(manifest, indent=1))
        (self.model_dir / "model.cpp").write_text(self.render_top())

    # ------------------------------------------------------------------ the C++ seam
    def render_top(self) -> str:
        """``model.cpp`` for the GPU backend: ``extern "C" void <name>_top(...)`` with EXACTLY the
        reference's signature (model.h.jinja:67-79: feature table, edge list, output, num_of_nodes,
        num_of_edges, copy_parameters_flag, then one ``<param>_fixed_in`` array per parameter in
        ``layer_parameter_names_flat`` order) forwarding to the C-ABI model handle -- what a
        maintainer renders instead of model.cpp.jinja:686-766.  The reference's own ``model.h``
        and ``model_tb.cpp`` compile and link against it unchanged (float build)."""
        self._check_top_renderable("render_top")
        d = self.model.describe()
        names = self.model.layer_parameter_names_flat
        shapes = self.model.layer_parameter_shapes_flat
        f_in, out_dim = d["in_dim"], d["mlp_out"]
        pools = list(d["pools"]) + [0] * (4 - len(d["pools"]))

        def dims(shape):
            return "".join(f"[{int(v)}]" for v in shape)

        def first(name, shape):
            return f"&{name}_fixed_in" + "[0]" * len(shape)

        def numel(shape):
            return int(np.prod(shape)) if len(shape) else 1

        args = "".join(f",\n    float {n}_fixed_in{dims(sh)}" for n, sh in zip(names, shapes))
        sets = "\n".join(
            f'        gnnb_check(gnnb_model_set_param(g_model, "{n}", {first(n, sh)}, {numel(sh)}));'
            for n, sh in zip(names, shapes))
        return f"""// Generated by gnn_builder_b200.Project.gen_hw_model -- do not edit.
// `{self.name}_top` with the reference's signature (gnnbuilder model.h.jinja:67-79), computed on
// the GPU through the C-ABI of libgnnb_b200.so (include/gnnb_b200.h).  Replaces the rendered
// model.cpp (model.cpp.jinja:686-766); model.h and model_tb.cpp of the reference stay as they are.
#include <cstdio>
#include <cstdlib>

#ifdef GNNB_REFERENCE_MODEL_H   // built next to the reference's rendered model.h: the compiler checks
#include "model.h"              // this definition against the reference's own declaration
#endif
#include "gnnb_b200.h"

static gnnb_model_t *g_model = nullptr;   // replaces the file-scope weight arrays (cpp:7-22)

static void gnnb_check(int rc)
{{
    if (rc != GNNB_OK) {{   // the reference's top is void: there is no status to return
        std::fprintf(stderr, "{self.name}_top: %s\\n", gnnb_last_error());
        std::abort();
    }}
}}

extern "C" void {self.name}_top(
    float node_feature_table_input[{self.max_nodes}][{f_in}],
    int edge_list_input[{self.max_edges}][2],
    float model_output[{out_dim}],
    int num_of_nodes,
    int num_of_edges,
    int copy_parameters_flag{args})
{{
    if (copy_parameters_flag) {{   // cpp:724-730: parameters are (re)loaded when the flag is set
        if (g_model == nullptr) {{
            gnnb_model_desc d = {{}};
            d.conv_type = {d["conv_type"]}; d.num_layers = {d["num_layers"]}; d.in_dim = {d["in_dim"]};
            d.hidden_dim = {d["hidden_dim"]}; d.out_dim = {d["out_dim"]}; d.skip = {d["skip"]};
            d.gnn_act = {d["gnn_act"]}; d.gin_eps = {float(d["gin_eps"])!r}f; d.pna_delta = {float(d["pna_delta"])!r}f;
            d.num_pools = {len(d["pools"])};
            d.pools[0] = {pools[0]}; d.pools[1] = {pools[1]}; d.pools[2] = {pools[2]}; d.pools[3] = {pools[3]};
            d.mlp_num_linear = {d["mlp_num_linear"]}; d.mlp_hidden = {d["mlp_hidden"]}; d.mlp_out = {d["mlp_out"]};
            d.mlp_act = {d["mlp_act"]}; d.out_act = {d["out_act"]};
            d.max_nodes = {self.max_nodes}; d.max_edges = {self.max_edges};
            gnnb_check(gnnb_model_create(&d, -1, &g_model));
        }}
{sets}
        gnnb_check(gnnb_model_finalize(g_model));
    }}
    if (g_model == nullptr) {{
        std::fprintf(stderr, "{self.name}_top: called before the parameters were loaded\\n");
        std::abort();
    }}
    gnnb_check(gnnb_model_run_graph(g_model, &node_feature_table_input[0][0], &edge_list_input[0][0],
                                    num_of_nodes, num_of_edges, model_output));
}}
"""

    def _check_top_renderable(self, what):
        if self.model is not None and self.model.describe()["conv_type"] == 5:
            raise NotImplementedError(
                f"{what}: the reference has no GAT kernel and its <name>_top no attention-head "
                "arguments, so a GATConv_GNNB model cannot be rendered; run it through Engine "
                "instead")
        if self.model is not None and self.model.describe()["conv_type"] == 7:
            raise NotImplementedError(
                f"{what}: the reference has no GATv2 kernel and its <name>_top no attention-head "
                "arguments, so a GATv2Conv_GNNB model cannot be rendered; run it through Engine "
                "instead")
        if self.model is not None and self.model.describe()["conv_type"] == 8:
            raise NotImplementedError(
                f"{what}: the reference has no TransformerConv kernel and its <name>_top no "
                "attention-head arguments, so a TransformerConv_GNNB model cannot be rendered; run "
                "it through Engine instead")
        if getattr(self.model, "uses_edge_features", False):
            raise NotImplementedError(
                f"{what}: the reference's <name>_top signature has no edge-feature argument, so a "
                "GINEConv_GNNB model cannot be rendered; run it through Engine instead")

    def build_top(self, testbench: Optional[Path] = None) -> Path:
        """Compile the generated ``model.cpp`` into ``lib<name>.so`` (exports ``<name>_top``).
        With ``testbench`` = a directory holding the REFERENCE's rendered ``model.h``,
        ``gnn_builder_lib.h`` and ``model_tb.cpp`` (what ``gnnbuilder.Project.gen_hw_model /
        gen_testbench`` write), also link the reference's own testbench against this top into
        ``result`` -- flags of makefile_testbench.jinja:22-24."""
        from . import _lib

        _lib.load()  # builds libgnnb_b200.so if it is missing
        src = self.model_dir / "model.cpp"
        if not src.exists():
            raise Exception(f"{self.name} - {src} does not exist. Call gen_hw_model() first.")
        inc = Path(__file__).resolve().parent.parent / "include"
        libdir = Path(_lib.LIB_PATH).parent
        link = [f"-L{libdir}", "-lgnnb_b200", f"-Wl,-rpath,{libdir}"]
        so = self.model_dir / f"lib{self.name}.so"
        base = ["g++", "-O3", "-std=c++14", "-fPIC", f"-I{inc}"]
        cmds = [base + ["-shared", str(src), "-o", str(so)] + link]
        if testbench is not None:
            tb = Path(testbench)
            cmds.append(base + ["-w", "-DGNNB_REFERENCE_MODEL_H", f"-I{tb}", str(tb / "model_tb.cpp"), str(src),
                                "-o", str(self.model_dir / "result")] + link)
        for cmd in cmds:
            r = subprocess.run(cmd, capture_output=True, text=True)
            if r.returncode != 0:
                raise RuntimeError(f"{' '.join(cmd)}\n{r.stdout}\n{r.stderr}")
        return so

    def gen_testbench(self, gen_testbench_data=True):
        os.makedirs(self.model_dir, exist_ok=True)
        if gen_testbench_data:
            self.gen_testbench_data()

    def gen_testbench_data(self):
        """code_gen.py:227-305: params + per-graph inputs + golden outputs of the torch model."""
        self.validate_project()
        graphs, golden, task = [], [], []
        out_dim = self.model.output_features_dim
        with torch.no_grad():
            for x, coo, y in iter_graphs(self.dataset):
                if x.shape[0] > self.max_nodes or coo.shape[0] > self.max_edges:
                    raise ValueError("graph exceeds max_nodes/max_edges")
                graphs.append((x, coo))
                ei = torch.from_numpy(np.ascontiguousarray(coo.T.astype(np.int64)))
                golden.append(self.model(torch.from_numpy(x), ei).view(-1).numpy())
                t = np.zeros(out_dim, np.float32)
                if y is not None:
                    yv = np.asarray(y.detach().cpu().numpy() if hasattr(y, "detach") else y,
                                    np.float32).reshape(-1)
                    if self.pyg_output_encoding == "classification_integer":
                        t[int(yv[0])] = 1.0
                    else:
                        t[: min(out_dim, yv.size)] = yv[:out_dim]
                task.append(t)
        write_tb_data(self.model_dir / "tb_data", self.model.named_parameter_arrays(),
                      GraphBatch.from_graphs(graphs), np.stack(golden), np.stack(task), out_dim)

    def gen_makefile(self):
        os.makedirs(self.model_dir, exist_ok=True)
        inc = Path(__file__).resolve().parent.parent / "include"
        libdir = Path(__file__).resolve().parent
        (self.model_dir / "makefile_testbench").write_text(
            "# gnn_builder_b200: the Python flow needs nothing compiled per model (libgnnb_b200.so takes\n"
            "# the model description at run time, see model_desc.json).  `make lib` builds the generated\n"
            "# model.cpp (<name>_top with the reference's signature, forwarding to the GPU library);\n"
            "# `make result` links the reference's own model_tb.cpp against it when model.h,\n"
            "# gnn_builder_lib.h and model_tb.cpp of the reference are placed next to it.\n"
            f"CXXFLAGS = -fPIC -O3 -std=c++14 -I{inc}\n"
            f"LDLIBS = -L{libdir} -lgnnb_b200 -Wl,-rpath,{libdir}\n"
            "run:\n\t@true\n"
            f"lib: model.cpp\n\t$(CXX) $(CXXFLAGS) -shared model.cpp -o lib{self.name}.so $(LDLIBS)\n"
            "result: model.cpp model_tb.cpp model.h\n"
            "\t$(CXX) $(CXXFLAGS) -Wno-unused-result model.cpp model_tb.cpp -o result $(LDLIBS)\n")

    # ------------------------------------------------------------------ running
    def build_and_run_testbench(self, batched: bool = False):
        """Run every graph of tb_data on the GPU.  Returns the reference's dict
        (code_gen.py:384-395): mean |golden - output| and mean seconds per graph (timed around
        each single-graph call with host buffers, like model_tb.cpp.jinja:200-204).  With
        ``batched=True`` the whole set goes through one batch call instead and
        ``model_runtime`` is total seconds / number of graphs."""
        for fp in (self.model_dir / "model_desc.json", self.model_dir / "makefile_testbench"):
            if not fp.exists():
                raise Exception(f"{self.name} - {fp} does not exist. Make sure you call the"
                                " gen_<...> functions to generate the model and testbench.")
        if self.engine is None:
            self.gen_hw_model()
        tb = self.model_dir / "tb_data"
        _, batch, golden = read_tb_data(tb, self.model.input_node_features_dim)
        self.engine.run_graph(*batch.graph(0))  # warm-up: the reference's untimed parameter load
        if batched:
            t0 = time.perf_counter()
            out = self.engine.run(batch)
            runtime = (time.perf_counter() - t0) / batch.n_graphs
        else:
            out = np.empty((batch.n_graphs, self.model.output_features_dim), np.float32)
            total = 0.0
            for g in range(batch.n_graphs):
                x, coo = batch.graph(g)
                t0 = time.perf_counter()
                out[g] = self.engine.run_graph(x, coo)
                total += time.perf_counter() - t0
            runtime = total / batch.n_graphs
        mae = float(np.abs(golden - out).mean())
        (tb / "model_output_mae.txt").write_text(f"model_output_mae {mae}\n")
        (tb / "model_runtime.txt").write_text(f"model_runtime {runtime}\n")
        return {"model_output_mae": mae, "model_runtime": runtime}

    # ------------------------------------------------------------------ FPGA-only surface
    def _fpga_only(self, what):
        raise NotImplementedError(f"{what} drives the Vitis HLS / FPGA flow, which has no GPU "
                                  "analogue in the B200 backend")

    def gen_vitis_hls_tcl_script(self):
        self._fpga_only("gen_vitis_hls_tcl_script")

    def gen_vitis_hls_cosim_tcl_script(self):
        self._fpga_only("gen_vitis_hls_cosim_tcl_script")

    def run_vitis_hls_synthesis(self, verbose=False):
        self._fpga_only("run_vitis_hls_synthesis")

    def gen_makefile_vitis(self):
        self._fpga_only("gen_makefile_vitis")

    def build_hw_kernel(self):
        self._fpga_only("build_hw_kernel")
