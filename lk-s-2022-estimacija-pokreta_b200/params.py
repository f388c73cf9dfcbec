"""Parameters of the discrete-optical-flow hot path.

Defaults are the constants hard-coded in the reference scripts
(`daisy i flann.py`:34-48, 88, 167-172, 207-208; `python bcd.py`:21-35, 48; README.md:65).
The reference fixes K = 150 (25 cells x 5 NN + <= 25 random); BASELINE.json's "K=300" / "K=500"
configurations are mapped here (`for_k`) as SURVEY.md section 8 suggests: the number of exact nearest
neighbours per cell and the number of Gaussian-sampled neighbour proposals grow, nothing else.
"""
from dataclasses import dataclass, replace


DEFAULT_KNN_MODE = 1          # FLOWB200_KNN_TCGEN05 (0 = float64 CUDA-core brute force)


@dataclass(frozen=True)
class FlowParams:
    H: int = 375                 # pich   (daisy i flann.py:35)
    W: int = 1241                # picw   (daisy i flann.py:34)
    cellw: int = 73              # :42
    cellh: int = 25              # :43
    cell_radius: int = 2         # cells searched on each side (:167-168)
    k_cell: int = 5              # neighbours per cell (:171-172)
    n_gauss: int = 25            # ngauss (:207)
    sigma: float = 8.0           # :208
    maxnprop: int = 150          # :88
    tphi: float = 2.5            # :46
    tpsi: int = 8                # :47
    lamda: float = 0.05          # :48
    con_tresh: float = 10.0      # README.md:65
    cost_shift: int = 12         # S: int32 BCD works in units of 2^-S (costs quantised to 20*m/2^S)
    knn_mode: int = 0            # FLOWB200_KNN_* (0 = float64 CUDA cores, 1 = tcgen05 prefilter + exact re-rank)
    cell_x0: int = 0             # target cell columns searched: [cell_x0, cell_x1); 0, 0 = all (huge.py: a rank's band)
    cell_x1: int = 0
    flow_refine: int = 0         # flow_pair's fields: 0 = integer vectors, 1 = sub-pixel (flowb200_flow_subpixel)

    @property
    def ncellx(self):
        return self.W // self.cellw

    @property
    def ncelly(self):
        return self.H // self.cellh

    @property
    def n_cells(self):
        return self.ncellx * self.ncelly

    @property
    def cell_size(self):
        return self.cellw * self.cellh

    @property
    def max_nn(self):
        r = 2 * self.cell_radius + 1
        return r * r * self.k_cell

    def with_shape(self, H, W):
        return replace(self, H=int(H), W=int(W))

    def validate(self):
        if self.ncellx < 1 or self.ncelly < 1:
            raise ValueError("image smaller than one cell")
        if self.max_nn + self.n_gauss > self.maxnprop:
            raise ValueError("maxnprop too small for k_cell/cell_radius/n_gauss")
        if self.k_cell > self.cell_size:
            raise ValueError("k_cell larger than a cell")
        if self.maxnprop > 512:
            raise ValueError("maxnprop > 512 not supported")
        if (self.cell_x0, self.cell_x1) != (0, 0) and not 0 <= self.cell_x0 < self.cell_x1 <= self.ncellx:
            raise ValueError("cell_x0 / cell_x1 must select a non-empty range of cell columns")
        if self.flow_refine not in (0, 1):
            raise ValueError("flow_refine must be 0 (integer vectors) or 1 (sub-pixel)")
        return self


def for_k(K, **kw):
    """Map a proposal budget K to (k_cell, n_gauss, maxnprop).

    150 -> reference (5/cell + 25 random); 300 -> 10/cell + 50 random;
    500 -> 12/cell (300 NN) + 200 random (the split of Menze et al., GCPR 2015)."""
    table = {150: (5, 25), 300: (10, 50), 500: (12, 200)}
    if K not in table:
        raise ValueError(f"no mapping for K={K}; known: {sorted(table)}")
    k_cell, n_gauss = table[K]
    return FlowParams(k_cell=k_cell, n_gauss=n_gauss, maxnprop=K, **kw)
