"""`Board`: the host-side position value type with the reference's surface (oinkoink/board.py:35-243), and
`BoardBatch`: the same operations batched on the GPU through the C ABI (c4_board_* in include/c4b200.h).

`Board` is deliberately a small host object -- it is what players, games and evaluators pass around, exactly as in
the reference.  Everything hot (search, self-play, network) takes bitboards from it and runs on the device.
Bit layout (board.py:23-30): bit 7*c + h, column c, height h from the bottom; bit 7*c + 6 is the column sentinel.
"""
from copy import deepcopy

import numpy as np

from .utils import Connect4Stats as info
from .utils import Result, Side

WIDTH = info.width
HEIGHT = info.height
H1 = HEIGHT + 1
H2 = HEIGHT + 2
SIZE = HEIGHT * WIDTH
SIZE1 = H1 * WIDTH
ALL1 = (1 << SIZE1) - 1
COL1 = (1 << H1) - 1
BOTTOM = ALL1 // COL1
TOP = BOTTOM << HEIGHT
HALF = WIDTH // 2
SHIFT = (WIDTH - 1) * H1

_BIT = np.array([[H1 * c + (HEIGHT - 1 - r) for c in range(WIDTH)] for r in range(HEIGHT)])  # plane (r,c) -> bit


def _has_four(b: int) -> bool:
    """Board._check_terminal_position (board.py:173-184)"""
    for s in (HEIGHT, H1, H2, 1):
        y = b & (b >> s)
        if y & (y >> (2 * s)):
            return True
    return False


def _mirror(p: int) -> int:
    """Board.flip_color (board.py:127-145)"""
    r = 0
    for c in range(WIDTH):
        r |= ((p >> (H1 * c)) & COL1) << (H1 * (WIDTH - 1 - c))
    return r


def _planes(p: int):
    return ((int(p) >> _BIT) & 1).astype(np.bool_)


class Board():
    def __init__(self):
        self.color = np.zeros((2,), dtype=np.int64)
        self.age = 0
        self.height = np.array([H1 * i for i in range(WIDTH)], dtype=np.int64)
        self.result = None

    @classmethod
    def from_pieces(cls, o_pieces, x_pieces):
        """board.py:43-62: 6x7 bool planes (row 0 = top) -> board; result: o-win, then x-win, then full board."""
        o = np.asarray(o_pieces).astype(bool)
        x = np.asarray(x_pieces).astype(bool)
        b = cls()
        b.color[0] = sum(1 << int(v) for v in _BIT[o])
        b.color[1] = sum(1 << int(v) for v in _BIT[x])
        return b._derive()

    @classmethod
    def from_bitboards(cls, c0, c1):
        """Position from the two colour bitboards (heights, age and result derived as in from_pieces)."""
        b = cls()
        b.color[0] = int(c0)
        b.color[1] = int(c1)
        return b._derive()

    def _derive(self):
        occ = int(self.color[0]) | int(self.color[1])
        self.age = bin(occ).count("1")
        for i in range(WIDTH):
            self.height[i] = H1 * i + bin((occ >> (H1 * i)) & COL1).count("1")
        if _has_four(int(self.color[0])):
            self.result = Result.o_win
        elif _has_four(int(self.color[1])):
            self.result = Result.x_win
        elif self.age == SIZE:
            self.result = Result.draw
        else:
            self.result = None
        return self

    @property
    def o_pieces(self):
        return _planes(self.color[0])

    @property
    def x_pieces(self):
        return _planes(self.color[1])

    @property
    def pieces(self):
        return self.o_pieces, self.x_pieces

    @property
    def player_to_move(self):
        return Side(self.age % 2)

    @property
    def valid_moves(self):
        if self.result is not None:
            return set()
        return set(i for i in range(WIDTH) if self._isplayable(i))

    @property
    def symmetrical(self):
        return self.is_symmetrical(self.color[0]) and self.is_symmetrical(self.color[1])

    def is_symmetrical(self, pieces):
        return _mirror(int(pieces)) == int(pieces)

    def create_fliplr(self):
        new_board = self.__class__()
        new_board.color[0] = self.flip_color(self.color[0])
        new_board.color[1] = self.flip_color(self.color[1])
        new_board.age = self.age
        base = np.array([H1 * i for i in range(WIDTH)], dtype=np.int64)
        new_board.height = base + np.flip(self.height - base)
        new_board.result = deepcopy(self.result)
        return new_board

    def flip_color(self, pieces):
        return _mirror(int(pieces))

    def to_array(self):
        """board.py:147-154: [3,6,7] uint8; ch0 = ones iff o to move, ch1 = o stones, ch2 = x stones."""
        o, x = self.pieces
        to_move = np.ones(o.shape, dtype=np.uint8) if self.age % 2 == 0 else np.zeros(o.shape, dtype=np.uint8)
        return np.stack([to_move, o, x])

    def to_int_tuple(self):
        return self.color[0], self.color[1]

    def make_move(self, move):
        """board.py:160-170 (no legality check, like the reference)"""
        me = self.age & 1
        self.color[me] = int(self.color[me]) ^ (1 << int(self.height[move]))
        self.height[move] = self.height[move] + 1
        winner = _has_four(int(self.color[me]))
        self.age += 1
        if winner:
            self.result = Result(self.age % 2)
        elif self.age == SIZE:
            self.result = Result.draw
        return self.result

    def _check_terminal_position(self, newboard):
        return _has_four(int(newboard))

    def _isplayable(self, col):
        return (int(self.color[self.age & 1]) | (1 << int(self.height[col]))) & TOP == 0

    def __copy__(self):
        b = self.__class__()
        b.color = self.color.copy()
        b.age = self.age
        b.height = self.height.copy()
        b.result = self.result
        return b

    def __eq__(self, obj):
        return isinstance(obj, Board) and np.array_equal(obj.color, self.color)

    def __hash__(self):
        return hash((int(self.color[0]), int(self.color[1])))

    def __str__(self):
        o, x = self.pieces
        rows = []
        for r in range(HEIGHT):
            rows.append(" ".join('o' if o[r, c] else ('x' if x[r, c] else '-') for c in range(WIDTH)))
        header = " ".join(str(c) for c in range(WIDTH))
        return header + "\n" + "\n".join(rows) + "\n" + header

    def __repr__(self):
        return "color: {}, age: {}, height: {}, result: {}\n{}".format(
            self.color, self.age, self.height, self.result, self.__str__())


def make_random_ips(plies):
    """board.py:225-243: the set of all distinct non-terminal positions after `plies` plies."""
    ips = set()
    expand(ips, Board(), plies)
    return ips


def expand(ips, board, plies):
    if plies == 0:
        if board.result is None:
            ips.add(board)
        return
    for move in board.valid_moves:
        nb = board.__copy__()
        nb.make_move(move)
        expand(ips, nb, plies - 1)


# element types of c4_board_to_planes (include/c4b200.h)
PLANE_DTYPES = {"uint8": 0, "float32": 1, "float16": 2, "bfloat16": 3}


class BoardBatch():
    """n positions as two uint64 CUDA tensors (viewed through int64 storage); batched bitboard engine on the GPU."""

    def __init__(self, c0, c1):
        import torch
        from . import _lib
        _lib.require_gpu()
        self.c0 = torch.as_tensor(np.asarray(c0, dtype=np.uint64).view(np.int64)).cuda() if not torch.is_tensor(c0) else c0
        self.c1 = torch.as_tensor(np.asarray(c1, dtype=np.uint64).view(np.int64)).cuda() if not torch.is_tensor(c1) else c1
        self.n = int(self.c0.numel())

    @classmethod
    def from_boards(cls, boards):
        return cls(np.array([int(b.color[0]) for b in boards], dtype=np.uint64),
                   np.array([int(b.color[1]) for b in boards], dtype=np.uint64))

    def _call(self, name, *args):
        from . import _lib
        _lib.check(getattr(_lib.load(), name)(*args, _lib.stream_ptr()))

    def result(self):
        import torch
        from ._lib import ptr
        out = torch.empty(self.n, dtype=torch.int8, device="cuda")
        self._call("c4_board_result", ptr(self.c0), ptr(self.c1), ptr(out), self.n)
        return out

    def legal_mask(self, result=None):
        import torch
        from ._lib import ptr
        out = torch.empty(self.n, dtype=torch.uint8, device="cuda")
        self._call("c4_board_legal_mask", ptr(self.c0), ptr(self.c1), ptr(result), ptr(out), self.n)
        return out

    def drop(self, moves):
        """in place; returns the new result codes"""
        import torch
        from ._lib import ptr
        mv = torch.as_tensor(moves, dtype=torch.int8).cuda()
        out = torch.empty(self.n, dtype=torch.int8, device="cuda")
        self._call("c4_board_drop", ptr(self.c0), ptr(self.c1), ptr(mv), ptr(out), self.n)
        return out

    def has_win(self, which):
        import torch
        from ._lib import ptr
        out = torch.empty(self.n, dtype=torch.uint8, device="cuda")
        self._call("c4_board_has_win", ptr(self.c1 if which else self.c0), ptr(out), self.n)
        return out

    def fliplr(self):
        import torch
        from ._lib import ptr
        f0 = torch.empty_like(self.c0)
        f1 = torch.empty_like(self.c1)
        self._call("c4_board_fliplr", ptr(self.c0), ptr(self.c1), ptr(f0), ptr(f1), self.n)
        return BoardBatch(f0, f1)

    def to_planes(self, dtype="uint8"):
        """Board.to_array of every position: [n, 3, 6, 7] in "uint8", "float32", "float16" or "bfloat16" """
        import torch
        from ._lib import ptr
        code = PLANE_DTYPES.get(dtype, 1)                  # (any other name: float32)
        td = (torch.uint8, torch.float32, torch.float16, torch.bfloat16)[code]
        out = torch.empty((self.n, 3, 6, 7), dtype=td, device="cuda")
        self._call("c4_board_to_planes", ptr(self.c0), ptr(self.c1), ptr(out), code, self.n)
        return out

    @classmethod
    def from_planes(cls, o, x):
        import torch
        from . import _lib
        from ._lib import ptr
        _lib.require_gpu()
        o = torch.as_tensor(o, dtype=torch.uint8).cuda().contiguous()
        x = torch.as_tensor(x, dtype=torch.uint8).cuda().contiguous()
        n = o.shape[0]
        c0 = torch.empty(n, dtype=torch.int64, device="cuda")
        c1 = torch.empty(n, dtype=torch.int64, device="cuda")
        _lib.check(_lib.load().c4_board_from_planes(ptr(o), ptr(x), ptr(c0), ptr(c1), n, _lib.stream_ptr()))
        return cls(c0, c1)

    def evaluate_centre(self):
        import torch
        from ._lib import ptr
        out = torch.empty(self.n, dtype=torch.float64, device="cuda")
        self._call("c4_board_evaluate_centre", ptr(self.c0), ptr(self.c1), ptr(out), self.n)
        return out

    def numpy(self):
        return (self.c0.cpu().numpy().view(np.uint64), self.c1.cpu().numpy().view(np.uint64))
