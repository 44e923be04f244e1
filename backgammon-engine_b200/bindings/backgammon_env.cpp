// backgammon_env — the reference's Python module surface (cppsrc/backgammon_bindings.cpp:41-93:
// PlayerType / Player / Pieces / Game, same method names, argument meaning and return types)
// re-hosted on the libbgx C-ABI (include/bgx.h), plus the batched entry points as BatchEngine.
//
// Nothing here implements rules: every Game method forwards to a bgx_* function.  Errors are
// return values, never exceptions, exactly as in the reference (tryMove -> (False, message)).
// Differences kept on purpose (SURVEY.md §5 "latent UB"): Game owns COPIES of the two Players
// (the reference keeps raw pointers without keep_alive), and an unset Player reads as
// ("", PLAYER1 / PLAYER2) instead of dereferencing garbage.
#include <pybind11/numpy.h>
#include <pybind11/pybind11.h>
#include <pybind11/stl.h>

#include <array>
#include <iostream>
#include <random>
#include <stdexcept>
#include <string>
#include <vector>

#include "bgx.h"

namespace py = pybind11;

enum PlayerType { PLAYER1 = 0, PLAYER2 = 1 };   // unscoped like Player::PLAYERS (player.hpp:14-18): int-comparable

class Player {                                    // player.hpp:6-27
  public:
    Player(std::string name, int num) : name_(std::move(name)), num_(num) {}
    std::string getName() const { return name_; }
    int getNum() const { return num_; }

  private:
    std::string name_;
    int num_;
};

class Game;
class Pieces {                                    // Pieces.hpp:5-45, a view on the owning Game's counters
  public:
    explicit Pieces(Game *g) : g_(g) {}
    int numJailed(int player) const;
    int numFreed(int player) const;

  private:
    Game *g_;
};

static std::mt19937_64 &shared_rng()
{
    // one generator per process: clone() no longer seeds a fresh mt19937_64 from random_device
    // (the reference's hot spot, game.hpp:45 / SURVEY.md §0)
    static std::mt19937_64 rng{std::random_device{}()};
    return rng;
}

class Game {
  public:
    explicit Game(int player) : pieces_(this)                           // game.cpp:44-56
    {
        turn_ = (player % 2 == 0) ? PLAYER1 : PLAYER2;
        populateBoard();
    }
    Game(const Game &o) : board_(o.board_), counters_(o.counters_), turn_(o.turn_), dice_(o.dice_), p1_(o.p1_), p2_(o.p2_), pieces_(this) {}
    Game &operator=(const Game &) = delete;

    void populateBoard() { board_ = {2, 0, 0, 0, 0, -5, 0, -3, 0, 0, 0, 5, -5, 0, 0, 0, 3, 0, 5, 0, 0, 0, 0, -2}; }   // game.cpp:251
    void setPlayers(const Player &a, const Player &b) { p1_ = a; p2_ = b; }
    Player getPlayers(int num) const { return num == 0 ? p1_ : p2_; }   // game.cpp:31-42
    int getTurn() const { return turn_; }
    void setTurn(int t) { turn_ = t; }
    std::vector<int> getGameBoard() const { return board_; }
    void setGameBoard(std::vector<int> b) { board_ = std::move(b); }    // no length check, like game.cpp:26-29
    Pieces &getPieces() { return pieces_; }
    int getJailedCount(int player) const { return counters_[player == PLAYER1 ? 0 : 1]; }
    int getBornOffCount(int player) const { return counters_[player == PLAYER1 ? 2 : 3]; }
    void setFreed(int player, int num) { counters_[player == 0 ? 2 : 3] = num; }   // game.cpp:14-24
    void setDice(int a, int b) { dice_ = {a, b}; }
    std::array<int, 2> getLastDice() const { return dice_; }
    std::array<int, 2> rollDice()                                        // game.cpp:665-670
    {
        std::uniform_int_distribution<int> die(1, 6);
        dice_[0] = die(shared_rng());
        dice_[1] = die(shared_rng());
        return dice_;
    }
    Game clone() const                                                   // game.cpp:68-77: dice are NOT copied
    {
        Game c(*this);
        c.dice_ = {1, 1};
        return c;
    }

    std::array<int32_t, 28> row() const
    {
        std::array<int32_t, 28> s{};
        for (size_t i = 0; i < 24 && i < board_.size(); i++) s[i] = board_[i];
        for (int i = 0; i < 4; i++) s[24 + i] = counters_[i];
        return s;
    }
    void take(const std::array<int32_t, 28> &s)
    {
        if (board_.size() < 24) board_.resize(24, 0);
        for (int i = 0; i < 24; i++) board_[i] = s[i];
        for (int i = 0; i < 4; i++) counters_[i] = s[24 + i];
    }

    std::vector<std::pair<int, int>> legalMoves(int player, int die) const   // game.cpp:80-105
    {
        auto s = row();
        int8_t buf[52];
        int n = 0;
        check(bgx_legal_moves(s.data(), player, die, buf, 26, &n));
        std::vector<std::pair<int, int>> out;
        for (int i = 0; i < n; i++) out.emplace_back(buf[2 * i], buf[2 * i + 1]);
        return out;
    }

    struct Eval {
        std::vector<std::vector<std::pair<int, int>>> sequences;
        std::vector<int32_t> states;
        int64_t n = 0;
    };
    Eval evaluate(int player, int d1, int d2, bool want_states) const     // game.cpp:134-222
    {
        auto s = row();
        int64_t cap = 256, n = 0;
        std::vector<int8_t> mv, ln;
        Eval ev;
        for (;;) {
            mv.assign((size_t)cap * 8, 0);
            ln.assign((size_t)cap, 0);
            if (want_states) ev.states.assign((size_t)cap * 28, 0);
            int rc = bgx_turn_sequences(s.data(), player, d1, d2, cap, mv.data(), ln.data(), want_states ? ev.states.data() : nullptr, &n);
            if (rc == BGX_E_CAPACITY) { cap = n; continue; }
            check(rc);
            break;
        }
        ev.n = n;
        ev.sequences.resize((size_t)n);
        for (int64_t i = 0; i < n; i++)
            for (int j = 0; j < ln[i]; j++) ev.sequences[i].emplace_back(mv[8 * i + 2 * j], mv[8 * i + 2 * j + 1]);
        return ev;
    }

    std::pair<bool, std::string> tryMove(const Player &pl, int dice, int origin, int dest)   // game.cpp:573-663
    {
        auto s = row();
        int code = 0;
        check(bgx_try_move(s.data(), pl.getNum(), dice, origin, dest, &code));
        if (code == BGX_MOVE_OK) take(s);
        return {code == BGX_MOVE_OK, bgx_move_error_string(code)};
    }

    std::pair<bool, int> over() const                                     // game.cpp:388-407
    {
        auto s = row();
        int w = -1;
        check(bgx_game_over(s.data(), &w));
        return {w >= 0, w};
    }

    // the console picture of game.cpp:260-385 (same layout: 12..1 on top, 13..24 below)
    void printGameBoard() const
    {
        std::vector<int> b(24, 0);
        for (size_t i = 0; i < 24 && i < board_.size(); i++) b[i] = board_[i];
        auto &o = std::cout;
        o << "\n" << p1_.getName() << ": " << "◉    |      " << p2_.getName() << ": " << "◯" << std::endl;
        o << "\n\n";
        o << "   12 11 10 9  8  7     6  5  4  3  2  1" << std::endl;
        o << "*-----------------------------------------*" << std::endl;
        for (int line = 0; line < 8; line++) {                // top half grows downwards
            o << "|  ";
            for (int p = 11; p >= 0; p--) {
                if (p == 5) o << "|  ";
                if (line == 0 && b[p] == 0) o << "'";
                else if (b[p] > 0) { o << "◉"; b[p]--; }
                else if (b[p] < 0) { o << "◯"; b[p]++; }
                else o << " ";
                o << "  ";
            }
            o << "|" << std::endl;
        }
        for (int level = 8; level >= 1; level--) {            // bottom half grows upwards
            o << "|  ";
            for (int p = 12; p < 24; p++) {
                if (p == 18) o << "|  ";
                if (std::abs(b[p]) == level) {
                    if (b[p] > 0) { o << "◉"; b[p]--; }
                    else if (b[p] < 0) { o << "◯"; b[p]++; }
                } else {
                    o << (level == 1 ? "'" : " ");
                }
                o << "  ";
            }
            o << "|" << std::endl;
        }
        o << "* ----------------------------------------*" << std::endl;
        o << "  13 14  15 16 17 18 | 19 20  21 22 23 24 " << std::endl;
        o << std::endl;
        o << "         Jail: ◉ x" << counters_[0] << "  |  ◯ x" << counters_[1] << std::endl;
        o << "\n         Free: ◉ x" << counters_[2] << "  |  ◯ x" << counters_[3] << std::endl;
        o << "\n\n" << std::endl;
    }

    static void check(int rc)
    {
        if (rc != BGX_OK) throw std::runtime_error(std::string("libbgx: ") + bgx_last_error());
    }

    std::vector<int> board_;
    std::array<int, 4> counters_{{0, 0, 0, 0}};   // jailed P1, jailed P2, freed P1, freed P2
    int turn_ = 0;
    std::array<int, 2> dice_{{1, 1}};
    Player p1_{"", PLAYER1}, p2_{"", PLAYER2};
    Pieces pieces_;
};

int Pieces::numJailed(int player) const { return g_->getJailedCount(player == PLAYER1 ? PLAYER1 : PLAYER2); }   // Pieces.cpp:70-80
int Pieces::numFreed(int player) const { return g_->getBornOffCount(player == PLAYER1 ? PLAYER1 : PLAYER2); }   // Pieces.cpp:58-68

static py::tuple evaluate_wrapper(const Game &g, int player, int d1, int d2)   // backgammon_bindings.cpp:27-39
{
    Game::Eval ev = g.evaluate(player, d1, d2, true);
    py::array_t<int> states({(py::ssize_t)ev.n, (py::ssize_t)28});
    if (ev.n) std::memcpy(states.mutable_data(), ev.states.data(), (size_t)ev.n * 28 * sizeof(int32_t));
    return py::make_tuple(ev.sequences, states);
}

// ---- the batched entry points the reference's binding file gains (INTEGRATION.md) -----------
class BatchEngine {
  public:
    explicit BatchEngine(int device) { Game::check(bgx_create(device, &e_)); }
    ~BatchEngine() { bgx_destroy(e_); }
    BatchEngine(const BatchEngine &) = delete;

    using F32 = py::array_t<float, py::array::c_style | py::array::forcecast>;
    using I8 = py::array_t<int8_t, py::array::c_style | py::array::forcecast>;

    void set_weights(F32 W1, F32 b1, F32 w2, F32 b2)
    {
        if (W1.size() != 128 * 198 || b1.size() != 128 || w2.size() != 128 || b2.size() != 1) throw std::invalid_argument("weight shapes");
        Game::check(bgx_set_weights(e_, W1.data(), b1.data(), w2.data(), b2.data()));
    }
    static int64_t rows(const I8 &q)
    {
        if (q.ndim() != 2 || q.shape(1) != 32) throw std::invalid_argument("records are int8[n, 32]");
        return q.shape(0);
    }
    py::tuple evaluate_turn_sequences_summary(I8 q)
    {
        int64_t n = rows(q);
        py::array_t<int32_t> n_seq(n), n_unique(n);
        py::array_t<uint64_t> digest(n);
        {
            py::gil_scoped_release nogil;
            Game::check(bgx_enumerate_summary_host(e_, q.data(), n, n_seq.mutable_data(), n_unique.mutable_data(), digest.mutable_data()));
        }
        return py::make_tuple(n_seq, n_unique, digest);
    }
    py::dict make_moves(I8 q, float epsilon, uint64_t seed)
    {
        int64_t n = rows(q);
        py::array_t<int8_t> chosen({(py::ssize_t)n, (py::ssize_t)32}), moves({(py::ssize_t)n, (py::ssize_t)4, (py::ssize_t)2}), len(n);
        py::array_t<float> value(n);
        py::array_t<int32_t> n_seq(n), n_scored(n);
        {
            py::gil_scoped_release nogil;
            Game::check(bgx_select_moves_host(e_, q.data(), n, epsilon, seed, chosen.mutable_data(), moves.mutable_data(), len.mutable_data(),
                                              value.mutable_data(), n_seq.mutable_data(), n_scored.mutable_data()));
        }
        py::dict d;
        d["chosen"] = chosen; d["moves"] = moves; d["moves_len"] = len; d["value"] = value; d["n_seq"] = n_seq; d["n_scored"] = n_scored;
        return d;
    }
    py::dict make_moves_2ply(I8 q, int32_t max_candidates)
    {
        int64_t n = rows(q);
        py::array_t<int8_t> chosen({(py::ssize_t)n, (py::ssize_t)32}), moves({(py::ssize_t)n, (py::ssize_t)4, (py::ssize_t)2}), len(n);
        py::array_t<float> value(n);
        py::array_t<int32_t> n_cand(n), n_exp(n);
        {
            py::gil_scoped_release nogil;
            Game::check(bgx_select_moves_2ply_host(e_, q.data(), n, max_candidates, chosen.mutable_data(), moves.mutable_data(),
                                                   len.mutable_data(), value.mutable_data(), n_cand.mutable_data(), n_exp.mutable_data()));
        }
        py::dict d;
        d["chosen"] = chosen; d["moves"] = moves; d["moves_len"] = len; d["value"] = value; d["n_candidates"] = n_cand; d["n_expanded"] = n_exp;
        return d;
    }
    py::dict rollout(I8 q, int32_t trials, int32_t max_plies, uint64_t seed, bool stratify, bool per_trial)
    {
        int64_t n = rows(q);
        const py::ssize_t T = per_trial && trials > 0 ? trials : 0;
        py::array_t<double> mean(n), std_err(n);
        py::array_t<int64_t> counts({(py::ssize_t)n, (py::ssize_t)8});
        py::array_t<float> value({(py::ssize_t)n, T});
        py::array_t<int8_t> outcome({(py::ssize_t)n, T});
        py::array_t<int32_t> plies({(py::ssize_t)n, T});
        {
            py::gil_scoped_release nogil;
            Game::check(bgx_rollout_host(e_, q.data(), n, trials, max_plies, seed, stratify ? BGX_ROLLOUT_STRATIFY : 0, mean.mutable_data(),
                                         std_err.mutable_data(), counts.mutable_data(), per_trial ? value.mutable_data() : nullptr,
                                         per_trial ? outcome.mutable_data() : nullptr, per_trial ? plies.mutable_data() : nullptr));
        }
        py::dict d;
        d["mean"] = mean; d["std_err"] = std_err; d["counts"] = counts;
        if (per_trial) { d["trial_value"] = value; d["trial_outcome"] = outcome; d["trial_plies"] = plies; }
        return d;
    }
    py::array_t<float> encode(I8 q)
    {
        int64_t n = rows(q);
        py::array_t<float> X({(py::ssize_t)n, (py::ssize_t)198});
        py::gil_scoped_release nogil;
        Game::check(bgx_encode_host(e_, q.data(), n, X.mutable_data()));
        return X;
    }
    py::array_t<float> evaluate(I8 q)
    {
        int64_t n = rows(q);
        py::array_t<float> V(n);
        py::gil_scoped_release nogil;
        Game::check(bgx_evaluate_host(e_, q.data(), n, V.mutable_data()));
        return V;
    }

    py::tuple get_weights()
    {
        py::array_t<float> W1({128, 198}), b1(128), w2({1, 128}), b2(1);
        Game::check(bgx_get_weights(e_, W1.mutable_data(), b1.mutable_data(), w2.mutable_data(), b2.mutable_data()));
        return py::make_tuple(W1, b1, w2, b2);
    }
    // batched evaluateTurnSequences (backgammon_bindings.cpp:27-39 for n positions): offsets[n+1], moves[N,4,2], lens[N], states[N,32]
    py::tuple evaluate_turn_sequences(I8 q)
    {
        int64_t n = rows(q);
        py::array_t<int32_t> n_seq(n), n_unique(n);
        py::array_t<uint64_t> digest(n);
        Game::check(bgx_enumerate_summary_host(e_, q.data(), n, n_seq.mutable_data(), n_unique.mutable_data(), digest.mutable_data()));
        int64_t total = 0;
        for (int64_t i = 0; i < n; i++) total += n_seq.data()[i];
        py::array_t<int64_t> offsets(n + 1);
        py::array_t<int8_t> moves({(py::ssize_t)total, (py::ssize_t)4, (py::ssize_t)2}), lens(total), states({(py::ssize_t)total, (py::ssize_t)32});
        {
            py::gil_scoped_release nogil;
            int64_t got = 0;
            Game::check(bgx_enumerate_host(e_, q.data(), n, total > 0 ? total : 1, offsets.mutable_data(), moves.mutable_data(), lens.mutable_data(),
                                           states.mutable_data(), &got));
        }
        return py::make_tuple(offsets, moves, lens, states);
    }
    // one iteration of play_game's loop for n games (train.py:103-121): (next_records[n,32], winner[n], value[n], n_seq[n])
    py::tuple play_ply(I8 q, py::array_t<int32_t, py::array::c_style | py::array::forcecast> next_ply,
                       py::array_t<int64_t, py::array::c_style | py::array::forcecast> game_id, float epsilon, uint64_t explore_seed, uint64_t dice_seed)
    {
        int64_t n = rows(q);
        if (next_ply.size() != n || game_id.size() != n) throw std::invalid_argument("next_ply and game_id are [n]");
        py::array_t<int8_t> next({(py::ssize_t)n, (py::ssize_t)32}), winner(n);
        py::array_t<float> value(n);
        py::array_t<int32_t> n_seq(n);
        {
            py::gil_scoped_release nogil;
            Game::check(bgx_play_ply_host_async(e_, 0, q.data(), next_ply.data(), game_id.data(), n, epsilon, explore_seed, dice_seed,
                                                next.mutable_data(), winner.mutable_data(), value.mutable_data(), n_seq.mutable_data()));
            Game::check(bgx_lane_wait(e_, 0));
        }
        return py::make_tuple(next, winner, value, n_seq);
    }
    // ---- the self-play population and the TD(lambda) round (train.py:64-172, 527-547)
    static py::dict stats_dict(const bgx_stats &s)
    {
        py::dict d;
        d["plies"] = s.plies; d["sequences"] = s.sequences; d["scored"] = s.scored; d["games_finished"] = s.games_finished;
        d["p1_wins"] = s.p1_wins; d["truncated"] = s.truncated; d["td_steps"] = s.td_steps; d["td_sq_error"] = s.td_sq_error;
        d["tree_edges"] = s.tree_edges; d["td_live_rows"] = s.td_live_rows; d["td_lazy_row_steps"] = s.td_lazy_row_steps;
        return d;
    }
    void selfplay_init(int64_t n_slots, int64_t first_id, int64_t id_stride, uint64_t seed, int first_mover, int traj_cap, bool record_chosen)
    {
        n_slots_ = n_slots; traj_cap_ = traj_cap; record_chosen_ = record_chosen;
        Game::check(bgx_selfplay_record_chosen(e_, record_chosen ? 1 : 0));
        Game::check(bgx_selfplay_init(e_, n_slots, first_id, id_stride > 0 ? id_stride : n_slots, seed, first_mover, traj_cap));
    }
    py::dict selfplay_step(int n_plies, float epsilon)
    {
        bgx_stats s;
        { py::gil_scoped_release nogil; Game::check(bgx_selfplay_step(e_, n_plies, epsilon, &s)); }
        return stats_dict(s);
    }
    py::dict selfplay_round(float epsilon)
    {
        bgx_stats s;
        { py::gil_scoped_release nogil; Game::check(bgx_selfplay_round(e_, epsilon, &s)); }
        return stats_dict(s);
    }
    void selfplay_next_round() { Game::check(bgx_selfplay_next_round(e_)); }
    py::tuple selfplay_read()
    {
        py::array_t<int8_t> rec({(py::ssize_t)n_slots_, (py::ssize_t)32});
        py::array_t<int32_t> ply(n_slots_);
        py::array_t<int64_t> gid(n_slots_);
        Game::check(bgx_selfplay_read(e_, rec.mutable_data(), ply.mutable_data(), gid.mutable_data()));
        return py::make_tuple(rec, ply, gid);
    }
    py::tuple export_trajectory(int64_t slot)
    {
        const int cap = traj_cap_ > 0 ? traj_cap_ : 1;
        std::vector<int8_t> pre((size_t)cap * 32), cho(record_chosen_ ? (size_t)cap * 32 : 0);
        int32_t T = 0;
        Game::check(bgx_export_trajectory(e_, slot, cap, pre.data(), record_chosen_ ? cho.data() : nullptr, &T));
        py::array_t<int8_t> p({(py::ssize_t)T, (py::ssize_t)32}), c({(py::ssize_t)(record_chosen_ ? T : 0), (py::ssize_t)32});
        std::memcpy(p.mutable_data(), pre.data(), (size_t)T * 32);
        if (record_chosen_) std::memcpy(c.mutable_data(), cho.data(), (size_t)T * 32);
        return py::make_tuple(p, c);
    }
    // exact online TD(lambda) replay of every finished game from the current weights, summed; weights += scale * delta
    py::tuple td_round(double lr, double lambda, float scale)
    {
        bgx_stats s;
        py::array_t<float> delta(BGX_NPARAMS);
        { py::gil_scoped_release nogil; Game::check(bgx_td_round_host(e_, lr, lambda, scale, delta.mutable_data(), &s)); }
        return py::make_tuple(delta, stats_dict(s));
    }

  private:
    bgx_engine *e_ = nullptr;
    int64_t n_slots_ = 0;
    int traj_cap_ = 0;
    bool record_chosen_ = false;
};

PYBIND11_MODULE(backgammon_env, m)
{
    m.doc() = "Backgammon game environment for Reinforcement Learning (libbgx-backed, B200 batched engine inside)";

    py::enum_<PlayerType>(m, "PlayerType").value("PLAYER1", PLAYER1).value("PLAYER2", PLAYER2);

    py::class_<Player>(m, "Player")
        .def(py::init([](const std::string &name, PlayerType t) { return Player(name, (int)t); }))
        .def("getName", &Player::getName)
        .def("getNum", &Player::getNum);

    py::class_<Pieces>(m, "Pieces").def("numJailed", &Pieces::numJailed).def("numFreed", &Pieces::numFreed);

    py::class_<Game>(m, "Game")
        .def(py::init<int>())
        .def("setPlayers", &Game::setPlayers)
        .def("getPlayers", &Game::getPlayers)
        .def("getTurn", &Game::getTurn)
        .def("setTurn", &Game::setTurn)
        .def("getGameBoard", &Game::getGameBoard)
        .def("getPieces", &Game::getPieces, py::return_value_policy::reference_internal)
        .def("legalMoves", &Game::legalMoves)
        .def("legalTurnSequences", [](const Game &g, int player, int d1, int d2) { return g.evaluate(player, d1, d2, false).sequences; })
        .def("evaluateTurnSequences", &evaluate_wrapper,
             "Enumerate all legal turn sequences and their resulting states in one call. Returns (sequences, states[N,28]).")
        .def("tryMove", &Game::tryMove)
        .def("is_game_over", &Game::over)
        .def("clone", &Game::clone)
        .def("getJailedCount", &Game::getJailedCount)
        .def("setBorneOffPieces", &Game::setFreed)
        .def("getBornOffCount", &Game::getBornOffCount)
        .def("setGameBoard", &Game::setGameBoard)
        .def("setDice", &Game::setDice)
        .def("printGameBoard", &Game::printGameBoard)
        .def("reset", &Game::populateBoard)
        .def("populateBoard", &Game::populateBoard)
        .def("roll_dice", &Game::rollDice, "Roll two dice and return an array [die1, die2]")
        .def("get_last_dice", &Game::getLastDice, "Return the most recently rolled dice as [die1, die2]");

    py::class_<BatchEngine>(m, "BatchEngine", "Batched GPU entry points (sm_100a); raises if no CUDA device is present")
        .def(py::init<int>(), py::arg("device") = 0)
        .def("set_weights", &BatchEngine::set_weights)
        .def("evaluate_turn_sequences_summary", &BatchEngine::evaluate_turn_sequences_summary)
        .def("make_moves", &BatchEngine::make_moves, py::arg("queries"), py::arg("epsilon") = 0.0f, py::arg("seed") = 0)
        .def("make_moves_2ply", &BatchEngine::make_moves_2ply, py::arg("queries"), py::arg("max_candidates") = 0)
        .def("rollout", &BatchEngine::rollout, py::arg("positions"), py::arg("trials"), py::arg("max_plies") = 0,
             py::arg("seed") = 0x5EED2026ull, py::arg("stratify") = true, py::arg("per_trial") = false)
        .def("encode", &BatchEngine::encode)
        .def("evaluate", &BatchEngine::evaluate)
        .def("get_weights", &BatchEngine::get_weights)
        .def("evaluate_turn_sequences", &BatchEngine::evaluate_turn_sequences)
        .def("play_ply", &BatchEngine::play_ply, py::arg("records"), py::arg("next_ply"), py::arg("game_id"), py::arg("epsilon") = 0.0f,
             py::arg("explore_seed") = 0, py::arg("dice_seed") = 0x5EED2026ull)
        .def("selfplay_init", &BatchEngine::selfplay_init, py::arg("n_slots"), py::arg("first_id") = 0, py::arg("id_stride") = 0,
             py::arg("seed") = 0x5EED2026ull, py::arg("first_mover") = BGX_FIRST_ROLLOFF, py::arg("traj_cap") = 0, py::arg("record_chosen") = false)
        .def("selfplay_step", &BatchEngine::selfplay_step, py::arg("n_plies"), py::arg("epsilon") = 0.0f)
        .def("selfplay_round", &BatchEngine::selfplay_round, py::arg("epsilon") = 0.0f)
        .def("selfplay_next_round", &BatchEngine::selfplay_next_round)
        .def("selfplay_read", &BatchEngine::selfplay_read)
        .def("export_trajectory", &BatchEngine::export_trajectory)
        .def("td_round", &BatchEngine::td_round, py::arg("lr"), py::arg("lambda_decay"), py::arg("scale"));
}
